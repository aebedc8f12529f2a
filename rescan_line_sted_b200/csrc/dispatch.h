// Kernel selection of the convolution engine: which compiled instance runs a row or column
// launch.  Pure host C++ (no CUDA API).  The CUDA backend (lsted_api.cu) and the CPU replay
// (tests/host_emul/emul.cpp) both choose through select_row / select_col and turn the choice
// into template arguments through run_row / run_col.  A backend derives from KernelSelection (the
// switches, and what the engine asks about them) and provides only the executors (row_generic,
// row_fast, row2, row_mid_dual, col_generic, col_fast, col_sub, col_ht_p2p).
#pragma once
#include <stdlib.h>
#include <string>
#include "plan.h"
#include "conv_fast.cuh"

// Compile-time plans of the fast path (conv_fast.cuh): 2160 = 16 * 9 * 15.
#ifndef LSTED_FAST_C32
#define LSTED_FAST_C32 4
#endif
#ifndef LSTED_FAST_CS32
#define LSTED_FAST_CS32 2   // columns per sub-block column CTA (real OTFs): 2 CTAs per SM
#endif
#ifndef LSTED_FAST_PR
#define LSTED_FAST_PR 1
#endif
#ifndef LSTED_FP64_PR
#define LSTED_FP64_PR 1   // row pairs per CTA of the fp64 plan (A/B at build time; 2: row_mid +13 %)
#endif
#ifndef LSTED_FP64_CS
#define LSTED_FP64_CS 1   // columns per column CTA of the fp64 plan (1 of 2: sub-block CTAs; 2: col_h +15 %, col_ht +35 %)
#endif

namespace lsted {

typedef FastPlan<float, 16, 9, 15, 144, LSTED_FAST_C32, LSTED_FAST_PR, LSTED_FAST_CS32> Plan2160f;
typedef FastPlan<double, 16, 9, 15, 144, 2, LSTED_FP64_PR, LSTED_FP64_CS> Plan2160d;
typedef FastPlan2<float, 48, 45, LSTED_FAST_C32, 2> Plan2160f2;   // two-pass rows, 2160 = 48 x 45
template <typename T> struct PlanFor;
template <> struct PlanFor<float> { typedef Plan2160f type; };
template <> struct PlanFor<double> { typedef Plan2160d type; };

// image geometry known at compile time: the 2048-wide / 107-wide-PSF headline case, and the
// same with centred real OTFs (no crop offset)
typedef RowGeomFixed<2048, 53> RowGeom2048;
typedef RowGeomFixed<2048, 0> RowGeom2048c;
typedef ColGeomFixed<2048, 53> ColGeom2048;
typedef ColGeomFixed<2048, 0> ColGeom2048c;

// profiling kinds of lsted_deconv_profile (lsted.h)
enum KernelKind { KK_ROW_FWD = 0, KK_ROW_INV_STORE, KK_ROW_INV_SIM, KK_ROW_MID, KK_ROW_FINAL,
                  KK_COL_OTF, KK_COL_H, KK_COL_HT, KK_EW };

template <class P> bool plan_fits_rows(const ConvGeom& g) { return g.Lx == P::L && g.C == P::C; }
template <class P> bool plan_fits_cols(const ConvGeom& g) { return g.Ly == P::L && g.C == P::C; }
inline bool fast_plan_fits_cols(const ConvGeom& g, int cplx_bytes) {
    return cplx_bytes == 8 ? plan_fits_cols<Plan2160f>(g) : plan_fits_cols<Plan2160d>(g);
}

// The kernel-selection options of lsted_deconv_set_option.  The A/B environment variables are
// read when a handle is created.
struct KernelSwitches {
    bool fast_path = true;    // compile-time 2160 plans where the geometry fits them
    // two-pass 48 x 45 row kernels (fp32): 35 % fewer warp instructions and half the shared-memory
    // wavefronts, but 0.334 ms vs 0.283 ms for ROW_MID: 4792 straight-line instructions run by
    // 9 warps per SM stall on instruction fetch (ncu: no_inst 32 %).  Kept behind this switch.
    bool row_plan2 = false;
    bool row_dual = false;    // measured: 0.326 ms vs 0.311 ms for the single-pair kernel (L1TEX-bound either way)
    int row_tma = 2;          // 0 off, 1 tensor-map spectrum copies, 2 also the two-buffer ROW_MID (6 CTAs/SM)
    bool col_sub = true;      // sub-block column CTAs (2 per SM) where the plan has them
    bool real_otf = true;     // centred real OTFs of point-symmetric PSFs (read at set_psfs)
    bool prefetch = true;     // row kernels L2-prefetch the operands of a CTA one wave ahead
    bool k_split = true;      // orientations of small frames over idle SMs (col_h)

    KernelSwitches() {
        if (const char* v = getenv("LSTED_ROW_TMA")) row_tma = atoi(v);
        env("LSTED_ROW_DUAL", row_dual);
        env("LSTED_ROW_PLAN2", row_plan2);
        env("LSTED_COL_SUB", col_sub);
        env("LSTED_REAL_OTF", real_otf);
        env("LSTED_PREFETCH", prefetch);
    }
    static void env(const char* name, bool& on) {
        if (const char* v = getenv(name)) on = atoi(v) != 0;
    }
};

// What the deconvolver (engine.h) and the C ABI (api_deconv.inl) ask a backend about kernel
// selection.  Both backends derive from it, so they hold the same switches and give the same
// answers.
struct KernelSelection {
    KernelSwitches sw;
    // columns per block of the compile-time plan for column length L (make_geom), 0: none
    static int fast_cols(int L, int cplx_bytes) {
        if (L == Plan2160f::L) return cplx_bytes == 8 ? (int)Plan2160f::C : (int)Plan2160d::C;
        return 0;
    }
    // centred real OTFs are read by the compile-time column kernels only
    bool real_otf_supported(const ConvGeom& g, int cplx_bytes) const {
        return sw.fast_path && sw.real_otf && fast_plan_fits_cols(g, cplx_bytes);
    }
    // tensor-map staging of the row spectra: fp32 plan with one pair per CTA; two boxes cover the
    // blocks, 128-byte aligned in shared memory
    bool row_tma_supported(const ConvGeom& g, int cplx_bytes) const {
        return sw.fast_path && sw.row_tma && cplx_bytes == 8 && plan_fits_rows<Plan2160f>(g) &&
               Plan2160f::PR == 1 && g.nxb >= kTmaBoxBlocks && g.nxb <= 2 * kTmaBoxBlocks &&
               (g.nxb - kTmaBoxBlocks) % 2 == 0;
    }
    void set_fast_path(bool on) { sw.fast_path = on; }
    void set_row_plan2(bool on) { sw.row_plan2 = on; }
    void set_row_dual(bool on) { sw.row_dual = on; }
    void set_row_tma(int v) { sw.row_tma = v; }
    void set_col_sub(bool on) { sw.col_sub = on; }
    void set_real_otf(bool on) { sw.real_otf = on; }
    void set_prefetch(bool on) { sw.prefetch = on; }
    void set_k_split(bool on) { sw.k_split = on; }
};

// What the device offers a launch: its SMs, the deconvolver handles alive in the process (with
// many of them the GPU is kept busy by the other handles' kernels) and the most CTAs one column
// block's orientations may be spread over.
struct DeviceShape { int num_sms, live_handles, max_k_split; };

enum class Geom { runtime, g2048, g2048c };
enum class RowVariant { generic, fast, row2, row_mid_dual };
enum class ColVariant { generic, fast, fast_sub, ht_p2p };
struct RowChoice {
    RowVariant variant;
    Geom geom;
    int tma;     // fast: 0 per-thread spectrum loads, 1 tensor-map copies, 2 also the two-buffer kernel
    int grid;
    int kind;    // KernelKind
};
struct ColChoice {
    ColVariant variant;
    Geom geom;
    bool real_otf;   // fast, fast_sub, ht_p2p: centred real OTFs
    int grid;
    int k_split;     // generic COL_H: CTAs per column block
    int kind;
};

template <int MODE, typename T>
RowChoice select_row(int grid, const RowArgs<T>& a, const KernelSwitches& sw) {
    typedef typename PlanFor<T>::type P;
    const bool fp32 = sizeof(T) == 4;
    RowChoice c = {RowVariant::generic, Geom::runtime, 0, grid, KK_ROW_FWD + MODE};
    if (!sw.fast_path || !plan_fits_rows<P>(a.g)) return c;
    const int pairs = (a.g.Ny + 1) / 2;
    if (fp32 && sw.row_plan2) {
        c.variant = RowVariant::row2;
        c.grid = a.nimg * ((pairs + Plan2160f2::PR - 1) / Plan2160f2::PR);
        return c;
    }
    if (fp32 && sw.row_dual && MODE == ROW_MID && a.g.Ny % 4 == 0) {
        c.variant = RowVariant::row_mid_dual;
        c.grid = a.nimg * (a.g.Ny / 4);
        return c;
    }
    // the plan's own pairs-per-CTA decides the grid (the generic geometry may differ)
    c.variant = RowVariant::fast;
    c.grid = a.nimg * ((pairs + P::PR - 1) / P::PR);
    // fp32 kernels that index pixels have instances with the headline geometry folded in
    if (fp32 && MODE != ROW_FWD && a.g.Nx == 2048 && a.g.Ny % 2 == 0)
        c.geom = a.g.sx == (int)RowGeom2048::SX ? Geom::g2048 : a.g.sx == 0 ? Geom::g2048c : Geom::runtime;
    // spectrum chunks by tensor-map bulk copies (fp32, one pair per CTA, ROW_MID / ROW_FINAL);
    // level 2, the "lean" ROW_MID, stages the measurement rows in the first exchange buffer:
    // two buffers, one more CTA per SM (bulk copies: 16-byte multiples, 16-byte aligned)
    if (fp32 && P::PR == 1 && (MODE == ROW_MID || MODE == ROW_FINAL) && a.tmap_in && a.tmap_out && sw.row_tma)
        c.tma = sw.row_tma == 2 && (a.g.Nx * sizeof(T)) % 16 == 0 && ((size_t)a.aux & 15) == 0 &&
                        (MODE == ROW_MID || ((size_t)a.real_out & 15) == 0) ? 2 : 1;
    return c;
}

template <int MODE, typename T>
ColChoice select_col(int grid, const ColArgs<T>& a, const KernelSwitches& sw, const DeviceShape& dev) {
    typedef typename PlanFor<T>::type P;
    const bool fp32 = sizeof(T) == 4;
    ColChoice c = {ColVariant::generic, Geom::runtime, false, grid, 1, KK_COL_OTF + MODE};
    if (MODE != COL_OTF && sw.fast_path && plan_fits_cols<P>(a.g)) {
        c.variant = ColVariant::fast;
        c.real_otf = a.otf_real != 0;
        if (MODE == COL_HT && a.p2p_world > 1) {
            c.variant = ColVariant::ht_p2p;   // fused cross-GPU sum
            return c;
        }
        if (fp32 && a.g.Ny == 2048 && a.rows_in == a.g.Ny) {
            if (c.real_otf && a.g.sy == 0) c.geom = Geom::g2048c;
            if (!c.real_otf && a.g.sy == (int)ColGeom2048::SY) c.geom = Geom::g2048;
        }
        // plans with sub-blocks (CS < C): NSUB CTAs per column block, two resident per SM
        if (c.real_otf && (int)P::CS < (int)P::C && sw.col_sub) {
            c.variant = ColVariant::fast_sub;
            c.grid = grid * (int)P::NSUB;
        }
        return c;
    }
    if (col_smem_bytes(a.g, (int)sizeof(cplx<T>), MODE == COL_OTF ? 2 : 3) > kSmemLimit)
        throw std::string("generic column kernel does not fit in shared memory for this geometry");
    if (MODE == COL_H && a.K > 1 && sw.k_split && 2 * grid <= dev.num_sms && dev.live_handles <= 2) {
        // a small frame (the reference's 128^2 objects: 25 column blocks): the K + 1 dependent
        // transforms of a block are the latency of this launch; spread the orientations over
        // the idle SMs, every CTA repeating the forward transform
        c.k_split = dev.num_sms / grid;
        if (c.k_split > a.K) c.k_split = a.K;
        if (c.k_split > dev.max_k_split) c.k_split = dev.max_k_split;
        c.grid = grid * c.k_split;
    }
    return c;
}

// Visits `f` with a value of the compile-time geometry type of `g`.
template <class F> void with_row_geom(Geom g, F f) {
    if (g == Geom::g2048) f(RowGeom2048());
    else if (g == Geom::g2048c) f(RowGeom2048c());
    else f(RowGeomRuntime());
}

template <int MODE, typename T, class BK> void run_row(BK& bk, const RowChoice& c, const RowArgs<T>& a) {
    typedef typename PlanFor<T>::type P;
    if (c.grid <= 0) return;
    switch (c.variant) {
    case RowVariant::generic: bk.template row_generic<MODE, T>(c, a); return;
    case RowVariant::row2:
        if constexpr (sizeof(T) == 4) bk.template row2<MODE, Plan2160f2>(c, a);
        return;
    case RowVariant::row_mid_dual:
        if constexpr (sizeof(T) == 4 && MODE == ROW_MID) bk.template row_mid_dual<Plan2160f>(c, a);
        return;
    case RowVariant::fast:
        with_row_geom(c.geom, [&](auto geom) {
            typedef decltype(geom) G;
            if constexpr (sizeof(T) == 4 && P::PR == 1 && (MODE == ROW_MID || MODE == ROW_FINAL)) {
                if (c.tma == 2) return bk.template row_fast<MODE, P, G, 2>(c, a);
                if (c.tma == 1) return bk.template row_fast<MODE, P, G, 1>(c, a);
            }
            bk.template row_fast<MODE, P, G, 0>(c, a);
        });
        return;
    }
}

template <int MODE, typename T, class BK> void run_col(BK& bk, const ColChoice& c, const ColArgs<T>& a) {
    typedef typename PlanFor<T>::type P;
    if (c.grid <= 0) return;
    if (c.variant == ColVariant::generic) {
        ColArgs<T> b = a;
        b.k_split = c.k_split;
        bk.template col_generic<MODE, T>(c, b);
        return;
    }
    if constexpr (MODE != COL_OTF) {
        const bool c2048 = c.geom == Geom::g2048c;
        switch (c.variant) {
        case ColVariant::ht_p2p:
            if (c.real_otf) bk.template col_ht_p2p<P, true>(c, a);
            else bk.template col_ht_p2p<P, false>(c, a);
            return;
        case ColVariant::fast_sub:
            if constexpr ((int)P::CS < (int)P::C) {
                if (c2048) bk.template col_sub<MODE, P, ColGeom2048c>(c, a);
                else bk.template col_sub<MODE, P, ColGeomRuntime>(c, a);
            }
            return;
        default:
            if (c.real_otf && c2048) bk.template col_fast<MODE, P, ColGeom2048c, true>(c, a);
            else if (c.real_otf) bk.template col_fast<MODE, P, ColGeomRuntime, true>(c, a);
            else if (c.geom == Geom::g2048) bk.template col_fast<MODE, P, ColGeom2048, false>(c, a);
            else bk.template col_fast<MODE, P, ColGeomRuntime, false>(c, a);
            return;
        }
    }
}

}  // namespace lsted
