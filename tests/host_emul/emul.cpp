// TEST INFRASTRUCTURE ONLY -- CPU replay of the kernel bodies.
//
// Compiles the very same row/column/FFT bodies that lsted_api.cu launches
// as sm_100a kernels, but runs every CTA serially (parallel_for = plain
// loop, one "block" after another).  It lets the `-m "not gpu"` tests check
// the numerics and the orchestration of the engine in the build container,
// which has no GPU.  The product never loads this library: the package
// binds liblsted.so only and fails loudly when that is missing.
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <new>
#include <initializer_list>
#include <string>
#include <vector>
#include "../../include/lsted.h"
#include "../../rescan_line_sted_b200/csrc/engine.h"
#include "../../rescan_line_sted_b200/csrc/tiled.h"
#include "../../rescan_line_sted_b200/csrc/conv_fast.cuh"
#include "../../rescan_line_sted_b200/csrc/ew_bodies.cuh"
#include "../../rescan_line_sted_b200/csrc/psf_kernels.cuh"
#include "../../rescan_line_sted_b200/csrc/dispatch.h"

namespace lsted {
struct ApiError { int code; std::string msg; };
}

static thread_local std::string g_error;
static int set_error(int code, const std::string& msg) { g_error = msg; return code; }
extern "C" const char* lsted_last_error(void) { return g_error.c_str(); }

struct HostCtx {
    int nthreads;
    HostCtx() : nthreads(1) {}
    template <class F> void parallel_for(int n, F f) { for (int w = 0; w < n; ++w) f(w); }
    // register-resident bodies: every "thread" keeps its own Regs between phases
    template <class R, class F> void phase(R* regs, F f) {
        for (int t = 0; t < nthreads; ++t) f(t, regs[t]);
    }
    template <class R, class F> void phase_nosync(R* regs, F f) { phase(regs, f); }
};

typedef void (*allreduce_cb)(double* buf, size_t n);
typedef void (*broadcast_cb)(double* buf, size_t n, int root);
// halo exchange of a tile-sharded object: npeers, peers, send pointers / counts, receive
// pointers / counts (float64 elements); the test routes it to torch.distributed isend / irecv
typedef void (*exchange_cb)(int npeers, const int* peers, double* const* send, const size_t* nsend,
                            double* const* recv, const size_t* nrecv);
static exchange_cb g_exchange = 0;
extern "C" void emul_set_exchange(exchange_cb cb) { g_exchange = cb; }
static allreduce_cb g_allreduce = 0;
static broadcast_cb g_broadcast = 0;
extern "C" void emul_set_allreduce(allreduce_cb cb) { g_allreduce = cb; }
extern "C" void emul_set_broadcast(broadcast_cb cb) { g_broadcast = cb; }

static int g_dual_launches = 0;
static int g_row2_launches = 0;
static int g_real_otf_launches = 0;
static int g_row_tma_launches = 0;
static int g_k_split_launches = 0;
static int g_col_sub_launches = 0;
extern "C" int emul_k_split_launches(void) { return g_k_split_launches; }
extern "C" int emul_col_sub_launches(void) { return g_col_sub_launches; }
extern "C" int emul_row_tma_launches(void) { return g_row_tma_launches; }
extern "C" int emul_real_otf_launches(void) { return g_real_otf_launches; }
extern "C" int emul_row2_launches(void) { return g_row2_launches; }
extern "C" int emul_dual_launches(void) { return g_dual_launches; }
// Every row / column launch's choice (dispatch.h), kLogInts per launch: kernel kind, variant,
// geometry, TMA level, real OTFs, grid, CTAs per column block.  Copies the records from `first`
// on (at most `cap`) and returns how many there are.
enum { kLogInts = 7 };
static std::vector<int> g_dispatch_log;
extern "C" int emul_dispatch_log(int first, int* out, int cap) {
    const int n = (int)g_dispatch_log.size() / kLogInts;
    for (int i = first; i < n && i - first < cap; ++i)
        memcpy(out + (size_t)(i - first) * kLogInts, &g_dispatch_log[(size_t)i * kLogInts], sizeof(int) * kLogInts);
    return n;
}
static void log_choice(std::initializer_list<int> r) { g_dispatch_log.insert(g_dispatch_log.end(), r); }

class HostBackend : public lsted::KernelSelection {
  public:
    explicit HostBackend(int) : bytes_(0) {}
    int row_prefetch_distance() const { return sw.prefetch ? 3 : 0; }
    int row_final_prefetch_distance() const { return sw.prefetch ? 5 : 0; }
    // NVLS needs the NVSwitch: never available on the CPU replay
    static bool nvls_device_supported(int) { return false; }
    bool nvls_ready(const void*) const { return false; }
    int nvls_create(int, size_t) { throw std::string("NVLS: GPU only"); }
    void nvls_import(int, size_t, int) { throw std::string("NVLS: GPU only"); }
    void nvls_add_device() { throw std::string("NVLS: GPU only"); }
    void* nvls_bind(int) { throw std::string("NVLS: GPU only"); }
    template <typename T> void nvls_allreduce(T*, size_t) { throw std::string("NVLS: GPU only"); }
    void set_nvls_shape(int, int) {}
    void set_nvls_probe(bool) {}
    void set_graph(bool) {}
    bool graph_capable() const { return false; }   // captured launches exist on the GPU only
    void graph_begin() {}
    void graph_abort() {}
    void* graph_end() { return 0; }
    void graph_launch(void*) {}
    void graph_destroy(void*) {}
    void activate() {}
    void sync() {}
    void* alloc(size_t bytes) { bytes_ += bytes; return malloc(bytes ? bytes : 1); }
    void free(void* p) { ::free(p); }
    size_t bytes_allocated() const { return bytes_; }
    void upload(void* d, const void* s, size_t n) { memcpy(d, s, n); }
    void download(void* d, const void* s, size_t n) { memcpy(d, s, n); }
    // collectives: a callback installed by the test (torch.distributed over gloo)
    void comm_init(const char*, int, int) {}
    void all_reduce_sum(double* p, size_t n) {
        if (!g_allreduce) throw std::string("no all-reduce callback installed");
        g_allreduce(p, n);
    }
    void all_reduce_sum(float* p, size_t n) {
        std::vector<double> tmp(p, p + n);
        all_reduce_sum(tmp.data(), n);
        for (size_t i = 0; i < n; ++i) p[i] = (float)tmp[i];
    }
    void broadcast(double* p, size_t n, int root) {
        if (!g_broadcast) throw std::string("no broadcast callback installed");
        g_broadcast(p, n, root);
    }
    void broadcast(float* p, size_t n, int root) {
        std::vector<double> tmp(p, p + n);
        broadcast(tmp.data(), n, root);
        for (size_t i = 0; i < n; ++i) p[i] = (float)tmp[i];
    }
    void fill_double(double* p, size_t n, double v) { for (size_t i = 0; i < n; ++i) p[i] = v; }
    // peer-memory reduction: GPU only (the CPU replay reduces through the callback)
    void zero_bytes(void* p, size_t n) { memset(p, 0, n); }
    template <typename T> void otf_center(const lsted::OtfCenterArgs<T>& a0) {
        lsted::OtfCenterArgs<T> a = a0;
        a.CS = (int)lsted::PlanFor<T>::type::CS;
        for (size_t i = 0; i < a.n; ++i) lsted::otf_center_apply<T>(a, i);
    }
    // tensor-map copies: the host replay runs the same staged code path with plain loops
    // (fft_core.cuh); the "descriptor" is just a non-null token
    void* make_spec_tmap(void*, int, int, int, int, int) { return alloc(8); }
    void p2p_export(void*, void*, void*, char*) { throw std::string("peer memory needs GPUs"); }
    void p2p_attach(int, int, const char*, size_t) { throw std::string("peer memory needs GPUs"); }
    bool p2p_ready(const lsted::ConvGeom&, int) const { return false; }
    template <typename T> void p2p_fill(lsted::ColArgs<T>&) {}
    void p2p_wait(int) {}
    void set_profile(bool) {}
    void timer_start() {}
    float timer_stop() { return 0.f; }
    void profile_collect(double* ms, long long* n) {
        for (int i = 0; i < LSTED_NUM_KERNEL_KINDS; ++i) { if (ms) ms[i] = 0; if (n) n[i] = 0; }
    }
    void profile_reset() {}

    // ---- launches: dispatch.h chooses as on the GPU; the executors run the CTAs one by one ----
    template <int MODE, typename T> void launch_row(int grid, const lsted::RowArgs<T>& a) {
        const lsted::RowChoice c = lsted::select_row<MODE>(grid, a, sw);
        log_choice({c.kind, (int)c.variant, (int)c.geom, c.tma, 0, c.grid, 1});
        g_row2_launches += c.variant == lsted::RowVariant::row2;
        g_dual_launches += c.variant == lsted::RowVariant::row_mid_dual;
        g_row_tma_launches += c.tma > 0;
        lsted::run_row<MODE>(*this, c, a);
    }
    template <int MODE, typename T> void launch_col(int grid, const lsted::ColArgs<T>& a) {
        // a B200 with one live handle; at most 3 CTAs per column block keeps the split of most K uneven
        const lsted::DeviceShape dev = {148, 1, 3};
        const lsted::ColChoice c = lsted::select_col<MODE>(grid, a, sw, dev);
        log_choice({c.kind, (int)c.variant, (int)c.geom, 0, c.real_otf, c.grid, c.k_split});
        g_col_sub_launches += c.variant == lsted::ColVariant::fast_sub;
        g_real_otf_launches += c.variant != lsted::ColVariant::generic && c.real_otf;
        g_k_split_launches += c.k_split > 1;
        lsted::run_col<MODE>(*this, c, a);
    }
    // the CTAs of one launch, each with its own shared memory and per-thread registers
    template <class S, class R, class F> void ctas(int grid, size_t smem_bytes, int threads, F body) {
#pragma omp parallel
        {
            std::vector<S> smem(smem_bytes / sizeof(S) + 1);
            std::vector<R> regs(threads);
            HostCtx cx;
            cx.nthreads = threads;
#pragma omp for schedule(dynamic)
            for (int b = 0; b < grid; ++b) body(cx, b, smem.data(), regs.data());
        }
    }
    template <int MODE, typename T> void row_generic(const lsted::RowChoice& c, const lsted::RowArgs<T>& a) {
        ctas<lsted::cplx<T>, char>(c.grid, lsted::row_smem_bytes(a.g, sizeof(lsted::cplx<T>)), 1,
                                   [&](HostCtx& cx, int b, auto* smem, auto*) { lsted::row_body<MODE, T>(cx, b, a, smem); });
    }
    template <int MODE, class P, class G, int TMA>
    void row_fast(const lsted::RowChoice& c, const lsted::RowArgs<typename P::T>& a) {
        ctas<lsted::cplx<typename P::T>, lsted::RowRegs<P> >(
            c.grid, lsted::fast_row_smem_bytes<P>(MODE, TMA == 2), P::ROW_THREADS,
            [&](HostCtx& cx, int b, auto* smem, auto* regs) { lsted::row_fast_body<MODE, P, HostCtx, G, TMA>(cx, b, a, smem, regs); });
    }
    template <int MODE, class P> void row2(const lsted::RowChoice& c, const lsted::RowArgs<float>& a) {
        ctas<lsted::cplx<float>, lsted::Row2Regs<P> >(
            c.grid, lsted::fast_row2_smem_bytes<P>(MODE), P::ROW_THREADS,
            [&](HostCtx& cx, int b, auto* smem, auto* regs) { lsted::row2_fast_body<MODE, P>(cx, b, a, smem, regs); });
    }
    template <class P> void row_mid_dual(const lsted::RowChoice& c, const lsted::RowArgs<float>& a) {
        typedef lsted::RowDual<P> D;
        ctas<lsted::c2, typename D::Regs>(c.grid, D::smem_bytes(), D::THREADS, [&](HostCtx& cx, int b, auto* smem, auto* regs) {
            lsted::row_mid_dual_body<P>(cx, b, a, (unsigned char*)smem, regs);
        });
    }
    template <int MODE, typename T> void col_generic(const lsted::ColChoice& c, const lsted::ColArgs<T>& a) {
        ctas<lsted::cplx<T>, char>(c.grid, lsted::col_smem_bytes(a.g, sizeof(lsted::cplx<T>), MODE == lsted::COL_OTF ? 2 : 3), 1,
                                   [&](HostCtx& cx, int b, auto* smem, auto*) { lsted::col_body<MODE, T>(cx, b, a, smem); });
    }
    template <int MODE, class P, class G, bool RO>
    void col_fast(const lsted::ColChoice& c, const lsted::ColArgs<typename P::T>& a) {
        ctas<lsted::cplx<typename P::T>, lsted::ColRegs<P> >(
            c.grid, lsted::fast_col_smem_bytes<P>(), P::COL_THREADS,
            [&](HostCtx& cx, int b, auto* smem, auto* regs) { lsted::col_fast_body<MODE, P, HostCtx, G, RO>(cx, b, a, smem, regs); });
    }
    template <int MODE, class P, class G>
    void col_sub(const lsted::ColChoice& c, const lsted::ColArgs<typename P::T>& a) {
        ctas<lsted::cplx<typename P::T>, lsted::ColRegs<P> >(
            c.grid, lsted::fast_col_sub_smem_bytes<P>(), P::SUB_THREADS,
            [&](HostCtx& cx, int b, auto* smem, auto* regs) { lsted::col_fast_body<MODE, P, HostCtx, G, true, true>(cx, b, a, smem, regs); });
    }
    template <class P, bool RO> void col_ht_p2p(const lsted::ColChoice&, const lsted::ColArgs<typename P::T>&) {
        throw std::string("peer memory needs GPUs");
    }
    template <int OP, typename T> void ew(const lsted::EwArgs<T>& a) {
        for (size_t i = 0; i < a.n; ++i) lsted::ew_apply<OP, T>(a, i);
    }
    template <int PASS, typename T> void dft_direct(const lsted::DftArgs<T>& a) {
        const size_t n = (size_t)a.Ny * a.Nx;
#pragma omp parallel for schedule(static)
        for (long long e = 0; e < (long long)n; ++e) lsted::dft_direct_apply<PASS, T>(a, (size_t)e);
    }
    template <typename T> void launch_rect(const lsted::RectArgs<T>& a) {
        const size_t n = (size_t)a.nimg * a.h * a.w;
        for (size_t e = 0; e < n; ++e) lsted::rect_apply<T>(a, e);
    }
    void exchange(int npeers, const int* peers, double* const* send, const size_t* nsend,
                  double* const* recv, const size_t* nrecv) {
        if (!g_exchange) throw std::string("no exchange callback installed");
        g_exchange(npeers, peers, send, nsend, recv, nrecv);
    }
    void exchange(int npeers, const int* peers, float* const* send, const size_t* nsend,
                  float* const* recv, const size_t* nrecv) {
        std::vector<std::vector<double> > s(npeers), r(npeers);
        std::vector<double*> sp(npeers), rp(npeers);
        for (int i = 0; i < npeers; ++i) {
            s[i].assign(send[i], send[i] + nsend[i]);
            r[i].resize(nrecv[i]);
            sp[i] = s[i].data(); rp[i] = r[i].data();
        }
        exchange(npeers, peers, sp.data(), nsend, rp.data(), nrecv);
        for (int i = 0; i < npeers; ++i)
            for (size_t k = 0; k < nrecv[i]; ++k) recv[i][k] = (float)r[i][k];
    }
    template <int OP, typename T> void launch_win(const lsted::WinArgs<T>& a) {
        const size_t n = (size_t)a.nimg * a.W * a.W;
        for (size_t e = 0; e < n; ++e) lsted::win_apply<OP, T>(a, e);
    }
    template <typename T> void cast_in(T* dst, const double* src, size_t n, double s) {
        lsted::EwArgs<T> a; memset(&a, 0, sizeof(a)); a.t0 = dst; a.d1 = src; a.s = s; a.n = n;
        ew<lsted::EW_CAST_IN, T>(a);
    }
    template <typename T> void cast_out(double* dst, const T* src, size_t n) {
        lsted::EwArgs<T> a; memset(&a, 0, sizeof(a)); a.d0 = dst; a.t1 = src; a.n = n;
        ew<lsted::EW_CAST_OUT, T>(a);
    }
    template <typename T> void fill(T* dst, size_t n, T v) {
        lsted::EwArgs<T> a; memset(&a, 0, sizeof(a)); a.t0 = dst; a.s = (double)v; a.n = n;
        ew<lsted::EW_FILL, T>(a);
    }
    template <typename T> void divide(T* io, const T* den, size_t n) {
        lsted::EwArgs<T> a; memset(&a, 0, sizeof(a)); a.t0 = io; a.t1 = den; a.n = n;
        ew<lsted::EW_DIVIDE, T>(a);
    }
    template <typename T> void subtract(T* dst, const T* a, const T* b, size_t n) {
        lsted::EwArgs<T> e; memset(&e, 0, sizeof(e)); e.t0 = dst; e.t1 = a; e.t2 = b; e.n = n;
        ew<lsted::EW_SUB, T>(e);
    }
    template <typename T> void launch_col_logmag(int grid, const lsted::ColArgs<T>& a) {
        std::vector<lsted::cplx<T> > smem((size_t)3 * a.g.C * a.g.Lpy);
        HostCtx cx;
        for (int b = 0; b < grid; ++b) lsted::col_body<lsted::COL_LOGMAG, T>(cx, b, a, smem.data());
    }
    template <typename T> void rl_update(T* est, const T* num, const T* den, size_t n) {
        lsted::EwArgs<T> a; memset(&a, 0, sizeof(a)); a.t0 = est; a.t1 = num; a.t2 = den; a.n = n;
        ew<lsted::EW_RL_UPDATE, T>(a);
    }
    double sum(const double* x, size_t n, double*) {
        long double s = 0;
        for (size_t i = 0; i < n; ++i) s += x[i];
        return (double)s;
    }

  private:
    size_t bytes_;
};

#define LSTED_BACKEND HostBackend
#include "../../rescan_line_sted_b200/csrc/api_deconv.inl"

// Direct access to the batched shared-memory FFT for unit tests:
// in/out are [nbatch][L] interleaved (re, im) float64.
template <typename T>
static void run_fft(int L, int dir, int nbatch, const double* in, double* out) {
    lsted::FftPlan plan;
    if (!lsted::make_fft_plan(L, &plan)) throw std::string("unsupported length");
    const int Lp = lsted::smem_pitch(L, (int)sizeof(lsted::cplx<T>), 1);
    std::vector<lsted::cplx<T> > a((size_t)nbatch * Lp), b((size_t)nbatch * Lp), tw(L);
    lsted::fill_twiddles<T>(L, tw.data());
    for (int f = 0; f < nbatch; ++f)
        for (int i = 0; i < L; ++i)
            a[(size_t)f * Lp + lsted::pad<T>(i)] =
                lsted::mk<T>((T)in[2 * ((size_t)f * L + i)], (T)in[2 * ((size_t)f * L + i) + 1]);
    HostCtx cx;
    lsted::SmemSrc<T> s = {a.data(), Lp};
    const lsted::cplx<T>* z = dir < 0
        ? lsted::fft_batch<-1, T>(cx, plan, tw.data(), s, b.data(), a.data(), nbatch, Lp)
        : lsted::fft_batch<+1, T>(cx, plan, tw.data(), s, b.data(), a.data(), nbatch, Lp);
    for (int f = 0; f < nbatch; ++f)
        for (int i = 0; i < L; ++i) {
            out[2 * ((size_t)f * L + i)] = (double)z[(size_t)f * Lp + lsted::pad<T>(i)].x;
            out[2 * ((size_t)f * L + i) + 1] = (double)z[(size_t)f * Lp + lsted::pad<T>(i)].y;
        }
}

extern "C" int emul_fft(int L, int dir, int nbatch, int precision, const double* in, double* out) {
    try {
        if (precision == 32) run_fft<float>(L, dir, nbatch, in, out);
        else run_fft<double>(L, dir, nbatch, in, out);
    } catch (const std::string& s) { return set_error(LSTED_ERR_ARG, s); }
    return 0;
}

extern "C" int emul_next_smooth_len(int n) { return lsted::next_smooth_len(n); }

extern "C" int emul_fft_plan(int L, int* radices, int cap) {
    lsted::FftPlan p;
    if (!lsted::make_fft_plan(L, &p)) return -1;
    for (int i = 0; i < p.npass && i < cap; ++i) radices[i] = p.radix[i];
    return p.npass;
}

extern "C" int emul_poisson(double lam, uint64_t seed, uint64_t first_pixel, int n, double* out) {
    for (int i = 0; i < n; ++i) out[i] = lsted::poisson_sample(lam, seed, first_pixel + i, 0);
    return 0;
}

// PSF synthesis bodies, replayed one CTA after another.
extern "C" int lsted_psf_illumination(int, int psf_type, int batch, int n, const double* taps,
                                      int radius, const double* eb, const double* db,
                                      double* excitation, double* depletion, double* exc_frac,
                                      double* dep_frac, double* sted) {
    if (n > lsted::kPsfMaxN || 2 * radius + 1 > lsted::kPsfMaxTaps)
        return set_error(LSTED_ERR_ARG, "PSF grid too large for the on-chip kernel");
    const size_t img = (size_t)n * n;
    std::vector<double> out(img * 5 * batch);
    lsted::PsfIlluminationArgs a;
    a.psf_type = psf_type; a.n = n; a.radius = radius; a.taps = taps;
    a.exc_brightness = eb; a.dep_brightness = db; a.out = out.data();
    std::vector<lsted::PsfSmem> sm(1);
    HostCtx cx;
    for (int b = 0; b < batch; ++b) lsted::psf_illumination_body(cx, b, a, sm.data());
    double* outs[5] = {excitation, depletion, exc_frac, dep_frac, sted};
    for (int b = 0; b < batch; ++b)
        for (int i = 0; i < 5; ++i)
            memcpy(outs[i] + img * b, out.data() + img * (5 * (size_t)b + i), sizeof(double) * img);
    return 0;
}

extern "C" int lsted_psf_rescan(int, int batch, int n, const double* taps, int radius,
                                const double* sted_rows, const int* ratios, double* emission,
                                double* rescan, double* descan, double* wide) {
    if (n > lsted::kPsfMaxN || 2 * radius + 1 > lsted::kPsfMaxTaps)
        return set_error(LSTED_ERR_ARG, "PSF grid too large for the on-chip kernel");
    if (wide && batch != 1) return set_error(LSTED_ERR_ARG, "`wide` output needs batch == 1");
    const size_t img = (size_t)n * n;
    std::vector<double> out(img * 3 * batch);
    lsted::PsfRescanArgs a;
    a.n = n; a.radius = radius; a.taps = taps; a.sted_rows = sted_rows; a.ratios = ratios;
    a.out = out.data(); a.wide = wide;
    std::vector<lsted::PsfSmem> sm(1);
    HostCtx cx;
    for (int b = 0; b < batch; ++b) lsted::psf_rescan_body(cx, b, a, sm.data());
    double* outs[3] = {emission, rescan, descan};
    for (int b = 0; b < batch; ++b)
        for (int i = 0; i < 3; ++i)
            memcpy(outs[i] + img * b, out.data() + img * (3 * (size_t)b + i), sizeof(double) * img);
    return 0;
}

extern "C" int lsted_psf_report_batch(int, int psf_type, int batch, const int* n, const int* radius,
                                      const double* taps, int tap_stride, const double* blur_sigma,
                                      const double* eb, const double* db, double* scalars, double* psfs) {
    int nmax = 0;
    for (int b = 0; b < batch; ++b) nmax = n[b] > nmax ? n[b] : nmax;
    if (nmax > lsted::kPsfMaxN) return set_error(LSTED_ERR_ARG, "PSF grid too large for the on-chip kernel");
    lsted::PsfReportArgs a;
    a.psf_type = psf_type; a.nmax = nmax; a.tap_stride = tap_stride; a.n = n; a.radius = radius;
    a.taps = taps; a.blur_sigma = blur_sigma; a.exc_brightness = eb; a.dep_brightness = db;
    a.scalars = scalars; a.psfs = psfs;
    std::vector<double> scratch(lsted::PsfReportSmem::doubles(nmax));
    lsted::PsfReportSmem sm;
    sm.carve(scratch.data(), nmax);
    HostCtx cx;
    for (int b = 0; b < batch; ++b) lsted::psf_report_body(cx, b, a, &sm);
    return 0;
}

extern "C" int lsted_gauss_fit(int, int batch, int n, const double* rows, double* out) {
    lsted::GaussFitArgs a;
    a.n = n; a.rows = rows; a.out = out;
    std::vector<double> scratch(lsted::PsfReportSmem::doubles(n));
    lsted::PsfReportSmem sm;
    sm.carve(scratch.data(), n);
    HostCtx cx;
    for (int b = 0; b < batch; ++b) lsted::gauss_fit_rows_body(cx, b, a, &sm);
    return 0;
}

extern "C" int lsted_psf_rotate(int, int batch, int n0, int n1, const double* plane,
                               const double* xform, double clip_hi, double* out) {
    const size_t img = (size_t)n0 * n1;
    std::vector<double> coef(img * batch);
    lsted::PsfRotateArgs a;
    a.n0 = n0; a.n1 = n1; a.plane = plane; a.xform = xform; a.clip_hi = clip_hi;
    a.coef = coef.data(); a.out = out;
    HostCtx cx;
    for (int b = 0; b < batch; ++b) lsted::psf_rotate_body(cx, b, a);
    return 0;
}

// Two-pass plan (fft_static.cuh: Fft2E) of the row kernels, 2160 = 48 x 45: one sequence,
// threads replayed one after another.  in/out: [2160] interleaved (re, im) float64.
template <typename T, int DIR, int RA, int RC>
static void run_fft2(const double* in, double* out) {
    typedef lsted::Fft2E<lsted::cplx<T>, DIR, RA, RC, 48> F;
    std::vector<lsted::cplx<T> > tw(F::L), sm(F::SEQ + 8);
    lsted::fill_twiddles<T>(F::L, tw.data());
    std::vector<std::vector<lsted::cplx<T> > > regs(48, std::vector<lsted::cplx<T> >(F::VREG));
    for (int t = 0; t < 48; ++t) {
        if (t < F::NA)
            for (int q = 0; q < F::RA; ++q)
                regs[t][q] = lsted::mk<T>((T)in[2 * (t + q * F::NA)], (T)in[2 * (t + q * F::NA) + 1]);
        F::pass_a(regs[t].data(), t, sm.data());
    }
    for (int t = 0; t < 48; ++t) {
        typename F::Tw w;
        F::load_tw(w, t, tw.data());
        F::pass_c(regs[t].data(), t, sm.data(), w);
        if (t < F::NC)
            for (int q = 0; q < F::RC; ++q) {
                out[2 * (t + q * F::NC)] = (double)regs[t][q].x;
                out[2 * (t + q * F::NC) + 1] = (double)regs[t][q].y;
            }
    }
}
extern "C" int emul_fft2_2160(int dir, int precision, const double* in, double* out) {
    if (precision == 32) { if (dir < 0) run_fft2<float, -1, 48, 45>(in, out); else run_fft2<float, +1, 45, 48>(in, out); }
    else { if (dir < 0) run_fft2<double, -1, 48, 45>(in, out); else run_fft2<double, +1, 45, 48>(in, out); }
    return 0;
}

// block order of the fused peer-memory reduction (conv_fast.cuh: p2p_block_at)
extern "C" int emul_p2p_block_at(int pos, int me, int world, int nxb) {
    return lsted::p2p_block_at(pos, me, world, nxb);
}

// Figure-3 scan engine and plane operators: the same element functors, run serially
// (OpenMP over elements where the build has it -- every element is independent).
#include "../../rescan_line_sted_b200/csrc/scan_kernels.cuh"
struct ScanHostBackend {
    std::vector<void*> live;
    explicit ScanHostBackend(int) {}
    ~ScanHostBackend() { for (void* p : live) ::free(p); }
    void activate() {}
    template <class T> T* alloc(size_t n) {
        void* p = calloc(n ? n : 1, sizeof(T));
        if (!p) throw std::bad_alloc();
        live.push_back(p);
        return (T*)p;
    }
    void free(void* p) {
        for (size_t i = 0; i < live.size(); ++i)
            if (live[i] == p) { live[i] = live.back(); live.pop_back(); break; }
        ::free(p);
    }
    void upload(void* d, const void* h, size_t bytes) { memcpy(d, h, bytes); }
    void download(void* h, const void* d, size_t bytes) { memcpy(h, d, bytes); }
    void copy(void* d, const void* s, size_t bytes) { memcpy(d, s, bytes); }
    void zero(void* d, size_t bytes) { memset(d, 0, bytes); }
    void sync() {}
    void timer_start() {}
    double timer_stop() { return 0.0; }
    template <class F> void for_each(size_t n, const F& f) {
#pragma omp parallel for schedule(static)
        for (long long e = 0; e < (long long)n; ++e) f((size_t)e);
    }
};
#define LSTED_SCAN_BACKEND ScanHostBackend
#include "../../rescan_line_sted_b200/csrc/api_scan.inl"
