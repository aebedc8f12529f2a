// Multi-view Richardson-Lucy engine: orchestration of the row/column passes
// of conv_bodies.cuh.  Templated on the storage precision T and on a
// Backend that owns memory and launches kernel bodies (CudaBackend in
// lsted_api.cu for the product; HostBackend in tests/host_emul for the
// CPU replay of the same bodies).
//
// State mirrors the attributes of the reference `Deconvolver`
// (figure_generation/line_sted_tools.py:478-594): psfs (as OTFs),
// true_object, noiseless_measurement[K], noisy_measurement[K], estimate,
// H_t_normalization.
#pragma once
#include <string>
#include <vector>
#include "plan.h"
#include "ew_bodies.cuh"

namespace lsted {

enum ArrayId {
    ARR_TRUE_OBJECT = 0,
    ARR_NOISELESS = 1,
    ARR_NOISY = 2,
    ARR_ESTIMATE = 3,
    ARR_NORMALIZATION = 4
};

// An image crossing the engine's boundary: host float64 (dtype 0, the host entry points) or a
// caller's device buffer of float32 / float64 (dtype 32 / 64, the _dev entry points).  Either
// way it passes through the engine's fp64 staging array: one host copy, or one conversion launch
// (ew_bodies.cuh stage_apply) that rounds like the host path.
struct ImageRef {
    void* p;
    int dtype;
    ImageRef at(size_t elems) const {
        ImageRef r = {(char*)p + elems * (dtype == 32 ? 4 : 8), dtype};
        return r;
    }
};
inline ImageRef host_image(const double* p) {
    ImageRef r = {(void*)p, 0};
    return r;
}
// caller buffer <-> fp64 staging: one element-wise launch (ew_bodies.cuh stage_apply)
template <int OP, typename U, class BK> void convert_stage(BK& bk, void* user, double* stage, size_t n) {
    EwArgs<U> a;
    memset(&a, 0, sizeof(a));
    if (OP == EW_TO_STAGE) { a.t1 = (const U*)user; a.d0 = stage; }
    else { a.t0 = (U*)user; a.d1 = stage; }
    a.elems = n;
    a.vec = ((uintptr_t)user & 15) == 0;
    a.n = stage_items<U>(n, a.vec != 0);
    bk.template ew<OP, U>(a);
}
// stage[0, n) <- src
template <class BK> void stage_in(BK& bk, double* stage, const ImageRef& src, size_t n) {
    if (src.dtype == 0) bk.upload(stage, src.p, sizeof(double) * n);
    else if (src.dtype == 32) convert_stage<EW_TO_STAGE, float>(bk, src.p, stage, n);
    else convert_stage<EW_TO_STAGE, double>(bk, src.p, stage, n);
}
// dst <- stage[0, n); a host destination is complete on return
template <class BK> void stage_out(BK& bk, const ImageRef& dst, double* stage, size_t n) {
    if (dst.dtype == 0) bk.download(dst.p, stage, sizeof(double) * n);
    else if (dst.dtype == 32) convert_stage<EW_FROM_STAGE, float>(bk, dst.p, stage, n);
    else convert_stage<EW_FROM_STAGE, double>(bk, dst.p, stage, n);
}

// Precision-independent face of an engine: what the C ABI talks to.
struct EngineInfo {
    int K, ny, nx, Ny, Nx, Ly, Lx, C, PR, iterations_done;
    size_t row_smem, col_smem;
    int tiles_y, tiles_x, tile_out_y, tile_out_x;   // 1 x 1 unless the object is tiled
    int band_y0, band_y1;                           // image rows owned by this rank (tiled + sharded)
    int band_x0, band_x1;                           // image columns owned by this rank
};
class EngineBase {
  public:
    virtual ~EngineBase() {}
    virtual void set_psfs(const double* psfs_host) = 0;
    virtual void upload_object(const ImageRef& obj) = 0;
    virtual void simulate(double total_brightness, bool rescale, unsigned long long seed) = 0;
    virtual void create_data(const double* obj_host, double total_brightness, bool rescale,
                             unsigned long long seed) = 0;
    virtual void iterate(int n) = 0;
    virtual void get_array(int id, int k, const ImageRef& out) = 0;
    virtual void set_array(int id, int k, const ImageRef& in) = 0;
    virtual void H(const ImageRef& x, const ImageRef& out) = 0;                    // out: K images
    virtual void Ht(const ImageRef& y, const ImageRef& out, bool normalize) = 0;   // y: K images
    virtual void forget_normalization() = 0;
    virtual void reset_estimate() = 0;     // the next iterate() starts from ones (ref:521-522)
    virtual void set_sharding(int rank, int world, int k_offset) = 0;
    virtual void set_exact_clip(bool on) = 0;
    virtual void options_changed() {}      // a kernel-selection switch moved: drop captured launches
    virtual void p2p_export(char* handles_out) = 0;                       // kIpcBytes
    virtual void p2p_attach(const char* all_handles) = 0;                 // [world][kIpcBytes]
    // NVLS reduction of orientation shards (fp32): see lsted.h / CudaBackend::nvls_*
    virtual int nvls_create(int) { throw std::string("the NVLS reduction needs an untiled fp32 handle"); }
    virtual void nvls_import(int, int) { throw std::string("the NVLS reduction needs an untiled fp32 handle"); }
    virtual void nvls_add_device() { throw std::string("the NVLS reduction needs an untiled fp32 handle"); }
    virtual void nvls_bind() { throw std::string("the NVLS reduction needs an untiled fp32 handle"); }
    virtual void info(EngineInfo* out) = 0;
    virtual bool ft_error(const double* image_host, double* out_host) = 0;
};

template <typename T, class BK> class DeconvEngine : public EngineBase {
  public:
    ConvGeom g;
    bool allow_centered, centered;   // centred real OTFs of point-symmetric PSFs (see OtfCenterArgs)
    T* otf_real;
    int sy0, sx0;                    // the 'same' crop offsets of the un-centred geometry
    int K, ny, nx;
    int iterations_done;
    bool have_norm, have_estimate, exact_clip;
    int rank, world, k_offset;

    DeconvEngine(BK& backend, int K_, int ny_, int nx_, int Ny, int Nx, int force_L = 0)
        : allow_centered(force_L == 0), centered(false), otf_real(0),
          K(K_), ny(ny_), nx(nx_), iterations_done(0), have_norm(false), have_estimate(false),
          exact_clip(false), rank(0), world(1), k_offset(0), bk(backend), tmpK(0), p2p_recv(0),
          p2p_flags(0), p2p_words(0), tmaps_tried(false), tmap_specK(0), tmap_spec1(0) {
        const char* why = make_geom(Ny, Nx, ny, nx, (int)sizeof(cplx<T>), &g, &BK::fast_cols, force_L);
        if (why[0]) throw std::string(why);
        npix = (size_t)Ny * Nx;
        sy0 = g.sy; sx0 = g.sx;
        std::vector<cplx<T> > tw;
        tw.resize(g.Lx); fill_twiddles<T>(g.Lx, tw.data());
        tw_x = (cplx<T>*)bk.alloc(sizeof(cplx<T>) * g.Lx);
        bk.upload(tw_x, tw.data(), sizeof(cplx<T>) * g.Lx);
        tw.resize(g.Ly); fill_twiddles<T>(g.Ly, tw.data());
        tw_y = (cplx<T>*)bk.alloc(sizeof(cplx<T>) * g.Ly);
        bk.upload(tw_y, tw.data(), sizeof(cplx<T>) * g.Ly);
        otf = (cplx<T>*)bk.alloc(sizeof(cplx<T>) * otf_elems(g) * K);
        spec1 = (cplx<T>*)bk.alloc(sizeof(cplx<T>) * spec_elems(g, g.Ny));
        specK = (cplx<T>*)bk.alloc(sizeof(cplx<T>) * spec_elems(g, g.Ny) * K);
        true_object = (T*)bk.alloc(sizeof(T) * npix);
        estimate = (T*)bk.alloc(sizeof(T) * npix);
        norm = (T*)bk.alloc(sizeof(T) * npix);
        scratch = (T*)bk.alloc(sizeof(T) * npix);
        noiseless = (T*)bk.alloc(sizeof(T) * npix * K);
        noisy = (T*)bk.alloc(sizeof(T) * npix * K);
        stage64 = (double*)bk.alloc(sizeof(double) * npix * K);
        object64 = (double*)bk.alloc(sizeof(double) * npix);
        partial = (double*)bk.alloc(sizeof(double) * kReduceBlocks);
    }
    ~DeconvEngine() {
        options_changed();
        void* all[] = {tw_x, tw_y, otf, spec1, specK, true_object, estimate, norm,
                       scratch, noiseless, noisy, stage64, object64, partial, tmpK, p2p_recv, p2p_flags,
                       otf_real, tmap_specK, tmap_spec1, tw_fx, tw_fy, spec_ft, tw_dx, tw_dy, spec_direct};
        for (size_t i = 0; i < sizeof(all) / sizeof(all[0]); ++i) bk.free(all[i]);
    }

    size_t pixels() const { return npix; }
    void set_exact_clip(bool on) { exact_clip = on; }
    void info(EngineInfo* o) {
        memset(o, 0, sizeof(*o));
        o->K = K; o->ny = ny; o->nx = nx; o->Ny = g.Ny; o->Nx = g.Nx; o->Ly = g.Ly; o->Lx = g.Lx;
        o->C = g.C; o->PR = g.PR; o->iterations_done = iterations_done;
        o->row_smem = row_smem_bytes(g, (int)sizeof(cplx<T>));
        o->col_smem = col_smem_bytes(g, (int)sizeof(cplx<T>));
        o->tiles_y = o->tiles_x = 1; o->tile_out_y = g.Ny; o->tile_out_x = g.Nx;
        o->band_y0 = 0; o->band_y1 = g.Ny;
        o->band_x0 = 0; o->band_x1 = g.Nx;
    }

    // K7: PSFs (host, float64, [K][ny][nx]) -> OTFs, 1/(Lx*Ly) folded in.
    void set_psfs(const double* psfs_host) {
        options_changed();
        const size_t n = (size_t)K * ny * nx;
        double* d64 = (double*)bk.alloc(sizeof(double) * n);
        T* dT = (T*)bk.alloc(sizeof(T) * n);
        bk.upload(d64, psfs_host, sizeof(double) * n);
        bk.cast_in(dT, d64, n, 1.0);
        ConvGeom gp = g;  // same transform lengths, image := PSF
        gp.Ny = ny; gp.Nx = nx;
        cplx<T>* rows = (cplx<T>*)bk.alloc(sizeof(cplx<T>) * spec_elems(gp, ny) * K);
        RowArgs<T> ra = row_args(gp);
        ra.nimg = K; ra.real_in = dT; ra.spec_out = rows;
        bk.template launch_row<ROW_FWD, T>(row_blocks(gp) * K, ra);
        ColArgs<T> ca = col_args(gp);
        ca.src = rows; ca.dst = otf; ca.K = K; ca.rows_in = ny;
        ca.scale = (T)(1.0 / ((double)g.Lx * (double)g.Ly));
        bk.template launch_col<COL_OTF, T>(g.nxb * K, ca);
        // Point-symmetric PSFs (every PSF the reference builds is): store the OTFs centred, as
        // real numbers, and drop the crop offsets from the geometry.  Only where the
        // compile-time column plan (which reads the real array) exists, and not inside tiles.
        g.sy = sy0; g.sx = sx0;
        centered = allow_centered && bk.real_otf_supported(g, (int)sizeof(cplx<T>)) &&
                   point_symmetric(psfs_host);
        if (centered) {
            if (!otf_real) otf_real = (T*)bk.alloc(sizeof(T) * otf_elems(g) * K);
            OtfCenterArgs<T> oc;
            oc.otf = otf; oc.otf_real = otf_real; oc.tw_y = tw_y; oc.tw_x = tw_x;
            oc.nxb = g.nxb; oc.Ly = g.Ly; oc.Lx = g.Lx; oc.C = g.C; oc.CS = g.C;
            oc.cy = (ny - 1) / 2; oc.cx = (nx - 1) / 2;
            oc.n = otf_elems(g) * K;
            bk.otf_center(oc);
            g.sy = 0; g.sx = 0;
        }
        bk.sync();
        bk.free(rows); bk.free(dT); bk.free(d64);
        have_norm = false;
    }
    // psf[c + a] == psf[c - a] for every PSF (odd sizes only), to 1e-12 of the peak
    bool point_symmetric(const double* psfs_host) const {
        if (ny % 2 == 0 || nx % 2 == 0) return false;
        const size_t n = (size_t)ny * nx;
        for (int k = 0; k < K; ++k) {
            const double* p = psfs_host + n * k;
            double peak = 0, worst = 0;
            for (size_t i = 0; i < n; ++i) {
                const double a = p[i] < 0 ? -p[i] : p[i];
                const double d = p[i] - p[n - 1 - i];
                if (a > peak) peak = a;
                if ((d < 0 ? -d : d) > worst) worst = (d < 0 ? -d : d);
            }
            if (!(worst <= 1e-12 * peak)) return false;
        }
        return true;
    }

    // ---- operators on device arrays ------------------------------------
    // H: x[Ny][Nx] -> out[K][Ny][Nx] (clipped); optional Poisson copy.
    void op_H(const T* x, T* out, T* out_noisy, unsigned long long seed) {
        RowArgs<T> ra = row_args(g);
        ra.nimg = 1; ra.real_in = x; ra.spec_out = spec1;
        bk.template launch_row<ROW_FWD, T>(row_blocks(g), ra);
        ColArgs<T> ca = col_args(g);
        ca.src = spec1; ca.dst = specK; ca.K = K;
        bk.template launch_col<COL_H, T>(g.nxb, ca);
        RowArgs<T> rb = row_args(g);
        rb.nimg = K; rb.spec_in = specK; rb.real_out = out; rb.clip = 1;
        if (out_noisy) {
            rb.real_out2 = out_noisy; rb.seed = seed; rb.img0 = (unsigned)k_offset;
            bk.template launch_row<ROW_INV_SIM, T>(row_blocks(g) * K, rb);
        } else {
            bk.template launch_row<ROW_INV_STORE, T>(row_blocks(g) * K, rb);
        }
    }

    // H_t without normalisation: y[K][Ny][Nx] -> out[Ny][Nx].
    // Default: products summed in the Fourier domain, one inverse transform,
    // clip after the sum.  exact_clip: inverse-transform and clip each term
    // before summing, like the reference loop (line_sted_tools.py:585-588).
    void op_Ht_raw(const T* y, T* out) {
        RowArgs<T> ra = row_args(g);
        ra.nimg = K; ra.real_in = y; ra.spec_out = specK;
        bk.template launch_row<ROW_FWD, T>(row_blocks(g) * K, ra);
        ht_from_specK(out);
    }

    // ---- Deconvolver methods ---------------------------------------------
    void upload_object(const ImageRef& obj) { stage_in(bk, object64, obj, npix); }
    // Forward model + shot noise from the object staged by upload_object().
    void simulate(double total_brightness, bool rescale, unsigned long long seed) {
        double s = 1.0;
        if (rescale) s = total_brightness / bk.sum(object64, npix, partial);
        bk.cast_in(true_object, object64, npix, s);
        op_H(true_object, noiseless, noisy, seed);
        // like the reference (ref:496-512) new data leave the estimate alone: the caller
        // decides whether the next iterate() restarts from ones (reset_estimate)
        invalidate_estimate_spectrum();   // op_H went through spec1
    }
    void create_data(const double* obj_host, double total_brightness, bool rescale,
                     unsigned long long seed) {
        upload_object(host_image(obj_host));
        simulate(total_brightness, rescale, seed);
    }
    void forget_normalization() { have_norm = false; }
    void reset_estimate() { have_estimate = false; iterations_done = 0; }
    // tensor maps of the two row-spectrum arrays (fp32 fast rows): see fft_core.cuh tma_load_chunks
    void ensure_tmaps() {
        if (tmaps_tried) return;
        tmaps_tried = true;
        if (!bk.row_tma_supported(g, (int)sizeof(cplx<T>))) return;
        const int chunk_floats = 2 * 1 * g.C * 2;   // 2 rows x C columns x (re, im), one pair per CTA
        tmap_specK = bk.make_spec_tmap(specK, even_rows(g.Ny), g.nxb, g.C, K, chunk_floats);
        tmap_spec1 = bk.make_spec_tmap(spec1, even_rows(g.Ny), g.nxb, g.C, 1, chunk_floats);
        if (!tmap_specK || !tmap_spec1) tmap_specK = tmap_spec1 = 0;
    }

    // Orientation sharding (SURVEY.md 8e): this handle owns `K` of the orientations
    // (global indices k_offset .. k_offset+K-1) plus replicas of the estimate and
    // the normalisation; the Fourier-domain partial sums of H_t are all-reduced
    // over `world` ranks once per iteration (the transforms are linear, so summing
    // spectra equals summing images) and everything else stays local.
    void set_sharding(int rank_, int world_, int k_offset_) {
        rank = rank_; world = world_; k_offset = k_offset_;
        have_norm = false;
        options_changed();
    }
    // Fused cross-GPU H_t reduction (fast path only): receive slabs for the partial sums of
    // every (source rank, column block) and the flag / counter words, exported to the peers.
    void p2p_export(char* out) {
        if (world < 2) throw std::string("p2p_export: shard the handle first");
        if (!p2p_recv) {
            const size_t part = (size_t)g.C * g.Ly + (size_t)g.C * g.Ly / 8 + 64;   // register pairs, padded
            p2p_recv = (cplx<T>*)bk.alloc(sizeof(cplx<T>) * part * g.nxb * world);
            p2p_words = (size_t)world * g.nxb;
            p2p_flags = (unsigned*)bk.alloc(sizeof(unsigned) * (p2p_words + 32));
            bk.zero_bytes(p2p_flags, sizeof(unsigned) * (p2p_words + 32));
            bk.sync();
        }
        bk.p2p_export(p2p_recv, p2p_flags, spec1, out);
    }
    void p2p_attach(const char* all) { bk.p2p_attach(rank, world, all, p2p_words); }
    void reduce_over_ranks(cplx<T>* spec) {
        if (world < 2) return;
        if (bk.nvls_ready(spec)) bk.nvls_allreduce((T*)spec, 2 * spec_elems(g, g.Ny));   // through the switch
        else bk.all_reduce_sum((T*)spec, 2 * spec_elems(g, g.Ny));
    }
    // NVLS: the spectrum that carries the partial H_t sums moves into memory bound to a CUDA
    // multicast object shared by the ranks (call before any data is on the handle)
    int nvls_create(int world_) {
        if (sizeof(T) != 4) throw std::string("the NVLS reduction is built for fp32 spectra");
        return bk.nvls_create(world_, sizeof(cplx<T>) * spec_elems(g, g.Ny));
    }
    void nvls_import(int world_, int fd) {
        if (sizeof(T) != 4) throw std::string("the NVLS reduction is built for fp32 spectra");
        bk.nvls_import(world_, sizeof(cplx<T>) * spec_elems(g, g.Ny), fd);
    }
    void nvls_add_device() { bk.nvls_add_device(); }
    void nvls_bind() {
        if (world < 2) throw std::string("nvls_bind: shard the handle first");
        cplx<T>* region = (cplx<T>*)bk.nvls_bind(rank);
        bk.sync();
        bk.free(spec1);
        spec1 = region;
        if (tmap_spec1) { bk.free(tmap_spec1); bk.free(tmap_specK); tmap_spec1 = tmap_specK = 0; }
        tmaps_tried = false;
        have_estimate = false; have_norm = false;
        options_changed();
    }

    // The steady-state RL iteration is four launches with fixed arguments.  For small objects
    // (the reference's own 128^2 / 160^2 frames) launch overhead is most of an iterate() call, so
    // after one plain pass (lazy attribute / tensor-map set-up) the four launches are captured
    // into a CUDA graph and replayed -- one driver call per iteration.  Any option change,
    // new PSFs or sharding drops the graph.
    void* iter_graph = 0;
    int steady_passes = 0;
    void options_changed() {
        if (iter_graph) { bk.graph_destroy(iter_graph); iter_graph = 0; }
        steady_passes = 0;
    }
    void launch_steady_iteration() {
        // expected = H(estimate); ratio = measurement / expected -> row spectra
        ColArgs<T> ca = col_args(g);
        ca.src = spec1; ca.dst = specK; ca.K = K;
        bk.template launch_col<COL_H, T>(g.nxb, ca);
        RowArgs<T> rm = row_args(g);
        rm.nimg = K; rm.spec_in = specK; rm.spec_out = specK; rm.aux = noisy;
        rm.tmap_in = rm.tmap_out = tmap_specK;
        bk.template launch_row<ROW_MID, T>(row_blocks(g) * K, rm);
        ColArgs<T> ct = col_args(g);
        ct.src = specK; ct.dst = spec1; ct.K = K;
        if (world > 1 && !bk.nvls_ready(spec1) && bk.p2p_ready(g, (int)sizeof(cplx<T>))) {
            // orientation shards: the sum over ranks happens inside the kernel (peer memory)
            bk.p2p_fill(ct);
            bk.template launch_col<COL_HT, T>(g.nxb, ct);
            bk.p2p_wait(g.nxb);
        } else {
            bk.template launch_col<COL_HT, T>(g.nxb, ct);
            reduce_over_ranks(spec1);   // orientation shards: NCCL sum of partial spectra
        }
        RowArgs<T> rf = row_args(g);
        rf.nimg = 1; rf.spec_in = spec1; rf.spec_out = spec1;
        rf.real_out = estimate; rf.aux = norm;
        rf.tmap_in = rf.tmap_out = tmap_spec1;
        rf.prefetch_ahead = bk.row_final_prefetch_distance();
        bk.template launch_row<ROW_FINAL, T>(row_blocks(g), rf);
    }

    void iterate(int n) {
        for (int it = 0; it < n; ++it) {
            ensure_norm();
            if (!have_estimate) {
                bk.fill(estimate, npix, (T)1);
                RowArgs<T> ra = row_args(g);
                ra.nimg = 1; ra.real_in = estimate; ra.spec_out = spec1;
                bk.template launch_row<ROW_FWD, T>(row_blocks(g), ra);
                have_estimate = true;
            }
            if (!exact_clip) {
                ensure_tmaps();
                if (world == 1 && bk.graph_capable()) {
                    if (!iter_graph && steady_passes >= 1) {
                        bk.graph_begin();
                        try { launch_steady_iteration(); }
                        catch (...) { bk.graph_abort(); throw; }
                        iter_graph = bk.graph_end();
                    }
                    if (iter_graph) bk.graph_launch(iter_graph);
                    else launch_steady_iteration();
                    ++steady_passes;
                } else {
                    launch_steady_iteration();
                }
            } else {
                ColArgs<T> ca = col_args(g);
                ca.src = spec1; ca.dst = specK; ca.K = K;
                bk.template launch_col<COL_H, T>(g.nxb, ca);
                ensure_tmaps();
                RowArgs<T> rm = row_args(g);
                rm.nimg = K; rm.spec_in = specK; rm.spec_out = specK; rm.aux = noisy;
                rm.tmap_in = rm.tmap_out = tmap_specK;
                bk.template launch_row<ROW_MID, T>(row_blocks(g) * K, rm);
                ht_from_specK(scratch);
                bk.rl_update(estimate, scratch, norm, npix);
                RowArgs<T> ra = row_args(g);
                ra.nimg = 1; ra.real_in = estimate; ra.spec_out = spec1;
                bk.template launch_row<ROW_FWD, T>(row_blocks(g), ra);
            }
            ++iterations_done;
        }
    }

    // The estimate spectrum cached in spec1 goes stale when anything else
    // uses spec1 or when the caller overwrites the estimate.
    void invalidate_estimate_spectrum() {
        if (!have_estimate) return;
        RowArgs<T> ra = row_args(g);
        ra.nimg = 1; ra.real_in = estimate; ra.spec_out = spec1;
        bk.template launch_row<ROW_FWD, T>(row_blocks(g), ra);
    }

    T* array(int id, int k) {
        switch (id) {
            case ARR_TRUE_OBJECT: return true_object;
            case ARR_NOISELESS: return noiseless + npix * k;
            case ARR_NOISY: return noisy + npix * k;
            case ARR_ESTIMATE: return estimate;
            case ARR_NORMALIZATION: return norm;
        }
        return 0;
    }

    void get_array(int id, int k, const ImageRef& out) {
        if (id == ARR_NORMALIZATION) ensure_norm();
        bk.cast_out(stage64, array(id, k), npix);
        stage_out(bk, out, stage64, npix);
    }
    void set_array(int id, int k, const ImageRef& in) {
        stage_in(bk, stage64, in, npix);
        bk.cast_in(array(id, k), stage64, npix, 1.0);
        if (id == ARR_ESTIMATE) { have_estimate = true; invalidate_estimate_spectrum(); }
        if (id == ARR_NORMALIZATION) have_norm = true;
    }

    // record_iteration's error spectrum (ref:539-546): log(1 + |fftshift(fft2(x - true_object))|)
    // with x = the estimate in HBM (image_host == 0) or a host image.  An un-padded Ny x Nx
    // transform with the generic kernels; when a side is not 2^a 3^b 5^c (or does not fit a
    // CTA) the direct transform of ew_bodies.cuh (dft_direct_apply) does it instead -- always
    // on the device, always true.
    bool ft_error(const double* image_host, double* out_host) {
        if (!ft_tried) {
            ft_tried = true;
            const char* why = make_geom(g.Ny, g.Nx, 1, 1, (int)sizeof(cplx<T>), &gft);
            ft_ok = !why[0] && gft.Ly == g.Ny && gft.Lx == g.Nx;
            if (ft_ok) {
                std::vector<cplx<T> > tw;
                tw.resize(gft.Lx); fill_twiddles<T>(gft.Lx, tw.data());
                tw_fx = (cplx<T>*)bk.alloc(sizeof(cplx<T>) * gft.Lx);
                bk.upload(tw_fx, tw.data(), sizeof(cplx<T>) * gft.Lx);
                tw.resize(gft.Ly); fill_twiddles<T>(gft.Ly, tw.data());
                tw_fy = (cplx<T>*)bk.alloc(sizeof(cplx<T>) * gft.Ly);
                bk.upload(tw_fy, tw.data(), sizeof(cplx<T>) * gft.Ly);
                spec_ft = (cplx<T>*)bk.alloc(sizeof(cplx<T>) * spec_elems(gft, gft.Ny));
                bk.sync();
            } else {
                std::vector<cplx<double> > tw;
                tw.resize(g.Nx); fill_twiddles<double>(g.Nx, tw.data());
                tw_dx = (cplx<double>*)bk.alloc(sizeof(cplx<double>) * g.Nx);
                bk.upload(tw_dx, tw.data(), sizeof(cplx<double>) * g.Nx);
                tw.resize(g.Ny); fill_twiddles<double>(g.Ny, tw.data());
                tw_dy = (cplx<double>*)bk.alloc(sizeof(cplx<double>) * g.Ny);
                bk.upload(tw_dy, tw.data(), sizeof(cplx<double>) * g.Ny);
                spec_direct = (cplx<double>*)bk.alloc(sizeof(cplx<double>) * npix);
                bk.sync();
            }
        }
        const T* x = estimate;
        if (image_host) {
            bk.upload(stage64, image_host, sizeof(double) * npix);
            bk.cast_in(scratch, stage64, npix, 1.0);
            x = scratch;
        }
        bk.subtract(scratch, x, true_object, npix);
        if (!ft_ok) {
            DftArgs<T> da;
            memset(&da, 0, sizeof(da));
            da.real_in = scratch; da.spec = spec_direct; da.twx = tw_dx; da.twy = tw_dy;
            da.logmag = stage64; da.Ny = g.Ny; da.Nx = g.Nx;
            bk.template dft_direct<0, T>(da);
            bk.template dft_direct<1, T>(da);
            bk.download(out_host, stage64, sizeof(double) * npix);
            return true;
        }
        RowArgs<T> ra;
        memset(&ra, 0, sizeof(ra));
        ra.g = gft; ra.tw = tw_fx; ra.nimg = 1; ra.real_in = scratch; ra.spec_out = spec_ft;
        bk.template launch_row<ROW_FWD, T>(row_blocks(gft), ra);
        ColArgs<T> ca;
        memset(&ca, 0, sizeof(ca));
        ca.g = gft; ca.tw = tw_fy; ca.src = spec_ft; ca.K = 1; ca.rows_in = gft.Ny; ca.logmag = stage64;
        bk.launch_col_logmag(gft.nxb, ca);
        bk.download(out_host, stage64, sizeof(double) * npix);
        return true;
    }

    // H / H_t of the Python methods, on host arrays or caller device buffers.
    void H(const ImageRef& x, const ImageRef& out) {
        stage_in(bk, stage64, x, npix);
        bk.cast_in(scratch, stage64, npix, 1.0);
        T* tmp = tmp_images();
        op_H(scratch, tmp, 0, 0);
        bk.cast_out(stage64, tmp, npix * K);
        stage_out(bk, out, stage64, npix * K);
        invalidate_estimate_spectrum();
    }
    void Ht(const ImageRef& y, const ImageRef& out, bool normalize) {
        T* tmp = tmp_images();
        if (normalize) ensure_norm();
        stage_in(bk, stage64, y, npix * K);
        bk.cast_in(tmp, stage64, npix * K, 1.0);
        op_Ht_raw(tmp, scratch);
        if (normalize) bk.divide(scratch, norm, npix);
        bk.cast_out(stage64, scratch, npix);
        stage_out(bk, out, stage64, npix);
        invalidate_estimate_spectrum();
    }

  private:
    enum { kReduceBlocks = 1024 };
    BK& bk;
    size_t npix;
    cplx<T>*tw_x, *tw_y, *otf, *spec1, *specK;
    T *true_object, *estimate, *norm, *scratch, *noiseless, *noisy;
    double *stage64, *object64, *partial;
    ConvGeom gft;                       // un-padded transform of the error spectrum (ft_error)
    bool ft_tried = false, ft_ok = false;
    cplx<T>*tw_fx = 0, *tw_fy = 0, *spec_ft = 0;
    cplx<double>*tw_dx = 0, *tw_dy = 0, *spec_direct = 0;   // direct transform (sides without a plan)
    T* tmpK;  // K images, allocated on first use by the host-array forms of H / H_t
    cplx<T>* p2p_recv; unsigned* p2p_flags; size_t p2p_words;
    bool tmaps_tried; void* tmap_specK; void* tmap_spec1;
    T* tmp_images() {
        if (!tmpK) tmpK = (T*)bk.alloc(sizeof(T) * npix * K);
        return tmpK;
    }

    RowArgs<T> row_args(const ConvGeom& gg) {
        RowArgs<T> a;
        memset(&a, 0, sizeof(a));
        a.g = gg; a.tw = tw_x;
        a.prefetch_ahead = bk.row_prefetch_distance();
        return a;
    }
    ColArgs<T> col_args(const ConvGeom& gg) {
        ColArgs<T> a;
        memset(&a, 0, sizeof(a));
        a.g = gg; a.tw = tw_y; a.otf = otf; a.rows_in = gg.Ny; a.scale = (T)1;
        a.otf_real = centered ? otf_real : 0;
        return a;
    }
    // specK holds K row-spectra -> out = sum_k conv_k (spec1 is clobbered)
    void ht_from_specK(T* out, bool same_input = false) {
        if (!exact_clip) {
            ColArgs<T> ct = col_args(g);
            ct.src = specK; ct.dst = spec1; ct.K = K; ct.src_same = same_input;
            bk.template launch_col<COL_HT, T>(g.nxb, ct);
            reduce_over_ranks(spec1);
            RowArgs<T> rb = row_args(g);
            rb.nimg = 1; rb.spec_in = spec1; rb.real_out = out; rb.clip = 1;
            bk.template launch_row<ROW_INV_STORE, T>(row_blocks(g), rb);
        } else {
            // one orientation at a time: product, inverse, clip, accumulate
            for (int k = 0; k < K; ++k) {
                ColArgs<T> ct = col_args(g);
                ct.src = specK + (same_input ? 0 : spec_elems(g, g.Ny) * k);
                ct.otf = otf + otf_elems(g) * k;
                if (centered) ct.otf_real = otf_real + otf_elems(g) * k;
                ct.dst = spec1; ct.K = 1;
                bk.template launch_col<COL_HT, T>(g.nxb, ct);
                RowArgs<T> rb = row_args(g);
                rb.nimg = 1; rb.spec_in = spec1; rb.real_out = out; rb.clip = 1;
                rb.accumulate = (k > 0);
                bk.template launch_row<ROW_INV_STORE, T>(row_blocks(g), rb);
            }
            // every term was clipped locally; the sum over ranks is a plain image sum
            if (world > 1) bk.all_reduce_sum(out, npix);
        }
    }
  public:
    // H_t_normalization = H_t(ones, normalize=False) (line_sted_tools.py:589-593)
    void ensure_norm() {
        if (have_norm) return;
        // All K inputs are the same all-ones image: one row pass, shared by every k,
        // and no temporary allocation (cudaMalloc/cudaFree would serialise the stream).
        bk.fill(scratch, npix, (T)1);
        RowArgs<T> ra = row_args(g);
        ra.nimg = 1; ra.real_in = scratch; ra.spec_out = specK;
        bk.template launch_row<ROW_FWD, T>(row_blocks(g), ra);
        ht_from_specK(norm, true);
        have_norm = true;
        invalidate_estimate_spectrum();  // op_Ht_raw clobbered spec1
    }
};

}  // namespace lsted
