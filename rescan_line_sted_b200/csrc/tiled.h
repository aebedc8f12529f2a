// Overlap-save tiling of the convolution engine for objects whose padded
// transform does not fit a CTA's shared memory (BASELINE config 5: 8192^2).
//
// The object is cut into tiles; each tile is convolved through a W x W window
// (W = the tile FFT length, 2160 by default so the compile-time plan applies)
// that carries the (n-1)-pixel halo, zero-filled outside the object exactly like
// the reference's linear 'same' convolution; only the alias-free interior
// W - (n-1) of a window is written back.  H and H_t therefore equal the
// untiled operators (tests compare them), and one RL iteration becomes two
// sweeps over the tiles: ratio = measurement / H(estimate), then
// estimate *= H_t(ratio) / norm (the ratio is materialised because its halo
// comes from the neighbouring tiles).
//
// Mirrors Deconvolver (figure_generation/line_sted_tools.py:478-594) like
// DeconvEngine does; full-size arrays live in HBM (3 x K x Ny x Nx elements
// for measurements and ratios: 52 GB at 8192^2, K = 32, fp64).
//
// Sharding over GPUs (SURVEY.md 8e, "object tiles with halo"): the TILES are dealt to a
// gy x gx grid of ranks (4 x 4 tiles of 8192^2 over 8 ranks: a 2 x 4 grid, two tiles each), so
// every rank sweeps only whole windows of its own -- 1/world of the single-GPU work.  A rank
// keeps measurements and ratios on its rectangle of the image; what its windows read beyond
// that rectangle -- the estimate and the K ratio images on a PSF-halo-wide ring (53 px for the
// 107^2 PSFs) -- arrives from the ranks owning those pixels: two halo exchanges per RL
// iteration (grouped ncclSend / ncclRecv of packed strips to the <= 8 neighbours).  Exchanging
// the ratio ring instead of recomputing it keeps the window count minimal: a rectangle grown
// by the halo no longer fits its windows' alias-free interiors, so recomputing would cost
// every rank an extra, almost empty row and column of windows (3 x 2 instead of 2 x 1).
#pragma once
#include "engine.h"
#include "ew_bodies.cuh"

namespace lsted {

template <typename T, class BK> class TiledEngine : public EngineBase {
  public:
    struct Rect {
        int y0, y1, x0, x1;
        bool empty() const { return y1 <= y0 || x1 <= x0; }
        int h() const { return y1 - y0; }
        int w() const { return x1 - x0; }
        size_t area() const { return empty() ? 0 : (size_t)h() * w(); }
    };
    static Rect intersect(const Rect& a, const Rect& b) {
        Rect r = {a.y0 > b.y0 ? a.y0 : b.y0, a.y1 < b.y1 ? a.y1 : b.y1,
                  a.x0 > b.x0 ? a.x0 : b.x0, a.x1 < b.x1 ? a.x1 : b.x1};
        return r;
    }

    TiledEngine(BK& backend, int K_, int ny_, int nx_, int Ny_, int Nx_, int tile_L)
        : K(K_), ny(ny_), nx(nx_), Ny(Ny_), Nx(Nx_), W(tile_L), iterations_done(0),
          have_norm(false), have_estimate(false), bk(backend),
          tile(backend, K_, ny_, nx_, tile_L, tile_L, tile_L) {
        if (W - (ny - 1) < 1 || W - (nx - 1) < 1) throw std::string("tile FFT length shorter than the PSF");
        sy = (ny - 1) / 2; sx = (nx - 1) / 2;
        iy0 = ny - 1 - sy; ix0 = nx - 1 - sx;     // first alias-free output of a window
        out_y = W - (ny - 1); out_x = W - (nx - 1);
        tiles_y = (Ny + out_y - 1) / out_y; tiles_x = (Nx + out_x - 1) / out_x;
        npix = (size_t)Ny * Nx;
        wpix = (size_t)W * W;
        rank = 0; world = 1;
        true_object = (T*)bk.alloc(sizeof(T) * npix);
        estimate = (T*)bk.alloc(sizeof(T) * npix);
        norm = (T*)bk.alloc(sizeof(T) * npix);
        noiseless = noisy = ratio = 0;
        halo_send = halo_recv = 0;
        stage_region = 0;
        set_region(0, 1);
        win1 = (T*)bk.alloc(sizeof(T) * wpix);
        win2 = (T*)bk.alloc(sizeof(T) * wpix);
        winK = (T*)bk.alloc(sizeof(T) * wpix * K);
        stage64 = (double*)bk.alloc(sizeof(double) * npix);
        object64 = (double*)bk.alloc(sizeof(double) * npix);
        partial = (double*)bk.alloc(sizeof(double) * 1024);
    }
    ~TiledEngine() {
        void* all[] = {true_object, estimate, norm, noiseless, noisy, ratio, win1, win2, winK,
                       stage64, object64, partial, halo_send, halo_recv, stage_region,
                       tmp1, tw_dx, tw_dy, spec_direct};
        for (size_t i = 0; i < sizeof(all) / sizeof(all[0]); ++i) bk.free(all[i]);
    }

    void set_psfs(const double* psfs_host) { tile.set_psfs(psfs_host); have_norm = false; }
    void set_exact_clip(bool on) { tile.set_exact_clip(on); have_norm = false; }
    void p2p_export(char*) { throw std::string("the peer-memory reduction applies to orientation sharding, not to tiles"); }
    void p2p_attach(const char*) { throw std::string("the peer-memory reduction applies to orientation sharding, not to tiles"); }
    void forget_normalization() { have_norm = false; }
    void reset_estimate() { have_estimate = false; iterations_done = 0; }

    // ---- regions ----
    static void split(int n, int r, int parts, int* a, int* b) {
        const int base = n / parts, extra = n % parts;
        *a = r * base + (r < extra ? r : extra);
        *b = *a + base + (r < extra ? 1 : 0);
    }
    // rank grid gy x gx = world with the fewest windows on the busiest rank; ties: the squarer
    // regions (shorter halo ring)
    static void choose_grid(int world, int tiles_y, int tiles_x, int* gy, int* gx) {
        long best = -1, best_ring = 0;
        for (int a = 1; a <= world; ++a) {
            if (world % a) continue;
            const int b = world / a;
            if (a > tiles_y || b > tiles_x) continue;
            const int my = (tiles_y + a - 1) / a, mx = (tiles_x + b - 1) / b;
            const long cost = (long)my * mx, ring = my + mx;
            if (best < 0 || cost < best || (cost == best && ring < best_ring)) {
                best = cost; best_ring = ring; *gy = a; *gx = b;
            }
        }
        if (best < 0) throw std::string("more ranks than tiles: no rank grid fits the tile grid");
    }
    Rect owned_of(int r) const {
        int ta, tb, ua, ub;
        split(tiles_y, r / grid_x, grid_y, &ta, &tb);
        split(tiles_x, r % grid_x, grid_x, &ua, &ub);
        Rect o = {ta * out_y, tb * out_y < Ny ? tb * out_y : Ny, ua * out_x, ub * out_x < Nx ? ub * out_x : Nx};
        return o;
    }
    Rect extended_of(int r) const {
        if (world == 1) { Rect all = {0, Ny, 0, Nx}; return all; }
        // what the windows of the owned tiles read: the tiles grown by the PSF halo
        const int hy = sy > ny - 1 - sy ? sy : ny - 1 - sy, hx = sx > nx - 1 - sx ? sx : nx - 1 - sx;
        const Rect o = owned_of(r);
        Rect e = {o.y0 - hy < 0 ? 0 : o.y0 - hy, o.y1 + hy > Ny ? Ny : o.y1 + hy,
                  o.x0 - hx < 0 ? 0 : o.x0 - hx, o.x1 + hx > Nx ? Nx : o.x1 + hx};
        return e;
    }
    void set_sharding(int rank_, int world_, int) { set_region(rank_, world_); }
    void set_region(int rank_, int world_) {
        rank = rank_; world = world_;
        grid_y = grid_x = 1;
        if (world > 1) choose_grid(world, tiles_y, tiles_x, &grid_y, &grid_x);
        O = owned_of(rank);
        E = extended_of(rank);
        split(tiles_y, rank / grid_x, grid_y, &ty0, &ty1);
        split(tiles_x, rank % grid_x, grid_x, &tx0, &tx1);
        bpix = E.area();
        bk.sync();
        bk.free(noiseless); bk.free(noisy); bk.free(ratio);
        bk.free(halo_send); bk.free(halo_recv); bk.free(stage_region);
        noiseless = (T*)bk.alloc(sizeof(T) * bpix * K);
        noisy = (T*)bk.alloc(sizeof(T) * bpix * K);
        ratio = (T*)bk.alloc(sizeof(T) * bpix * K);
        stage_region = (double*)bk.alloc(sizeof(double) * bpix);
        // halo strips: what this rank owns of a neighbour's extended rectangle goes out, what a
        // neighbour owns of this rank's extended rectangle comes in
        peers.clear(); send_rect.clear(); recv_rect.clear();
        size_t total_send = 0, total_recv = 0;
        for (int q = 0; q < world; ++q) {
            if (q == rank) continue;
            const Rect s = intersect(O, extended_of(q)), r = intersect(E, owned_of(q));
            if (s.empty() && r.empty()) continue;
            peers.push_back(q); send_rect.push_back(s); recv_rect.push_back(r);
            total_send += s.area(); total_recv += r.area();
        }
        halo_send = (T*)bk.alloc(sizeof(T) * total_send * K);
        halo_recv = (T*)bk.alloc(sizeof(T) * total_recv * K);
        halo_pixels = total_recv;
        have_norm = false; have_estimate = false;
    }
    // record_iteration's error spectrum of a tiled object: the direct transform of
    // ew_bodies.cuh over the whole image (a tiled object's sides have no single-CTA plan).
    // A rank of a sharded object holds only its region of the estimate: false without a host
    // image there (the caller passes the gathered estimate instead).
    bool ft_error(const double* image_host, double* out_host) {
        if (!image_host && world > 1) return false;
        if (!spec_direct) {
            std::vector<cplx<double> > tw;
            tw.resize(Nx); fill_twiddles<double>(Nx, tw.data());
            tw_dx = (cplx<double>*)bk.alloc(sizeof(cplx<double>) * Nx);
            bk.upload(tw_dx, tw.data(), sizeof(cplx<double>) * Nx);
            tw.resize(Ny); fill_twiddles<double>(Ny, tw.data());
            tw_dy = (cplx<double>*)bk.alloc(sizeof(cplx<double>) * Ny);
            bk.upload(tw_dy, tw.data(), sizeof(cplx<double>) * Ny);
            spec_direct = (cplx<double>*)bk.alloc(sizeof(cplx<double>) * npix);
            bk.sync();
        }
        T* diff = image_tmp();
        const T* x = estimate;
        if (image_host) {
            bk.upload(stage64, image_host, sizeof(double) * npix);
            bk.cast_in(diff, stage64, npix, 1.0);
            x = diff;
        }
        bk.subtract(diff, x, true_object, npix);
        DftArgs<T> da;
        memset(&da, 0, sizeof(da));
        da.real_in = diff; da.spec = spec_direct; da.twx = tw_dx; da.twy = tw_dy;
        da.logmag = stage64; da.Ny = Ny; da.Nx = Nx;
        bk.template dft_direct<0, T>(da);
        bk.template dft_direct<1, T>(da);
        bk.download(out_host, stage64, sizeof(double) * npix);
        return true;
    }
    void info(EngineInfo* o) {
        tile.info(o);
        o->Ny = Ny; o->Nx = Nx; o->iterations_done = iterations_done;
        o->tiles_y = tiles_y; o->tiles_x = tiles_x; o->tile_out_y = out_y; o->tile_out_x = out_x;
        o->band_y0 = O.y0; o->band_y1 = O.y1; o->band_x0 = O.x0; o->band_x1 = O.x1;
    }

    // Refresh the halo ring of `arr` from the ranks owning it.  region_layout: the array holds
    // the extended rectangle E ([nimg][E.h][E.w]); else it is a full-size image.
    void exchange_halo(T* arr, bool region_layout, int nimg) {
        if (world == 1 || peers.empty()) return;
        const size_t pitch = region_layout ? (size_t)E.w() : (size_t)Nx;
        const size_t img = region_layout ? bpix : npix;
        const int oy = region_layout ? E.y0 : 0, ox = region_layout ? E.x0 : 0;
        std::vector<T*> sp(peers.size()), rp(peers.size());
        std::vector<size_t> ns(peers.size()), nr(peers.size());
        size_t so = 0, ro = 0;
        for (size_t i = 0; i < peers.size(); ++i) {
            const Rect& s = send_rect[i];
            sp[i] = halo_send + so; ns[i] = s.area() * nimg; so += ns[i];
            rp[i] = halo_recv + ro; nr[i] = recv_rect[i].area() * nimg; ro += nr[i];
            if (!ns[i]) continue;
            RectArgs<T> a;
            a.dst = sp[i]; a.src = arr; a.nimg = nimg; a.h = s.h(); a.w = s.w();
            a.dst_img = s.area(); a.dst_pitch = s.w(); a.dst_off = 0;
            a.src_img = img; a.src_pitch = pitch; a.src_off = (size_t)(s.y0 - oy) * pitch + (s.x0 - ox);
            bk.launch_rect(a);
        }
        bk.exchange((int)peers.size(), peers.data(), sp.data(), ns.data(), rp.data(), nr.data());
        for (size_t i = 0; i < peers.size(); ++i) {
            const Rect& r = recv_rect[i];
            if (!nr[i]) continue;
            RectArgs<T> a;
            a.dst = arr; a.src = rp[i]; a.nimg = nimg; a.h = r.h(); a.w = r.w();
            a.src_img = r.area(); a.src_pitch = r.w(); a.src_off = 0;
            a.dst_img = img; a.dst_pitch = pitch; a.dst_off = (size_t)(r.y0 - oy) * pitch + (r.x0 - ox);
            bk.launch_rect(a);
        }
    }

    // The staged object has a buffer of its own: stage64 is the host-transfer scratch of every
    // get / set / H / H_t / ft_error, any of which may run between upload_object and simulate
    // (a frame loop uploads once and simulates a new noise field per frame).
    void upload_object(const ImageRef& obj) { stage_in(bk, object64, obj, npix); }
    void simulate(double total_brightness, bool rescale, unsigned long long seed) {
        double s = 1.0;
        if (rescale) s = total_brightness / bk.sum(object64, npix, partial);
        bk.cast_in(true_object, object64, npix, s);
        for (int ty = ty0; ty < ty1; ++ty)
            for (int tx = tx0; tx < tx1; ++tx) {
                window(WIN_LOAD, ty, tx, win1, true_object, 0, 1, false);
                tile.op_H(win1, winK, 0, 0);
                WinArgs<T> a = win_args(ty, tx, winK, noiseless, noisy, K, true);
                a.seed = seed; a.img0 = 0;
                bk.template launch_win<WIN_SIMULATE, T>(a);
            }
    }
    void create_data(const double* obj_host, double total_brightness, bool rescale,
                     unsigned long long seed) {
        upload_object(host_image(obj_host));
        simulate(total_brightness, rescale, seed);
    }

    void ensure_norm() {
        if (have_norm) return;
        for (int ty = ty0; ty < ty1; ++ty)     // only the owned pixels are ever used
            for (int tx = tx0; tx < tx1; ++tx) {
                window(WIN_ONES, ty, tx, winK, 0, 0, K, false);
                tile.op_Ht_raw(winK, win2);
                window(WIN_STORE, ty, tx, win2, norm, 0, 1, false);
            }
        have_norm = true;
    }
    // H: big x -> big out[K] (clipped), tile by tile
    // (host-array operators: unsharded handles only; full-size K-image arrays)
    void apply_H(const T* x, T* out) {
        for (int ty = 0; ty < tiles_y; ++ty)
            for (int tx = 0; tx < tiles_x; ++tx) {
                window(WIN_LOAD, ty, tx, win1, const_cast<T*>(x), 0, 1, false);
                tile.op_H(win1, winK, 0, 0);
                window(WIN_STORE, ty, tx, winK, out, 0, K, false);
            }
    }
    void apply_Ht_raw(const T* y, T* out) {
        for (int ty = 0; ty < tiles_y; ++ty)
            for (int tx = 0; tx < tiles_x; ++tx) {
                window(WIN_LOAD, ty, tx, winK, const_cast<T*>(y), 0, K, false);
                tile.op_Ht_raw(winK, win2);
                window(WIN_STORE, ty, tx, win2, out, 0, 1, false);
            }
    }

    void iterate(int n) {
        for (int it = 0; it < n; ++it) {
            ensure_norm();
            if (!have_estimate) { bk.fill(estimate, npix, (T)1); have_estimate = true; halo_fresh = true; }
            // the estimate on the halo ring comes from its owners (first exchange)
            if (!halo_fresh) exchange_halo(estimate, false, 1);
            // ratio = measurement / H(estimate) on the owned tiles
            for (int ty = ty0; ty < ty1; ++ty)
                for (int tx = tx0; tx < tx1; ++tx) {
                    window(WIN_LOAD, ty, tx, win1, estimate, 0, 1, false);
                    tile.op_H(win1, winK, 0, 0);
                    window(WIN_RATIO, ty, tx, winK, ratio, noisy, K, true);
                }
            // the K ratio images on the halo ring come from their owners (second exchange)
            exchange_halo(ratio, true, K);
            // estimate *= H_t(ratio) / norm on the owned tiles
            for (int ty = ty0; ty < ty1; ++ty)
                for (int tx = tx0; tx < tx1; ++tx) {
                    window(WIN_LOAD, ty, tx, winK, ratio, 0, K, true);
                    tile.op_Ht_raw(winK, win2);
                    window(WIN_UPDATE, ty, tx, win2, estimate, norm, 1, false);
                }
            halo_fresh = false;
            ++iterations_done;
        }
    }

    // Per-orientation arrays hold the rank's rectangle only.  Host images are always full size:
    // pixels a rank does not own read as 0 / are ignored on a sharded handle (of
    // H_t_normalization only the owned pixels are meaningful).  The ESTIMATE of a sharded handle
    // is assembled from the owners by one all-reduce: a collective call, every rank gets it all.
    void place_region(const T* region_arr, const Rect& r) {   // stage64 = 0 except r from a region array
        bk.cast_out(stage_region, region_arr, bpix);
        bk.fill_double(stage64, npix, 0.0);
        RectArgs<double> a;
        a.dst = stage64; a.src = stage_region; a.nimg = 1; a.h = r.h(); a.w = r.w();
        a.dst_img = npix; a.dst_pitch = Nx; a.dst_off = (size_t)r.y0 * Nx + r.x0;
        a.src_img = bpix; a.src_pitch = E.w(); a.src_off = (size_t)(r.y0 - E.y0) * E.w() + (r.x0 - E.x0);
        bk.launch_rect(a);
    }
    void get_array(int id, int k, const ImageRef& out) {
        if (id == ARR_NORMALIZATION) ensure_norm();
        if (id == ARR_NOISELESS || id == ARR_NOISY) {
            place_region((id == ARR_NOISY ? noisy : noiseless) + bpix * k, O);
        } else if (id == ARR_ESTIMATE && world > 1) {
            T* tmp = (T*)bk.alloc(sizeof(T) * npix);
            bk.fill(tmp, npix, (T)0);
            RectArgs<T> a;
            a.dst = tmp; a.src = estimate; a.nimg = 1; a.h = O.h(); a.w = O.w();
            a.dst_img = a.src_img = npix; a.dst_pitch = a.src_pitch = Nx;
            a.dst_off = a.src_off = (size_t)O.y0 * Nx + O.x0;
            bk.launch_rect(a);
            bk.all_reduce_sum(tmp, npix);
            bk.cast_out(stage64, tmp, npix);
            bk.sync();
            bk.free(tmp);
        } else {
            bk.cast_out(stage64, id == ARR_TRUE_OBJECT ? true_object
                                 : id == ARR_ESTIMATE ? estimate : norm, npix);
        }
        stage_out(bk, out, stage64, npix);
    }
    void set_array(int id, int k, const ImageRef& in) {
        stage_in(bk, stage64, in, npix);
        if (id == ARR_NOISELESS || id == ARR_NOISY) {
            T* dst = (id == ARR_NOISY ? noisy : noiseless) + bpix * k;
            RectArgs<double> a;
            a.dst = stage_region; a.src = stage64; a.nimg = 1; a.h = E.h(); a.w = E.w();
            a.dst_img = bpix; a.dst_pitch = E.w(); a.dst_off = 0;
            a.src_img = npix; a.src_pitch = Nx; a.src_off = (size_t)E.y0 * Nx + E.x0;
            bk.launch_rect(a);
            bk.cast_in(dst, stage_region, bpix, 1.0);
        } else {
            bk.cast_in(id == ARR_TRUE_OBJECT ? true_object : id == ARR_ESTIMATE ? estimate : norm,
                       stage64, npix, 1.0);
        }
        if (id == ARR_ESTIMATE) { have_estimate = true; halo_fresh = true; }
        if (id == ARR_NORMALIZATION) have_norm = true;
    }
    // H / H_t on full-size images (host arrays or caller device buffers) reuse `ratio` as the
    // K-image temporary (it is rebuilt by every iteration anyway).  The one-image temporary is
    // kept rather than freed: cudaFree would wait for the whole device.
    void H(const ImageRef& x, const ImageRef& out) {
        if (world > 1) throw std::string("H/H_t on full-size images need an unsharded handle");
        T* xin = image_tmp();
        stage_in(bk, stage64, x, npix);
        bk.cast_in(xin, stage64, npix, 1.0);
        apply_H(xin, ratio);
        for (int k = 0; k < K; ++k) {
            bk.cast_out(stage64, ratio + npix * k, npix);
            stage_out(bk, out.at(npix * k), stage64, npix);
        }
    }
    void Ht(const ImageRef& y, const ImageRef& out, bool normalize) {
        if (world > 1) throw std::string("H/H_t on full-size images need an unsharded handle");
        if (normalize) ensure_norm();
        T* res = image_tmp();
        for (int k = 0; k < K; ++k) {
            stage_in(bk, stage64, y.at(npix * k), npix);
            bk.cast_in(ratio + npix * k, stage64, npix, 1.0);
        }
        apply_Ht_raw(ratio, res);
        if (normalize) bk.divide(res, norm, npix);
        bk.cast_out(stage64, res, npix);
        stage_out(bk, out, stage64, npix);
    }

  private:
    int K, ny, nx, Ny, Nx, W;
    int sy, sx, iy0, ix0, out_y, out_x, tiles_y, tiles_x;
    int iterations_done;
    bool have_norm, have_estimate;
    BK& bk;
    DeconvEngine<T, BK> tile;
    size_t npix, wpix, bpix, halo_pixels;
    int rank, world, grid_y, grid_x;
    int ty0, ty1, tx0, tx1;            // tiles of this rank
    Rect O, E;                         // owned pixels; owned + halo ring (what is held)
    bool halo_fresh = true;            // the estimate's halo ring is valid (all ones / just set)
    std::vector<int> peers;
    std::vector<Rect> send_rect, recv_rect;
    T *true_object, *estimate, *norm, *noiseless, *noisy, *ratio, *win1, *win2, *winK;
    T *halo_send, *halo_recv;
    double *stage64, *object64, *partial, *stage_region;
    T* tmp1 = 0;                                            // one full-size image: ft_error, H, H_t (lazy)
    cplx<double>*tw_dx = 0, *tw_dy = 0, *spec_direct = 0;   // ft_error (lazy)
    T* image_tmp() {
        if (!tmp1) tmp1 = (T*)bk.alloc(sizeof(T) * npix);
        return tmp1;
    }

    // Tile (ty, tx) of the global tile grid; `region` = the big arrays hold the rank's
    // rectangle E rather than the full image.  Only pixels of O are written back.
    WinArgs<T> win_args(int ty, int tx, T* tile_buf, T* big, T* big2, int nimg, bool region) {
        WinArgs<T> a;
        memset(&a, 0, sizeof(a));
        a.tile = tile_buf; a.big = big; a.big2 = big2; a.nimg = nimg;
        a.W = W; a.Ny = Ny; a.Nx = Nx;
        a.y0 = ty * out_y - iy0; a.x0 = tx * out_x - ix0;
        a.iy0 = iy0; a.iy1 = iy0 + out_y; a.ix0 = ix0; a.ix1 = ix0 + out_x;
        a.by0 = region ? E.y0 : 0; a.brows = region ? E.h() : Ny;
        a.bx0 = region ? E.x0 : 0; a.bcols = region ? E.w() : Nx;
        a.sy0 = 0; a.sy1 = Ny; a.sx0 = 0; a.sx1 = Nx;
        return a;
    }
    void window(int op, int ty, int tx, T* tile_buf, T* big, T* big2, int nimg, bool region) {
        WinArgs<T> a = win_args(ty, tx, tile_buf, big, big2, nimg, region);
        switch (op) {
            case WIN_LOAD: bk.template launch_win<WIN_LOAD, T>(a); break;
            case WIN_ONES: bk.template launch_win<WIN_ONES, T>(a); break;
            case WIN_STORE: bk.template launch_win<WIN_STORE, T>(a); break;
            case WIN_RATIO: bk.template launch_win<WIN_RATIO, T>(a); break;
            default: bk.template launch_win<WIN_UPDATE, T>(a); break;
        }
    }
};

}  // namespace lsted
