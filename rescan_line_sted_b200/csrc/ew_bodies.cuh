// Small elementwise / reduction bodies shared by the CUDA and the
// host-replay backends (grid-stride over `i`).
#pragma once
#include "fft_core.cuh"

namespace lsted {

enum EwOp { EW_CAST_IN = 0, EW_CAST_OUT = 1, EW_FILL = 2, EW_DIVIDE = 3, EW_RL_UPDATE = 4, EW_SUB = 5,
            EW_TO_STAGE = 6, EW_FROM_STAGE = 7 };

template <typename T> struct EwArgs {
    T* t0;            // destination (or in/out)
    const T* t1;
    const T* t2;
    double* d0;
    const double* d1;
    double s;
    size_t n;         // items
    size_t elems;     // EW_TO_STAGE / EW_FROM_STAGE: elements
    int vec;          // EW_TO_STAGE / EW_FROM_STAGE: the caller buffer is 16-byte aligned
};

// Conversion between a caller's device buffer of T = float or double (the _dev entry points of
// lsted.h) and the engine's fp64 staging array.  EW_TO_STAGE: d0 = (double)t1, exact;
// EW_FROM_STAGE: t0 = (T)d1, rounded to nearest once -- the values the host entry points
// exchange, so a device call gives the bits of its host twin fed the same values.  With `vec`
// item i covers the G = 16 / sizeof(T) elements from G * i with one 16-byte access of the caller
// buffer; otherwise (a view at a storage offset is only element-aligned) item i is element i.
template <typename T> struct alignas(16) Vec16 { T v[16 / sizeof(T)]; };

template <typename T> LSTED_HD size_t stage_items(size_t elems, bool vec) {
    const size_t G = 16 / sizeof(T);
    return vec ? (elems + G - 1) / G : elems;
}

template <int OP, typename T> LSTED_HD void stage_apply(const EwArgs<T>& a, size_t i) {
    const int G = (int)(16 / sizeof(T));
    if (a.vec && (i + 1) * G <= a.elems) {
        if (OP == EW_TO_STAGE) {
            const Vec16<T> w = reinterpret_cast<const Vec16<T>*>(a.t1)[i];
            for (int g = 0; g < G; ++g) a.d0[i * G + g] = (double)w.v[g];
        } else {
            Vec16<T> w;
            for (int g = 0; g < G; ++g) w.v[g] = (T)a.d1[i * G + g];
            reinterpret_cast<Vec16<T>*>(a.t0)[i] = w;
        }
        return;
    }
    const size_t e0 = a.vec ? i * G : i;
    const size_t e1 = a.vec ? (e0 + G < a.elems ? e0 + G : a.elems) : e0 + 1;
    for (size_t e = e0; e < e1; ++e) {
        if (OP == EW_TO_STAGE) a.d0[e] = (double)a.t1[e];
        else a.t0[e] = (T)a.d1[e];
    }
}

template <int OP, typename T> LSTED_HD void ew_apply(const EwArgs<T>& a, size_t i) {
    if (OP == EW_CAST_IN) a.t0[i] = (T)(a.d1[i] * a.s);
    else if (OP == EW_CAST_OUT) a.d0[i] = (double)a.t1[i];
    else if (OP == EW_FILL) a.t0[i] = (T)a.s;
    else if (OP == EW_DIVIDE) a.t0[i] = a.t0[i] / a.t1[i];
    else if (OP == EW_RL_UPDATE) a.t0[i] = a.t0[i] * (a.t1[i] / a.t2[i]);  // est *= H_t(ratio)/norm
    else if (OP == EW_SUB) a.t0[i] = a.t1[i] - a.t2[i];
    else if (OP == EW_TO_STAGE || OP == EW_FROM_STAGE) stage_apply<OP, T>(a, i);
}


// Direct (O(N) per bin) 2-D transform for record_iteration's error spectrum on image sides the
// Stockham plans do not cover (a prime factor above 5, or a column that does not fit a CTA):
// pass 0 = rows (real image -> full complex spectrum), pass 1 = columns + log(1 + |.|) + fftshift.
// Twiddles come from a table by a running index (j*k mod N without a multiply), sums are fp64
// whatever the engine's precision -- this is a diagnostic output, not the iteration.
template <typename T> struct DftArgs {
    const T* real_in;              // [Ny][Nx] (pass 0)
    cplx<double>* spec;            // [Ny][Nx] pass 0 out / pass 1 in
    const cplx<double>* twx;       // exp(-2 pi i j / Nx), j < Nx
    const cplx<double>* twy;       // exp(-2 pi i j / Ny), j < Ny
    double* logmag;                // [Ny][Nx] (pass 1), fftshifted like np.fft.fftshift
    int Ny, Nx;
};

template <int PASS, typename T> LSTED_HD void dft_direct_apply(const DftArgs<T>& a, size_t e) {
    const int y = (int)(e / a.Nx), x = (int)(e - (size_t)y * a.Nx);   // output bin (ky | y, kx)
    double re = 0.0, im = 0.0;
    if (PASS == 0) {
        const T* row = a.real_in + (size_t)y * a.Nx;
        int idx = 0;
        for (int n = 0; n < a.Nx; ++n) {
            const cplx<double> w = a.twx[idx];
            const double v = (double)row[n];
            re += v * w.x; im += v * w.y;
            idx += x; if (idx >= a.Nx) idx -= a.Nx;
        }
        a.spec[e] = mk<double>(re, im);
    } else {
        int idx = 0;
        for (int n = 0; n < a.Ny; ++n) {
            const cplx<double> w = a.twy[idx];
            const cplx<double> v = a.spec[(size_t)n * a.Nx + x];
            re += v.x * w.x - v.y * w.y; im += v.x * w.y + v.y * w.x;
            idx += y; if (idx >= a.Ny) idx -= a.Ny;
        }
        int ys = y + a.Ny / 2, xs = x + a.Nx / 2;
        if (ys >= a.Ny) ys -= a.Ny;
        if (xs >= a.Nx) xs -= a.Nx;
        a.logmag[(size_t)ys * a.Nx + xs] = log(1.0 + sqrt(re * re + im * im));
    }
}

}  // namespace lsted

// ---------------------------------------------------------------------------
// Window kernels of the tiled (overlap-save) engine: move data between the full
// image arrays and one tile window of W x W pixels whose top-left corner sits at
// (y0, x0) of the image (may be negative / past the edge: zero padding, like the
// linear convolution of the reference).  Only the alias-free interior
// [iy0, iy1) x [ix0, ix1) of a window is ever written back.
// ---------------------------------------------------------------------------
#include "poisson.cuh"
namespace lsted {

enum WinOp {
    WIN_LOAD = 0,     // tile = window of big (zero outside the image)
    WIN_ONES = 1,     // tile = 1 inside the image, 0 outside
    WIN_STORE = 2,    // big[interior] = tile
    WIN_SIMULATE = 3, // big[interior] = tile (noiseless); big2[interior] = Poisson(tile) + 1e-9
    WIN_RATIO = 4,    // big[interior] = big2[interior] / tile      (ratio = measurement / expected)
    WIN_UPDATE = 5    // big[interior] *= tile / big2[interior]     (estimate *= H_t(ratio) / norm)
};

template <typename T> struct WinArgs {
    T* tile;          // [nimg][W][W]
    T* big;           // [nimg][Ny][Nx]
    T* big2;
    int nimg, W, Ny, Nx;
    int y0, x0;       // image coordinates of tile pixel (0, 0)
    int iy0, iy1, ix0, ix1;  // interior of the window (tile coordinates)
    int by0, brows;   // the big arrays hold image rows [by0, by0 + brows) ...
    int bx0, bcols;   // ... and columns [bx0, bx0 + bcols): the region a rank of a sharded object keeps
    int sy0, sy1;     // only image rows [sy0, sy1) ...
    int sx0, sx1;     // ... and columns [sx0, sx1) are written back (the rank's own tiles)
    unsigned long long seed;
    unsigned int img0;
};

template <int OP, typename T> LSTED_HD void win_apply(const WinArgs<T>& a, size_t e) {
    const size_t per = (size_t)a.W * a.W;
    const int img = (int)(e / per);
    const size_t r = e - (size_t)img * per;
    const int wy = (int)(r / a.W), wx = (int)(r - (size_t)wy * a.W);
    const int gy = a.y0 + wy, gx = a.x0 + wx;
    const bool inside = gy >= 0 && gy < a.Ny && gx >= 0 && gx < a.Nx;
    const bool held = inside && gy >= a.by0 && gy < a.by0 + a.brows &&
                      gx >= a.bx0 && gx < a.bx0 + a.bcols;             // pixel present in `big`
    const size_t gi = (size_t)img * a.brows * a.bcols + (size_t)(held ? gy - a.by0 : 0) * a.bcols +
                      (held ? gx - a.bx0 : 0);
    if (OP == WIN_LOAD) { a.tile[e] = held ? a.big[gi] : (T)0; return; }
    if (OP == WIN_ONES) { a.tile[e] = inside ? (T)1 : (T)0; return; }
    if (!held || gy < a.sy0 || gy >= a.sy1 || gx < a.sx0 || gx >= a.sx1 ||
        wy < a.iy0 || wy >= a.iy1 || wx < a.ix0 || wx >= a.ix1)
        return;
    const T v = a.tile[e];
    if (OP == WIN_STORE) a.big[gi] = v;
    else if (OP == WIN_SIMULATE) {
        a.big[gi] = v;
        const unsigned long long pix = (unsigned long long)gy * a.Nx + gx;
        a.big2[gi] = (T)(poisson_sample((double)v, a.seed, pix, a.img0 + img) + 1e-9);
    } else if (OP == WIN_RATIO) a.big[gi] = v > (T)0 ? a.big2[gi] / v : (T)0;   // see rl_ratio (conv_bodies.cuh)
    else if (OP == WIN_UPDATE) a.big[gi] = a.big[gi] * (v / a.big2[gi]);
}

// Rectangle copy between strided image stacks: packs / unpacks the halo strips a sharded tiled
// object exchanges with its neighbours, and places a rank's region in a full-size image.
template <typename T> struct RectArgs {
    T* dst; const T* src;
    int nimg, h, w;                        // rectangle: h rows of w pixels in each of nimg images
    size_t dst_img, dst_pitch, dst_off;    // element strides; offset of the rectangle's first pixel
    size_t src_img, src_pitch, src_off;
};
template <typename T> LSTED_HD void rect_apply(const RectArgs<T>& a, size_t e) {
    const int x = (int)(e % a.w);
    const size_t t = e / a.w;
    const int y = (int)(t % a.h);
    const size_t img = t / a.h;
    a.dst[a.dst_off + img * a.dst_img + (size_t)y * a.dst_pitch + x] =
        a.src[a.src_off + img * a.src_img + (size_t)y * a.src_pitch + x];
}

}  // namespace lsted
