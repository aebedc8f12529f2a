/* liblsted -- C ABI of the B200-native line_sted_tools hot path.
 *
 * Every entry point returns 0 on success and a non-zero status otherwise;
 * lsted_last_error() then returns a thread-local, human-readable message.
 * All array arguments are HOST pointers to C-contiguous float64 data unless
 * the name says otherwise (the _dev entry points take device buffers of float32
 * or float64); the library owns all device memory it allocates.  Handles are
 * not thread-safe; each owns one CUDA stream.  There is no CPU fallback: a
 * call without a usable CUDA device fails with LSTED_ERR_CUDA.
 *
 * Each function names the reference interface it replaces
 * (figure_generation/line_sted_tools.py of AndrewGYork/rescan_line_sted).
 */
#ifndef LSTED_H
#define LSTED_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
    LSTED_OK = 0,
    LSTED_ERR_ARG = 1,   /* bad argument / unsupported size */
    LSTED_ERR_CUDA = 2,  /* CUDA runtime failure (message has the details) */
    LSTED_ERR_NCCL = 3,
    LSTED_ERR_STATE = 4  /* call order (e.g. iterate before data) */
};

/* which-array selectors of lsted_deconv_get / lsted_deconv_set: the public
 * attributes of the reference Deconvolver (line_sted_tools.py:478-594) */
enum {
    LSTED_TRUE_OBJECT = 0,
    LSTED_NOISELESS = 1,     /* noiseless_measurement[k] */
    LSTED_NOISY = 2,         /* noisy_measurement[k]     */
    LSTED_ESTIMATE = 3,
    LSTED_NORMALIZATION = 4  /* H_t_normalization        */
};

int lsted_version(void);
const char* lsted_last_error(void);
int lsted_device_count(int* count);
/* Pinned host buffers for end-to-end pipelines (numpy wraps them). */
int lsted_host_alloc(void** ptr, size_t bytes);
int lsted_host_free(void* ptr);

/* ---------------- PSF synthesis: generate_psfs, line_sted_tools.py:168-363 -------------
 * One operating point = (excitation_brightness, depletion_brightness); `taps`
 * are the 2*radius+1 normalised Gaussian FIR taps (scipy truncate=4 rule,
 * computed by the host mirror exactly like scipy does).
 * psf_type: 0 = point, 1 = line.  All outputs are [batch][n][n] float64.   */
int lsted_psf_illumination(int device, int psf_type, int batch, int n, const double* taps,
                           int radius, const double* excitation_brightness,
                           const double* depletion_brightness, double* excitation,
                           double* depletion, double* excitation_fraction,
                           double* depletion_fraction, double* sted); /* :180-243 */
/* Rescan / descan system PSFs from the STED centre rows ([batch][n]) and the
 * integer rescan ratios ([batch], from the host Gaussian fit :252-256).
 * `wide` ([n][ratio*n], batch 1 only) may be NULL.                          :258-310 */
int lsted_psf_rescan(int device, int batch, int n, const double* taps, int radius,
                     const double* sted_rows, const int* ratios, double* emission,
                     double* rescan, double* descan, double* wide);

/* psf_report (:75-166) for a batch of operating points without returning to the host in
 * between: illumination, the Gaussian width fits (get_width :653-668, a Levenberg-Marquardt
 * fit from the reference's start (1, n/2, 1), run on the device to the fp64 floor), the
 * integer rescan ratio the fit decides (:252-256), rescan / descan PSFs and the dose sums
 * (:134-144, per pulse).  One CTA per point; every point has its own grid size n[b] and FIR
 * taps (taps[b][0 .. 2*radius[b]], rows `tap_stride` apart).
 * scalars [batch][16]: 0 excitation sigma, 1 STED sigma, 2 rescan sigma (line), 3 real and
 * 4 rounded rescan ratio (line), 5 excitation dose, 6 depletion dose, 7 emission (all per
 * pulse), 8 function evaluations of the fits, 9 fit status (0 = every fit ended with MINPACK
 * info 1..4, which is what scipy accepts), 10-12 centre-row-maximum checks
 * (:105-106, :120).  psfs: NULL, or [batch][7][nmax*nmax] (nmax = max n[b]; plane i of point
 * b holds n[b]*n[b] packed values): excitation, depletion, excitation_fraction,
 * depletion_fraction, sted, rescan_sted, descan_sted (the last two for lines only).       */
int lsted_psf_report_batch(int device, int psf_type, int batch, const int* n, const int* radius,
                           const double* taps, int tap_stride, const double* blur_sigma,
                           const double* excitation_brightness, const double* depletion_brightness,
                           double* scalars, double* psfs);

/* get_width (:653-668) for a batch of profiles rows[batch][n]: the same in-kernel lmdif.
 * out [batch][5]: A, mu, sigma, function evaluations, MINPACK info (scipy accepts 1..4). */
int lsted_gauss_fit(int device, int batch, int n, const double* rows, double* out);

/* Orientation step of Deconvolver's caller (line_sted_figure_2.py:264-272, used at
 * :244-247): rotate one plane [n0][n1] to `batch` orientations like
 * scipy.ndimage.rotate(order=3, mode='constant', cval=0, reshape=False) and clip to
 * [0, clip_hi].  xform = [batch][6] = the 2x2 matrix [[c, s], [-s, c]] (row-major) and
 * the offset centre - matrix*centre of each angle (host: cosdg/sindg).  out [batch][n0][n1]. */
int lsted_psf_rotate(int device, int batch, int n0, int n1, const double* plane,
                     const double* xform, double clip_hi, double* out);

/* ---------------- Deconvolver, line_sted_tools.py:478-594 -------------------------------- */
typedef struct lsted_deconv lsted_deconv;

typedef struct {
    int K, ny, nx, Ny, Nx;       /* PSF count / size, image size                     */
    int Ly, Lx;                  /* FFT lengths (columns, rows)                      */
    int cols_per_cta, row_pairs_per_cta;
    int precision;               /* 32 or 64                                         */
    int iterations_done;
    int device;
    size_t row_smem_bytes, col_smem_bytes;
    size_t device_bytes;         /* HBM held by the handle                           */
    /* algorithmic bytes (SURVEY.md 8d): A = sizeof(T)*Ny*Nx                         */
    double bytes_forward;        /* (2K+1) A                                         */
    double bytes_normalization;  /* A                                                */
    double bytes_iteration;      /* (K+4) A                                          */
    int tiles_y, tiles_x;        /* overlap-save tiling of large objects (1 x 1: none) */
    int tile_out_y, tile_out_x;  /* pixels of the object each tile produces            */
    int band_y0, band_y1;        /* image rows owned by this rank (tiled + sharded)    */
    int band_x0, band_x1;        /* image columns owned by this rank                    */
} lsted_deconv_info_t;

/* Deconvolver.__init__ (:479-494): psfs = [K][ny][nx].  precision 32 | 64.          */
int lsted_deconv_create(lsted_deconv** out, int device, const double* psfs, int K, int ny, int nx,
                        int Ny, int Nx, int precision);
/* Same, with overlap-save tiling: the object is processed through windows of
 * tile_fft_len^2 pixels (halo included) and may be arbitrarily large.  0 = decide
 * automatically (lsted_deconv_create tiles with 2160 when one transform of the padded
 * object does not fit a CTA's shared memory, e.g. 8192^2).                            */
int lsted_deconv_create_tiled(lsted_deconv** out, int device, const double* psfs, int K, int ny,
                              int nx, int Ny, int Nx, int precision, int tile_fft_len);
int lsted_deconv_destroy(lsted_deconv* h);
int lsted_deconv_info(lsted_deconv* h, lsted_deconv_info_t* info);
/* options: "exact_clip" (0|1: clip every H_t term before the sum, like :587),
 *          "profile" (0|1: per-kernel CUDA-event timing),
 *          "graph" (0|1, default 1: replay the four launches of a steady RL iteration as one
 *          captured CUDA graph -- what makes iterate() at the reference's 128^2 frames cheap),
 *          "forget_normalization" (drop the cached H_t_normalization, :590),
 *          "reset_estimate" (the next iterate() starts from an all-ones estimate, :521-522;
 *          new data alone do not reset it, as in the reference),
 *          "fast_path" (0|1, default 1: use the compile-time-planned kernels when
 *          the transform length has one; 0 forces the generic mixed-radix kernels),
 *          A/B switches of kernel variants with identical results: "row_tma" (0|1|2, default 2:
 *          row spectra moved by tensor-map bulk copies; 2 = also the two-buffer ROW_MID), "real_otf", "row_dual", "row_plan2",
 *          "prefetch" */
int lsted_deconv_set_option(lsted_deconv* h, const char* name, double value);
/* record_iteration's error spectrum (:539-546): out[Ny][Nx] = log(1 + |fftshift(fft2(x -
 * true_object))|) with x = `image` (host, [Ny][Nx]) or, when image is NULL, the estimate in
 * HBM.  Sides with a prime factor above 5 (or longer than one CTA holds) and tiled objects
 * take a direct O(N)-per-bin transform, also on the device.  *done = 0 (out untouched) only
 * for image == NULL on a rank of a sharded tiled object, which holds a region of the
 * estimate: pass the gathered estimate as `image` there.                                  */
int lsted_deconv_ft_error(lsted_deconv* h, const double* image, double* out, int* done);
/* create_data_from_object (:496-512).  rescale != 0 applies total_brightness.
 * Noise: in-kernel Philox4x32-10 Poisson, stream selected by `seed`.               */
int lsted_deconv_create_data(lsted_deconv* h, const double* object, double total_brightness,
                             int rescale, uint64_t seed);
/* The same in two asynchronous halves for pipelines that keep the object in HBM:
 * stage the object (H2D on the handle's stream; pass pinned memory to overlap),
 * then run the forward model + Poisson on whatever object is staged.              */
int lsted_deconv_upload_object(lsted_deconv* h, const double* object);
int lsted_deconv_simulate(lsted_deconv* h, double total_brightness, int rescale, uint64_t seed);
/* Orientation sharding over the GPUs of one node (SURVEY.md 8e): the handle was created
 * with this rank's subset of the PSFs (global orientation indices k_offset ...); every
 * rank keeps a replica of the estimate and of the normalisation, and the partial H_t sums
 * are combined by ONE ncclAllReduce per RL iteration (of the Fourier-domain partial sum)
 * on the handle's stream.  `unique_id` = the 128 bytes lsted_nccl_unique_id() produced
 * on rank 0, distributed by the caller (e.g. torch.distributed broadcast).  NCCL is
 * dlopen()ed on first use; single-GPU users do not need it.
 * A TILED handle (lsted_deconv_create_tiled) shards differently: every rank gets ALL
 * PSFs and the overlap-save tiles are dealt to a 2-D grid of ranks (k_offset is ignored);
 * a rank keeps measurements and ratios on its rectangle of the image (band_y0..band_x1 of
 * lsted_deconv_info; identical noise on any rank count because the Poisson stream is keyed
 * by the global pixel index) and per RL iteration receives the PSF-halo ring of the
 * estimate and of the K ratio images from the neighbouring ranks (grouped ncclSend /
 * ncclRecv of packed strips).  lsted_deconv_get(LSTED_ESTIMATE) on such a handle is a
 * collective call (one all-reduce assembles the owners' rectangles on every rank).     */
enum { LSTED_NCCL_UNIQUE_ID_BYTES = 128 };
int lsted_nccl_unique_id(char* out);
int lsted_deconv_shard(lsted_deconv* h, int rank, int world, int k_offset, const char* unique_id);
/* Orientation sharding, fast path: sum the partial H_t spectra of the ranks INSIDE the column
 * kernel over NVLink peer memory (no all-reduce after it).  One process per GPU: every rank
 * exports LSTED_P2P_HANDLE_BYTES of CUDA-IPC handles (after lsted_deconv_shard), the caller
 * all-gathers them (torch.distributed) and hands every rank the [world][...] table.  Without
 * these two calls the reduction is the NCCL all-reduce of lsted_deconv_shard.              */
#define LSTED_P2P_HANDLE_BYTES 192
int lsted_deconv_p2p_export(lsted_deconv* h, char* handles_out, int capacity);
int lsted_deconv_p2p_attach(lsted_deconv* h, const char* all_handles, int world);
/* Orientation sharding, fp32: sum the partial H_t spectra THROUGH THE NVSWITCH (NVLS).  The
 * spectrum that carries the partial sums is bound to one CUDA multicast object shared by the
 * ranks; after the column kernel every rank pulls the sum of its 1/world of the buffer with
 * multimem.ld_reduce (added inside the switch) and pushes it to every replica with multimem.st
 * -- one kernel, (world-1)/world of the buffer per NVLink direction, no staging.  Choreography
 * (one process per GPU; rescan_line_sted_b200/sharded.py does it over torch.distributed and a
 * Unix socket), after lsted_deconv_shard and before any data is on the handle:
 *   rank 0:       lsted_deconv_nvls_create(h, world, &fd)   POSIX descriptor of the object
 *   other ranks:  receive a duplicate of that descriptor (SCM_RIGHTS), lsted_deconv_nvls_import
 *   every rank:   lsted_deconv_nvls_add_device; barrier; lsted_deconv_nvls_bind; barrier.
 * Without these calls the reduction is the peer-memory kernel above or the NCCL all-reduce. */
int lsted_deconv_nvls_supported(int device, int* supported);
int lsted_deconv_nvls_create(lsted_deconv* h, int world, int* fd_out);
int lsted_deconv_nvls_import(lsted_deconv* h, int world, int fd);
int lsted_deconv_nvls_add_device(lsted_deconv* h);
int lsted_deconv_nvls_bind(lsted_deconv* h);
/* iterate() n times (:520-531); no host transfers.                                 */
int lsted_deconv_iterate(lsted_deconv* h, int n);
/* attribute access; k is the PSF index for the per-PSF lists, else 0.
 * Setting LSTED_NOISY is the injection point for bit-exact noise fields.           */
int lsted_deconv_get(lsted_deconv* h, int which, int k, double* out);
int lsted_deconv_set(lsted_deconv* h, int which, int k, const double* in);
/* H (:567-577): x[Ny][Nx] -> out[K][Ny][Nx];  H_t (:579-594): y[K][Ny][Nx] -> out[Ny][Nx]. */
int lsted_deconv_H(lsted_deconv* h, const double* x, double* out);
int lsted_deconv_Ht(lsted_deconv* h, const double* y, double* out, int normalize);

/* ---- the same on DEVICE buffers (e.g. torch.Tensor.data_ptr()), no host round trip ----
 * Each _dev call mirrors its host twin above (shapes, `which` / `k`, side effects on the
 * handle); lsted_deconv_simulate after lsted_deconv_upload_object_dev is the device form of
 * lsted_deconv_create_data.  Buffers are C-contiguous, of element type `dtype`, at least
 * element-aligned (16-byte alignment takes vector accesses), in device (or managed) memory of
 * the handle's device.  float32 values enter exactly and leave rounded to nearest once, so a
 * call gives the bits of the host call fed the same values.
 * Stream contract: `stream` is a cudaStream_t on the handle's device (NULL: the legacy default
 * stream), in PyTorch torch.cuda.current_stream().cuda_stream.  The handle's work starts after
 * everything already enqueued on `stream`; everything enqueued on `stream` later waits for the
 * call's reads and writes (one event each way), so an input may be freed or reused as soon as
 * the call returns.  No call blocks the host.  A stream being captured into a CUDA graph is
 * refused with LSTED_ERR_STATE.  Every argument is checked before anything is enqueued: a bad
 * dtype, a misaligned pointer, host memory, memory of another device, or a range running past
 * its allocation fails with LSTED_ERR_ARG.                                                      */
enum { LSTED_F32 = 32, LSTED_F64 = 64 };   /* element type of caller device buffers */
int lsted_deconv_get_dev(lsted_deconv* h, int which, int k, void* out, int dtype, void* stream);
int lsted_deconv_set_dev(lsted_deconv* h, int which, int k, const void* in, int dtype, void* stream);
int lsted_deconv_upload_object_dev(lsted_deconv* h, const void* object, int dtype, void* stream);
/* x[Ny][Nx] -> out[K][Ny][Nx];  y[K][Ny][Nx] -> out[Ny][Nx]; x / y and out share `dtype`.    */
int lsted_deconv_H_dev(lsted_deconv* h, const void* x, void* out, int dtype, void* stream);
int lsted_deconv_Ht_dev(lsted_deconv* h, const void* y, void* out, int dtype, int normalize, void* stream);
int lsted_deconv_sync(lsted_deconv* h);
/* CUDA-event stopwatch on the handle's stream.                                     */
int lsted_deconv_timer_start(lsted_deconv* h);
int lsted_deconv_timer_stop(lsted_deconv* h, float* milliseconds);
/* Per-kernel statistics gathered while option "profile" is on.  Kernel kinds:
 * 0 row_fwd, 1 row_inv_store, 2 row_inv_sim, 3 row_mid, 4 row_final,
 * 5 col_otf, 6 col_h, 7 col_ht, 8 elementwise.                                      */
enum { LSTED_NUM_KERNEL_KINDS = 9 };
int lsted_deconv_profile(lsted_deconv* h, int reset, double* total_ms, long long* launches);

/* ---------------- figure-3 scan-position engine, line_sted_figure_3.py:76-273 -------------
 * The explicit acquisition simulation `simulate_imaging` of the reference: for every scan
 * position the excitation is shifted over the (rotated, zero-padded) object, the glow is
 * (de)scanned, blurred onto the detector and summed the way each method reads its detector.
 * One handle = one (imaging type, object shape, scan) ; lsted_scan_run does one orientation
 * with ALL scan positions in flight at once; lsted_scan_frames returns the display planes the
 * reference hands to its generate_figure (:262-271) for the positions kept by the run.
 * imaging_type: 0 descan_point, 1 nondescan_multipoint, 2 descan_line, 3 rescan_line (:95-96). */
typedef struct lsted_scan lsted_scan;
typedef struct {
    int imaging_type;
    int n_y, n_x, pad;      /* object shape before padding, zero padding on every side (:100-102) */
    int step;               /* scan step in pixels, round(psf_width / (4 R))             (:91)     */
    int exc_sep;            /* multipoint: spot separation (:131), else 0                          */
    int num_positions;      /* scan positions (:109-137)                                           */
    double zoom_factor;     /* rescan line: scale_y factor 1 / (R^2 + 1) (:221-223), else 0        */
    int blur_radius;        /* detector blur gaussian_filter(., psf_sigma): taps radius (truncate 4) */
    int exc_radius;         /* excitation blur (sted sigma, truncate=8, :139): taps radius         */
    size_t chunk_bytes;     /* device memory for the per-position planes in flight; 0 = 4 GiB      */
} lsted_scan_params_t;
/* positions [num_positions][2] = (shift_y, shift_x) in the reference's order; blur_taps
 * [2*blur_radius+1], exc_taps [2*exc_radius+1]: normalised Gaussian taps as scipy builds them. */
int lsted_scan_create(lsted_scan** out, int device, const lsted_scan_params_t* params,
                      const int* positions, const double* blur_taps, const double* exc_taps);
int lsted_scan_destroy(lsted_scan* h);
/* centered_exc (:104-140), out [n_y+2pad][n_x+2pad] */
int lsted_scan_excitation(lsted_scan* h, double* out);
/* One orientation (:152-229).  obj_padded [n0][n1] (n = n + 2 pad); rot_xform = NULL for 0
 * degrees, else the 6 numbers (2x2 matrix, offset) scipy.ndimage.rotate builds for
 * rotate(obj, rot) (:382-391: order 3, mode='nearest', clip to [0, 1.1 max]).
 * frame_positions [num_frames]: ascending scan-position indices whose planes are kept for
 * lsted_scan_frames (may be NULL / 0).  Outputs (each may be NULL): maxima [num_positions][5]
 * = maxima of glow, inst_detector_sig, cum_detector_sig, reconstruction, new_signal after every
 * position (:231-235); reconstruction and cum_detector_sig [n0][n1] after the last position;
 * device_ms = CUDA-event time of the call's device work.                                     */
int lsted_scan_run(lsted_scan* h, const double* obj_padded, const double* rot_xform,
                   const int* frame_positions, int num_frames, double* maxima,
                   double* reconstruction, double* cum_detector_sig, double* device_ms);
/* Kept frames first .. first+count-1 of the last run: out [count][6][n_y][n_x] = de-rotated
 * excitation, de-rotated glow, inst_detector_sig, cum_detector_sig, new_signal, reconstruction,
 * cropped by `pad` and divided by display_max[6] (:262-271).  inv_xform = NULL for 0 degrees,
 * else scipy's matrix/offset of rotate(., -rot) (:169-170).                                   */
int lsted_scan_frames(lsted_scan* h, int first, int count, const double* display_max,
                      const double* inv_xform, double* out);

/* The resampling helpers of figure 3 (:382-409) as one operator: cubic-spline
 * scipy.ndimage.affine_transform of `batch` planes [n0][n1] -> [m0][m1], output pixel (i, j)
 * reads input coordinate matrix*(i, j) + offset (xform [batch][6] = m00 m01 m10 m11 o0 o1).
 * mode 0 = 'constant' (cval 0; what shift :393-396 and zoom :398-409 use),
 * mode 1 = 'nearest' (12-sample edge pad before the prefilter; what rotate :382-391 uses).
 * clip != 0: clip every plane to [0, 1.1 * max(input plane)] like the reference's wrappers.   */
int lsted_img_spline(int device, int batch, int n0, int n1, const double* planes,
                     const double* xform, int m0, int m1, int mode, int clip, double* out);
/* scipy.ndimage.gaussian_filter(mode='reflect') of `batch` planes along axis 0 (taps0) and
 * axis 1 (taps1); a NULL tap pointer leaves that axis alone (sigma 0), :139,:173,:202,:221.   */
int lsted_img_gauss(int device, int batch, int n0, int n1, const double* planes,
                    const double* taps0, int radius0, const double* taps1, int radius1, double* out);

#ifdef __cplusplus
}
#endif
#endif
