// liblsted.so -- sm_100a kernels + the C ABI of include/lsted.h.
//
// Build: see Makefile (nvcc -gencode arch=compute_100a,code=sm_100a).
// The kernels are thin __global__ shells around the bodies in
// conv_bodies.cuh / psf_kernels.cuh; orchestration lives in engine.h.
#include <cuda.h>
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <new>
#include <string>
#include <map>
#include <vector>

#include "../../include/lsted.h"
#include "engine.h"
#include "tiled.h"
#include "conv_fast.cuh"
#include "ew_bodies.cuh"
#include "psf_kernels.cuh"
#include "dispatch.h"

namespace lsted {
struct ApiError { int code; std::string msg; };
}

static thread_local std::string g_error;
static int set_error(int code, const std::string& msg) { g_error = msg; return code; }

#define CUDA_CHECK(expr)                                                                  \
    do {                                                                                  \
        cudaError_t err__ = (expr);                                                       \
        if (err__ != cudaSuccess) {                                                       \
            lsted::ApiError e__;                                                          \
            e__.code = LSTED_ERR_CUDA;                                                    \
            e__.msg = std::string(#expr) + ": " + cudaGetErrorString(err__);              \
            throw e__;                                                                    \
        }                                                                                 \
    } while (0)

// ---------------------------------------------------------------------------
// Device-side CTA context and kernel shells
// ---------------------------------------------------------------------------
struct DeviceCtx {
    template <class F> __device__ __forceinline__ void parallel_for(int n, F f) {
        for (int w = threadIdx.x; w < n; w += blockDim.x) f(w);
        __syncthreads();
    }
    // one per-thread phase of a register-resident body, then a CTA barrier
    template <class R, class F> __device__ __forceinline__ void phase(R* regs, F f) {
        f((int)threadIdx.x, *regs);
        __syncthreads();
    }
    // a phase nothing later depends on through shared memory (prefetches, final stores)
    template <class R, class F> __device__ __forceinline__ void phase_nosync(R* regs, F f) {
        f((int)threadIdx.x, *regs);
    }
};

// Launch bounds of the fast-path kernels (plans and selection: dispatch.h)
#ifndef LSTED_ROW_LEAN_CTAS
#define LSTED_ROW_LEAN_CTAS 6   // "lean" ROW_MID (two shared-memory buffers, 35 KB): CTAs per SM -> 64 registers, no spills
#endif
#ifndef LSTED_ROW_SIM_CTAS
#define LSTED_ROW_SIM_CTAS 4   // ROW_INV_SIM (fp64 Poisson arithmetic in an fp32 kernel): CTAs per SM
#endif
#ifndef LSTED_ROW_RESIDENT_THREADS
#define LSTED_ROW_RESIDENT_THREADS 480  // 3 row CTAs per SM: no register spills
#endif
// G: image geometry known at compile time (the 2048-wide / 107-wide-PSF headline case) or not
template <int MODE, class P, class G = lsted::RowGeomRuntime, int TMA = 0>
__global__ void __launch_bounds__(P::ROW_THREADS, TMA == 2 ? (MODE == lsted::ROW_MID ? LSTED_ROW_LEAN_CTAS : 4) : sizeof(typename P::T) == 4 ? (MODE == lsted::ROW_INV_SIM ? LSTED_ROW_SIM_CTAS : LSTED_ROW_RESIDENT_THREADS / P::ROW_THREADS) : 1)
row_fast_kernel(const __grid_constant__ lsted::RowArgs<typename P::T> a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    DeviceCtx cx;
    lsted::RowRegs<P> r;
    lsted::row_fast_body<MODE, P, DeviceCtx, G, TMA>(cx, blockIdx.x, a,
                                  reinterpret_cast<lsted::cplx<typename P::T>*>(smem_raw), &r);
}

// Row kernels on the two-pass plan 2160 = 48 x 45 (conv_fast.cuh: row2_fast_body), fp32
#ifndef LSTED_ROW2_CTAS
#define LSTED_ROW2_CTAS 3
#endif
template <int MODE, class P, class G = lsted::RowGeomRuntime>
__global__ void __launch_bounds__(P::ROW_THREADS, LSTED_ROW2_CTAS)
row2_fast_kernel(const __grid_constant__ lsted::RowArgs<typename P::T> a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DeviceCtx cx;
    lsted::Row2Regs<P> r;
    lsted::row2_fast_body<MODE, P, DeviceCtx, G>(cx, blockIdx.x, a,
                                  reinterpret_cast<lsted::cplx<typename P::T>*>(smem_raw), &r);
}

// ROW_MID with two row pairs per thread group (conv_fast.cuh: row_mid_dual_body)
template <class P>
__global__ void __launch_bounds__(lsted::RowDual<P>::THREADS, 2)
row_mid_dual_kernel(const __grid_constant__ lsted::RowArgs<typename P::T> a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DeviceCtx cx;
    typename lsted::RowDual<P>::Regs r;
    lsted::row_mid_dual_body<P>(cx, blockIdx.x, a, smem_raw, &r);
}

// sub-block column CTAs (real OTFs): CS of the C columns of a block, two CTAs per SM
template <int MODE, class P, class G = lsted::ColGeomRuntime>
__global__ void __launch_bounds__(P::SUB_THREADS, 2)
col_sub_kernel(const __grid_constant__ lsted::ColArgs<typename P::T> a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DeviceCtx cx;
    lsted::ColRegs<P> r;
    lsted::col_fast_body<MODE, P, DeviceCtx, G, true, true>(cx, blockIdx.x, a,
                                  reinterpret_cast<lsted::cplx<typename P::T>*>(smem_raw), &r);
}
template <int MODE, class P, class G = lsted::ColGeomRuntime, bool RO = false>
__global__ void __launch_bounds__(P::COL_THREADS, 1)
col_fast_kernel(const __grid_constant__ lsted::ColArgs<typename P::T> a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DeviceCtx cx;
    lsted::ColRegs<P> r;
    lsted::col_fast_body<MODE, P, DeviceCtx, G, RO>(cx, blockIdx.x, a,
                                  reinterpret_cast<lsted::cplx<typename P::T>*>(smem_raw), &r);
}

// COL_HT with the cross-GPU sum fused in (persistent: one CTA per SM walks several blocks)
template <class P, bool RO = false>
__global__ void __launch_bounds__(P::COL_THREADS, 1)
col_ht_p2p_kernel(const __grid_constant__ lsted::ColArgs<typename P::T> a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DeviceCtx cx;
    lsted::ColRegs<P> r;
    lsted::col_ht_p2p_body<P, DeviceCtx, lsted::ColGeomRuntime, RO>(cx, blockIdx.x, gridDim.x, a,
                                  reinterpret_cast<lsted::cplx<typename P::T>*>(smem_raw), &r);
}

enum { kRowThreads = 256, kColThreads32 = 512, kColThreads64 = 256, kEwThreads = 256 };

template <int MODE, typename T>
__global__ void __launch_bounds__(kRowThreads)
row_kernel(const __grid_constant__ lsted::RowArgs<T> a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DeviceCtx cx;
    lsted::row_body<MODE, T>(cx, blockIdx.x, a, reinterpret_cast<lsted::cplx<T>*>(smem_raw));
}

template <int MODE, typename T>
__global__ void __launch_bounds__(sizeof(T) == 4 ? kColThreads32 : kColThreads64)
col_kernel(const __grid_constant__ lsted::ColArgs<T> a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DeviceCtx cx;
    lsted::col_body<MODE, T>(cx, blockIdx.x, a, reinterpret_cast<lsted::cplx<T>*>(smem_raw));
}

template <int OP, typename T>
__global__ void __launch_bounds__(kEwThreads) ew_kernel(const lsted::EwArgs<T> a) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += stride)
        lsted::ew_apply<OP, T>(a, i);
}

template <int PASS, typename T>
__global__ void __launch_bounds__(kEwThreads) dft_direct_kernel(const lsted::DftArgs<T> a) {
    const size_t n = (size_t)a.Ny * a.Nx;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride)
        lsted::dft_direct_apply<PASS, T>(a, e);
}

template <int OP, typename T>
__global__ void __launch_bounds__(kEwThreads) win_kernel(const lsted::WinArgs<T> a) {
    const size_t n = (size_t)a.nimg * a.W * a.W;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride)
        lsted::win_apply<OP, T>(a, e);
}

// ---------------------------------------------------------------------------
// All-reduce of the partial H_t spectra of orientation-sharded ranks THROUGH THE NVSWITCH
// (NVLS): every rank's spectrum buffer is bound to one CUDA multicast object; rank r owns 1/world
// of the buffer, pulls the sum of the `world` replicas with multimem.ld_reduce (the switch adds
// them on the way) and pushes it back with multimem.st (the switch copies it into every
// replica).  Per GPU the NVLink carries (world-1)/world of the buffer in each direction once;
// nothing is staged, no rank reads another's memory element by element.
// flags (in the same multicast region, 64-bit counters that only grow):
//   [0] ranks whose partial sums are complete (the column kernel before this one has ended),
//   [1] ranks whose slice has been pushed to every replica ([2]: this rank's CTAs, local).
// The grid must be co-resident (at most one CTA per SM): CTAs spin on counters other CTAs raise.
// ---------------------------------------------------------------------------
enum { kNvlsUnroll = 2 };
__device__ __forceinline__ void nvls_signal(unsigned long long* mc_flag) {
    asm volatile("multimem.red.release.sys.global.add.u64 [%0], %1;" ::"l"(mc_flag), "l"(1ull) : "memory");
}
__device__ __forceinline__ void nvls_wait(const unsigned long long* uc_flag, unsigned long long target) {
    unsigned long long v;
    do {
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(uc_flag) : "memory");
    } while (v < target);
}
__global__ void __launch_bounds__(512) nvls_allreduce_f32_kernel(float* mc, size_t n4, unsigned long long* mc_flags,
                                                                 const unsigned long long* uc_flags, int rank,
                                                                 int world, unsigned long long epoch) {
    if (threadIdx.x == 0) {
        if (blockIdx.x == 0) nvls_signal(mc_flags + 0);
        nvls_wait(uc_flags + 0, epoch * (unsigned long long)world);
    }
    __syncthreads();
    const size_t lo = n4 * (size_t)rank / world, hi = n4 * (size_t)(rank + 1) / world;   // (n4 == 0: barriers only, a timing probe)
    // kNvlsUnroll reductions in flight per thread: a round trip through the switch is microseconds
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i0 = lo + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < hi; i0 += stride * kNvlsUnroll) {
        float v[kNvlsUnroll][4];
#pragma unroll
        for (int u = 0; u < kNvlsUnroll; ++u) {
            const size_t i = i0 + u * stride;
            if (i < hi)
                asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
                             : "=f"(v[u][0]), "=f"(v[u][1]), "=f"(v[u][2]), "=f"(v[u][3]) : "l"(mc + 4 * i) : "memory");
        }
#pragma unroll
        for (int u = 0; u < kNvlsUnroll; ++u) {
            const size_t i = i0 + u * stride;
            if (i < hi)
                asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};"
                             ::"l"(mc + 4 * i), "f"(v[u][0]), "f"(v[u][1]), "f"(v[u][2]), "f"(v[u][3]) : "memory");
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        // the CTAs of this rank count themselves on a local word; the last one tells every rank
        unsigned long long* local = (unsigned long long*)uc_flags + 2;
        const unsigned long long seen = atomicAdd(local, 1ull) + 1;
        if (seen == epoch * gridDim.x) nvls_signal(mc_flags + 1);
        nvls_wait(uc_flags + 1, epoch * (unsigned long long)world);
    }
}

template <typename T>
__global__ void __launch_bounds__(kEwThreads) rect_kernel(const lsted::RectArgs<T> a) {
    const size_t n = (size_t)a.nimg * a.h * a.w;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride)
        lsted::rect_apply<T>(a, e);
}

template <typename T>
__global__ void __launch_bounds__(256) otf_center_kernel(const lsted::OtfCenterArgs<T> a) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += stride)
        lsted::otf_center_apply<T>(a, i);
}

// Fused cross-GPU H_t reduction (conv_fast.cuh): the kernels after it on this stream may read
// the spectrum only when all column blocks -- finished by their owner ranks, over NVLink --
// have been counted.
__global__ void p2p_wait_kernel(const unsigned* done, unsigned target) {
    if (threadIdx.x == 0) lsted::flag_wait(done, target);
}

// Two-stage deterministic sum in double: per-block partials, then block 0.
__global__ void __launch_bounds__(256) sum_partial_kernel(const double* x, size_t n, double* partial) {
    __shared__ double sh[256];
    double s = 0;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) s += x[i];
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[blockIdx.x] = sh[0];
}
__global__ void __launch_bounds__(256) sum_final_kernel(double* partial, int nblocks) {
    __shared__ double sh[256];
    double s = 0;
    for (int i = threadIdx.x; i < nblocks; i += 256) s += partial[i];
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[0] = sh[0];
}

// ---------------------------------------------------------------------------
// NCCL, resolved at run time (dlopen) so that single-GPU use has no NCCL dependency
// ---------------------------------------------------------------------------
struct NcclApi {
    ncclResult_t (*GetUniqueId)(ncclUniqueId*);
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int);
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t,
                              cudaStream_t);
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*CommDestroy)(ncclComm_t);
    const char* (*GetErrorString)(ncclResult_t);
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*GroupStart)();
    ncclResult_t (*GroupEnd)();
    bool ok;
};
static NcclApi& nccl_api() {
    static NcclApi api = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, false};
    if (api.ok) return api;
    void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) {
        lsted::ApiError e; e.code = LSTED_ERR_NCCL;
        e.msg = std::string("cannot load libnccl.so.2: ") + dlerror();
        throw e;
    }
    api.GetUniqueId = (ncclResult_t(*)(ncclUniqueId*))dlsym(lib, "ncclGetUniqueId");
    api.CommInitRank = (ncclResult_t(*)(ncclComm_t*, int, ncclUniqueId, int))dlsym(lib, "ncclCommInitRank");
    api.AllReduce = (ncclResult_t(*)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t,
                                     cudaStream_t))dlsym(lib, "ncclAllReduce");
    api.Broadcast = (ncclResult_t(*)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t,
                                     cudaStream_t))dlsym(lib, "ncclBroadcast");
    api.CommDestroy = (ncclResult_t(*)(ncclComm_t))dlsym(lib, "ncclCommDestroy");
    api.GetErrorString = (const char* (*)(ncclResult_t))dlsym(lib, "ncclGetErrorString");
    api.Send = (ncclResult_t(*)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t))dlsym(lib, "ncclSend");
    api.Recv = (ncclResult_t(*)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t))dlsym(lib, "ncclRecv");
    api.GroupStart = (ncclResult_t(*)())dlsym(lib, "ncclGroupStart");
    api.GroupEnd = (ncclResult_t(*)())dlsym(lib, "ncclGroupEnd");
    if (!api.Send || !api.Recv || !api.GroupStart || !api.GroupEnd || !api.Broadcast || !api.GetUniqueId || !api.CommInitRank || !api.AllReduce || !api.CommDestroy || !api.GetErrorString) {
        lsted::ApiError e; e.code = LSTED_ERR_NCCL; e.msg = "libnccl lacks a required symbol";
        throw e;
    }
    api.ok = true;
    return api;
}
#define NCCL_CHECK(expr)                                                                  \
    do {                                                                                  \
        ncclResult_t res__ = (expr);                                                      \
        if (res__ != ncclSuccess) {                                                       \
            lsted::ApiError e__;                                                          \
            e__.code = LSTED_ERR_NCCL;                                                    \
            e__.msg = std::string(#expr) + ": " + nccl_api().GetErrorString(res__);       \
            throw e__;                                                                    \
        }                                                                                 \
    } while (0)

// ---------------------------------------------------------------------------
// CUDA backend of the engine
// ---------------------------------------------------------------------------
// Deconvolver handles alive in this process: with many of them (figure 2 iterates 24 round-robin,
// each on its own stream) the GPU is kept busy by the other handles' kernels and spreading one
// frame's orientations over more CTAs only adds work (measured: 24 handles 6.5 -> 7.5 us / iteration).
static int g_live_backends = 0;

class CudaBackend : public lsted::KernelSelection {
  public:
    explicit CudaBackend(int device) : device_(device), stream_(0), bytes_(0), profile_(false),
                                       t0_(0), t1_(0), num_sms_(148) {
        int count = 0;
        CUDA_CHECK(cudaGetDeviceCount(&count));
        if (device < 0 || device >= count) {
            lsted::ApiError e; e.code = LSTED_ERR_CUDA;
            e.msg = "CUDA device " + std::to_string(device) + " not available (" +
                    std::to_string(count) + " visible); there is no CPU fallback";
            throw e;
        }
        CUDA_CHECK(cudaSetDevice(device));
        CUDA_CHECK(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
        CUDA_CHECK(cudaEventCreate(&t0_));
        CUDA_CHECK(cudaEventCreate(&t1_));
        CUDA_CHECK(cudaDeviceGetAttribute(&num_sms_, cudaDevAttrMultiProcessorCount, device));
        ++g_live_backends;
        memset(prof_ms_, 0, sizeof(prof_ms_));
        memset(prof_n_, 0, sizeof(prof_n_));
        const char* pq = getenv("LSTED_PREFETCH_CTAS_PER_SM");   // prefetch distance in CTAs per SM
        if (pq && atoi(pq) > 0) { prefetch_quarters_ = atoi(pq); prefetch_final_quarters_ = 0; }
    }
    ~CudaBackend() {
        cudaSetDevice(device_);
        --g_live_backends;
        try { nvls_release(); } catch (...) {}
        for (size_t i = 0; i < p2p_opened_.size(); ++i) cudaIpcCloseMemHandle(p2p_opened_[i]);
        if (comm_) nccl_api().CommDestroy(comm_);
        for (size_t i = 0; i < ev_pool_.size(); ++i) cudaEventDestroy(ev_pool_[i]);
        if (t0_) cudaEventDestroy(t0_);
        if (t1_) cudaEventDestroy(t1_);
        if (stream_) cudaStreamDestroy(stream_);
    }
    void activate() { CUDA_CHECK(cudaSetDevice(device_)); }
    void sync() { CUDA_CHECK(cudaStreamSynchronize(stream_)); }

    // ---- collectives (orientation sharding) ----
    void comm_init(const char* unique_id, int rank, int world) {
        if (!unique_id) { lsted::ApiError e; e.code = LSTED_ERR_ARG; e.msg = "null NCCL id"; throw e; }
        if (comm_) { nccl_api().CommDestroy(comm_); comm_ = 0; }
        ncclUniqueId id;
        memcpy(id.internal, unique_id, sizeof(id.internal));
        NCCL_CHECK(nccl_api().CommInitRank(&comm_, world, id, rank));
    }
    void all_reduce_sum(float* p, size_t n) {
        before(lsted::KK_EW);
        NCCL_CHECK(nccl_api().AllReduce(p, p, n, ncclFloat, ncclSum, comm_, stream_));
        after();
    }
    void all_reduce_sum(double* p, size_t n) {
        before(lsted::KK_EW);
        NCCL_CHECK(nccl_api().AllReduce(p, p, n, ncclDouble, ncclSum, comm_, stream_));
        after();
    }
    void broadcast(float* p, size_t n, int root) {
        before(lsted::KK_EW);
        NCCL_CHECK(nccl_api().Broadcast(p, p, n, ncclFloat, root, comm_, stream_));
        after();
    }
    void broadcast(double* p, size_t n, int root) {
        before(lsted::KK_EW);
        NCCL_CHECK(nccl_api().Broadcast(p, p, n, ncclDouble, root, comm_, stream_));
        after();
    }
    // ---- NVLS: all-reduce through the NVSwitch over a CUDA multicast object (fp32 spectra) ----
    // Driver entry points are looked up at run time (no libcuda link dependency).
    template <class Fn> static Fn drv(const char* name) {
        void* fn = 0;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint(name, &fn, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess || !fn) {
            lsted::ApiError e; e.code = LSTED_ERR_CUDA; e.msg = std::string("driver entry point missing: ") + name; throw e;
        }
        return (Fn)fn;
    }
    static void cu_check(CUresult r, const char* what) {
        if (r == CUDA_SUCCESS) return;
        lsted::ApiError e; e.code = LSTED_ERR_CUDA;
        e.msg = std::string(what) + " failed with CUresult " + std::to_string((int)r);
        throw e;
    }
    static bool nvls_device_supported(int device) {
        int v = 0;
        typedef CUresult (*attr_fn)(int*, CUdevice_attribute, CUdevice);
        typedef CUresult (*get_fn)(CUdevice*, int);
        CUdevice d;
        if (drv<get_fn>("cuDeviceGet")(&d, device) != CUDA_SUCCESS) return false;
        if (drv<attr_fn>("cuDeviceGetAttribute")(&v, CU_DEVICE_ATTRIBUTE_MULTICAST_SUPPORTED, d) != CUDA_SUCCESS) return false;
        return v != 0;
    }
    // multicast region = data (16-byte multiple) + 256 bytes of counters, rounded up to the
    // granularity of multicast objects and of physical allocations on this device
    size_t nvls_region_bytes(size_t data_bytes, int world) {
        CUmulticastObjectProp mp;
        memset(&mp, 0, sizeof(mp));
        mp.numDevices = world; mp.size = data_bytes + 256; mp.handleTypes = CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR;
        size_t g1 = 0, g2 = 0;
        typedef CUresult (*gran_fn)(size_t*, const CUmulticastObjectProp*, CUmulticastGranularity_flags);
        cu_check(drv<gran_fn>("cuMulticastGetGranularity")(&g1, &mp, CU_MULTICAST_GRANULARITY_MINIMUM), "cuMulticastGetGranularity");
        CUmemAllocationProp ap = nvls_alloc_prop();
        typedef CUresult (*agran_fn)(size_t*, const CUmemAllocationProp*, CUmemAllocationGranularity_flags);
        cu_check(drv<agran_fn>("cuMemGetAllocationGranularity")(&g2, &ap, CU_MEM_ALLOC_GRANULARITY_MINIMUM), "cuMemGetAllocationGranularity");
        const size_t g = g1 > g2 ? g1 : g2;
        nvls_gran_ = g;
        return (data_bytes + 256 + g - 1) / g * g;
    }
    CUmemAllocationProp nvls_alloc_prop() const {
        CUmemAllocationProp ap;
        memset(&ap, 0, sizeof(ap));
        ap.type = CU_MEM_ALLOCATION_TYPE_PINNED;
        ap.location.type = CU_MEM_LOCATION_TYPE_DEVICE; ap.location.id = device_;
        ap.requestedHandleTypes = CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR;
        return ap;
    }
    // one multicast team per handle: a bound region is the handle's spectrum until it is destroyed
    void nvls_refuse_rebind() {
        if (nvls_bound_) {
            lsted::ApiError e; e.code = LSTED_ERR_STATE; e.msg = "this handle is already bound to a multicast object"; throw e;
        }
        if (nvls_have_mc_) nvls_release();   // an attach that was abandoned half way
    }
    // rank 0: create the multicast object, hand out a POSIX file descriptor of it
    int nvls_create(int world, size_t data_bytes) {
        nvls_refuse_rebind();
        nvls_world_ = world; nvls_data_bytes_ = (data_bytes + 15) / 16 * 16;
        nvls_bytes_ = nvls_region_bytes(nvls_data_bytes_, world);
        CUmulticastObjectProp mp;
        memset(&mp, 0, sizeof(mp));
        mp.numDevices = world; mp.size = nvls_bytes_; mp.handleTypes = CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR;
        typedef CUresult (*create_fn)(CUmemGenericAllocationHandle*, const CUmulticastObjectProp*);
        cu_check(drv<create_fn>("cuMulticastCreate")(&nvls_mc_, &mp), "cuMulticastCreate");
        int fd = -1;
        typedef CUresult (*export_fn)(void*, CUmemGenericAllocationHandle, CUmemAllocationHandleType, unsigned long long);
        cu_check(drv<export_fn>("cuMemExportToShareableHandle")(&fd, nvls_mc_, CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR, 0),
                 "cuMemExportToShareableHandle");
        nvls_have_mc_ = true;
        return fd;
    }
    // other ranks: import the object from a duplicate of rank 0's descriptor
    void nvls_import(int world, size_t data_bytes, int fd) {
        nvls_refuse_rebind();
        nvls_world_ = world; nvls_data_bytes_ = (data_bytes + 15) / 16 * 16;
        nvls_bytes_ = nvls_region_bytes(nvls_data_bytes_, world);
        typedef CUresult (*import_fn)(CUmemGenericAllocationHandle*, void*, CUmemAllocationHandleType);
        cu_check(drv<import_fn>("cuMemImportFromShareableHandle")(&nvls_mc_, (void*)(uintptr_t)fd,
                                                                  CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR),
                 "cuMemImportFromShareableHandle");
        nvls_have_mc_ = true;
    }
    void nvls_add_device() {
        typedef CUresult (*get_fn)(CUdevice*, int);
        typedef CUresult (*add_fn)(CUmemGenericAllocationHandle, CUdevice);
        CUdevice d;
        cu_check(drv<get_fn>("cuDeviceGet")(&d, device_), "cuDeviceGet");
        cu_check(drv<add_fn>("cuMulticastAddDevice")(nvls_mc_, d), "cuMulticastAddDevice");
    }
    // after every rank has added its device: back the region with local memory, map both views
    void* nvls_bind(int rank) {
        if (!nvls_have_mc_ || nvls_bound_) {
            lsted::ApiError e; e.code = LSTED_ERR_STATE; e.msg = "nvls_bind: create / import the multicast object first (once)"; throw e;
        }
        typedef CUresult (*mcreate_fn)(CUmemGenericAllocationHandle*, size_t, const CUmemAllocationProp*, unsigned long long);
        typedef CUresult (*bind_fn)(CUmemGenericAllocationHandle, size_t, CUmemGenericAllocationHandle, size_t, size_t, unsigned long long);
        typedef CUresult (*reserve_fn)(CUdeviceptr*, size_t, size_t, CUdeviceptr, unsigned long long);
        typedef CUresult (*map_fn)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long);
        typedef CUresult (*access_fn)(CUdeviceptr, size_t, const CUmemAccessDesc*, size_t);
        CUmemAllocationProp ap = nvls_alloc_prop();
        cu_check(drv<mcreate_fn>("cuMemCreate")(&nvls_mem_, nvls_bytes_, &ap, 0), "cuMemCreate");
        cu_check(drv<bind_fn>("cuMulticastBindMem")(nvls_mc_, 0, nvls_mem_, 0, nvls_bytes_, 0), "cuMulticastBindMem");
        CUmemAccessDesc ad;
        memset(&ad, 0, sizeof(ad));
        ad.location.type = CU_MEM_LOCATION_TYPE_DEVICE; ad.location.id = device_; ad.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
        cu_check(drv<reserve_fn>("cuMemAddressReserve")(&nvls_uc_, nvls_bytes_, nvls_gran_, 0, 0), "cuMemAddressReserve");
        cu_check(drv<map_fn>("cuMemMap")(nvls_uc_, nvls_bytes_, 0, nvls_mem_, 0), "cuMemMap (unicast)");
        cu_check(drv<access_fn>("cuMemSetAccess")(nvls_uc_, nvls_bytes_, &ad, 1), "cuMemSetAccess (unicast)");
        cu_check(drv<reserve_fn>("cuMemAddressReserve")(&nvls_mcp_, nvls_bytes_, nvls_gran_, 0, 0), "cuMemAddressReserve");
        cu_check(drv<map_fn>("cuMemMap")(nvls_mcp_, nvls_bytes_, 0, nvls_mc_, 0), "cuMemMap (multicast)");
        cu_check(drv<access_fn>("cuMemSetAccess")(nvls_mcp_, nvls_bytes_, &ad, 1), "cuMemSetAccess (multicast)");
        CUDA_CHECK(cudaMemsetAsync((void*)nvls_uc_, 0, nvls_bytes_, stream_));
        CUDA_CHECK(cudaStreamSynchronize(stream_));
        nvls_rank_ = rank; nvls_epoch_ = 0; nvls_bound_ = true;
        bytes_ += nvls_bytes_;
        return (void*)nvls_uc_;
    }
    void nvls_release() {
        if (!nvls_have_mc_) return;
        typedef CUresult (*unmap_fn)(CUdeviceptr, size_t);
        typedef CUresult (*release_fn)(CUmemGenericAllocationHandle);
        typedef CUresult (*afree_fn)(CUdeviceptr, size_t);
        if (nvls_bound_) {
            drv<unmap_fn>("cuMemUnmap")(nvls_mcp_, nvls_bytes_);
            drv<unmap_fn>("cuMemUnmap")(nvls_uc_, nvls_bytes_);
            drv<afree_fn>("cuMemAddressFree")(nvls_mcp_, nvls_bytes_);
            drv<afree_fn>("cuMemAddressFree")(nvls_uc_, nvls_bytes_);
            drv<release_fn>("cuMemRelease")(nvls_mem_);
        }
        drv<release_fn>("cuMemRelease")(nvls_mc_);
        nvls_have_mc_ = nvls_bound_ = false;
    }
    bool nvls_ready(const void* buf) const { return nvls_bound_ && buf == (const void*)nvls_uc_; }
    // in-place sum over the ranks of the fp32 buffer that nvls_bind returned
    void nvls_allreduce(float* buf, size_t n) {
        if (!nvls_ready(buf) || n * sizeof(float) > nvls_data_bytes_) {
            lsted::ApiError e; e.code = LSTED_ERR_STATE; e.msg = "NVLS all-reduce on a buffer that is not bound"; throw e;
        }
        unsigned long long* mc_flags = (unsigned long long*)((char*)nvls_mcp_ + nvls_data_bytes_);
        const unsigned long long* uc_flags = (const unsigned long long*)((char*)nvls_uc_ + nvls_data_bytes_);
        before(lsted::KK_EW);
        // 32 CTAs x 512 threads: measured on 8 GPUs (17.8 MB): 0.061 ms, of which 0.024 ms are the two
        // cross-GPU barriers; 148 CTAs: 0.072, 8 CTAs: 0.065 (scripts/nvls_sweep.py)
        const int ctas = nvls_ctas_ > 0 && nvls_ctas_ <= num_sms_ ? nvls_ctas_ : (num_sms_ < 32 ? num_sms_ : 32);
        const int threads = nvls_threads_ >= 32 && nvls_threads_ <= 512 ? nvls_threads_ / 32 * 32 : 512;
        nvls_allreduce_f32_kernel<<<ctas, threads, 0, stream_>>>((float*)nvls_mcp_, nvls_probe_ ? 0 : (n + 3) / 4, mc_flags, uc_flags,
                                                                 nvls_rank_, nvls_world_, ++nvls_epoch_);
        after();
    }
    void nvls_allreduce(double*, size_t) {
        lsted::ApiError e; e.code = LSTED_ERR_STATE; e.msg = "the NVLS all-reduce is built for fp32 spectra"; throw e;
    }

    // Halo exchange of a tile-sharded object (tiled.h): one grouped ncclSend / ncclRecv pair per
    // neighbour, contiguous staging buffers (counts in elements of T).
    template <typename T> void exchange(int npeers, const int* peers, T* const* send, const size_t* nsend,
                                        T* const* recv, const size_t* nrecv) {
        const ncclDataType_t dt = sizeof(T) == 4 ? ncclFloat : ncclDouble;
        before(lsted::KK_EW);
        NCCL_CHECK(nccl_api().GroupStart());
        for (int i = 0; i < npeers; ++i) {
            if (nsend[i]) NCCL_CHECK(nccl_api().Send(send[i], nsend[i], dt, peers[i], comm_, stream_));
            if (nrecv[i]) NCCL_CHECK(nccl_api().Recv(recv[i], nrecv[i], dt, peers[i], comm_, stream_));
        }
        NCCL_CHECK(nccl_api().GroupEnd());
        after();
    }
    template <typename T> void launch_rect(const lsted::RectArgs<T>& a) {
        const size_t n = (size_t)a.nimg * a.h * a.w;
        if (n == 0) return;
        size_t blocks = (n + kEwThreads - 1) / kEwThreads;
        const size_t cap = (size_t)num_sms_ * 16;
        if (blocks > cap) blocks = cap;
        before(lsted::KK_EW);
        rect_kernel<T><<<(int)blocks, kEwThreads, 0, stream_>>>(a);
        after();
    }
    // ---- fused cross-GPU reduction over peer memory (orientation sharding, fast path) ----
    // Buffers are plain cudaMalloc allocations exported / opened with CUDA IPC (one process
    // per GPU); `handles` = [world][3] cudaIpcMemHandle_t: receive slabs, flags, spectrum.
    enum { kIpcBytes = 3 * (int)sizeof(cudaIpcMemHandle_t) };
    void p2p_export(void* recv, void* flags, void* spec, char* out) {
        void* ptrs[3] = {recv, flags, spec};
        for (int i = 0; i < 3; ++i) {
            cudaIpcMemHandle_t h;
            CUDA_CHECK(cudaIpcGetMemHandle(&h, ptrs[i]));
            memcpy(out + i * sizeof(h), &h, sizeof(h));
        }
        p2p_local_[0] = recv; p2p_local_[1] = flags; p2p_local_[2] = spec;
    }
    void p2p_attach(int rank, int world, const char* handles, size_t done_offset_words) {
        if (world > lsted::kMaxPeers) {
            lsted::ApiError e; e.code = LSTED_ERR_ARG; e.msg = "too many ranks for the peer-memory reduction"; throw e;
        }
        for (int r = 0; r < world; ++r) {
            void* ptrs[3];
            for (int i = 0; i < 3; ++i) {
                if (r == rank) { ptrs[i] = p2p_local_[i]; continue; }
                cudaIpcMemHandle_t h;
                memcpy(&h, handles + ((size_t)r * 3 + i) * sizeof(h), sizeof(h));
                CUDA_CHECK(cudaIpcOpenMemHandle(&ptrs[i], h, cudaIpcMemLazyEnablePeerAccess));
                p2p_opened_.push_back(ptrs[i]);
            }
            p2p_recv_[r] = ptrs[0];
            p2p_flags_[r] = (unsigned*)ptrs[1];
            p2p_done_[r] = (unsigned*)ptrs[1] + done_offset_words;
            p2p_spec_[r] = ptrs[2];
        }
        p2p_rank_ = rank; p2p_world_ = world; p2p_epoch_ = 0;
    }
    bool p2p_ready(const lsted::ConvGeom& g, int cplx_bytes) const {
        return p2p_world_ > 1 && sw.fast_path && lsted::fast_plan_fits_cols(g, cplx_bytes);
    }
    template <typename T> void p2p_fill(lsted::ColArgs<T>& a) {
        a.p2p_world = p2p_world_; a.p2p_rank = p2p_rank_; a.p2p_epoch = ++p2p_epoch_;
        for (int r = 0; r < p2p_world_; ++r) {
            a.p2p_recv[r] = (lsted::cplx<T>*)p2p_recv_[r];
            a.p2p_flags[r] = p2p_flags_[r];
            a.p2p_spec[r] = (lsted::cplx<T>*)p2p_spec_[r];
            a.p2p_done[r] = p2p_done_[r];
        }
    }
    // blocks counted on this rank so far = epoch * nxb
    void p2p_wait(int nxb) {
        before(lsted::KK_EW);
        p2p_wait_kernel<<<1, 32, 0, stream_>>>(p2p_done_[p2p_rank_], p2p_epoch_ * (unsigned)nxb);
        after();
    }
    void zero_bytes(void* p, size_t n) { CUDA_CHECK(cudaMemsetAsync(p, 0, n, stream_)); }
    template <typename T> void otf_center(const lsted::OtfCenterArgs<T>& a0) {
        lsted::OtfCenterArgs<T> a = a0;   // the real array is read by the compile-time plans only
        a.CS = (int)lsted::PlanFor<T>::type::CS;
        before(lsted::KK_EW);
        otf_center_kernel<T><<<num_sms_ * 8, 256, 0, stream_>>>(a);
        after();
    }
    void fill_double(double* p, size_t n, double v) {
        if (v != 0.0) { lsted::ApiError e; e.code = LSTED_ERR_ARG; e.msg = "fill_double: zero only"; throw e; }
        CUDA_CHECK(cudaMemsetAsync(p, 0, n * sizeof(double), stream_));
    }
    cudaStream_t stream() const { return stream_; }

    void* alloc(size_t bytes) {
        void* p = 0;
        CUDA_CHECK(cudaMalloc(&p, bytes ? bytes : 1));
        bytes_ += bytes;
        sizes_[p] = bytes;
        return p;
    }
    void free(void* p) {
        if (!p) return;
        if (p == (void*)nvls_uc_) return;   // multicast-bound region: unmapped by nvls_release()
        std::map<void*, size_t>::iterator it = sizes_.find(p);
        if (it != sizes_.end()) { bytes_ -= it->second; sizes_.erase(it); }
        cudaFree(p);
    }
    size_t bytes_allocated() const { return bytes_; }
    void upload(void* d, const void* s, size_t n) {
        CUDA_CHECK(cudaMemcpyAsync(d, s, n, cudaMemcpyHostToDevice, stream_));
    }
    void download(void* d, const void* s, size_t n) {
        CUDA_CHECK(cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToHost, stream_));
        sync();
    }

    // ---- timing ----
    void timer_start() { CUDA_CHECK(cudaEventRecord(t0_, stream_)); }
    float timer_stop() {
        CUDA_CHECK(cudaEventRecord(t1_, stream_));
        CUDA_CHECK(cudaEventSynchronize(t1_));
        float ms = 0;
        CUDA_CHECK(cudaEventElapsedTime(&ms, t0_, t1_));
        return ms;
    }
    void set_profile(bool on) { profile_ = on; }
    void set_nvls_probe(bool on) { nvls_probe_ = on; }
    void set_nvls_shape(int ctas, int threads) { if (ctas >= 0) nvls_ctas_ = ctas; if (threads > 0) nvls_threads_ = threads; }
    // ---- CUDA graphs: the steady RL iteration replayed as one driver call (engine.h) ----
    void set_graph(bool on) { graph_ = on; }
    bool graph_capable() const { return graph_ && !profile_; }
    void graph_begin() { CUDA_CHECK(cudaStreamBeginCapture(stream_, cudaStreamCaptureModeThreadLocal)); }
    void graph_abort() {
        cudaGraph_t g = 0;
        cudaStreamEndCapture(stream_, &g);
        if (g) cudaGraphDestroy(g);
        cudaGetLastError();
    }
    void* graph_end() {
        cudaGraph_t g = 0;
        CUDA_CHECK(cudaStreamEndCapture(stream_, &g));
        cudaGraphExec_t exec = 0;
        cudaError_t err = cudaGraphInstantiate(&exec, g, 0);
        cudaGraphDestroy(g);
        CUDA_CHECK(err);
        return (void*)exec;
    }
    void graph_launch(void* exec) { CUDA_CHECK(cudaGraphLaunch((cudaGraphExec_t)exec, stream_)); }
    void graph_destroy(void* exec) { if (exec) cudaGraphExecDestroy((cudaGraphExec_t)exec); }
    // row CTAs resident at once (4 per SM): prefetch for the CTA one wave ahead
    int row_prefetch_distance() const { return sw.prefetch ? (num_sms_ * prefetch_quarters_) : 0; }
    // ROW_FINAL has few CTAs (one image): its prefetch must reach past everything resident
    // (4 CTAs per SM) to be of any use -- measured best at 6 CTAs per SM ahead
    int row_final_prefetch_distance() const {
        return sw.prefetch ? num_sms_ * (prefetch_final_quarters_ > 0 ? prefetch_final_quarters_ : prefetch_quarters_) : 0;
    }
    void profile_reset() {
        profile_drain();
        memset(prof_ms_, 0, sizeof(prof_ms_));
        memset(prof_n_, 0, sizeof(prof_n_));
    }
    void profile_collect(double* ms, long long* n) {
        profile_drain();
        for (int i = 0; i < LSTED_NUM_KERNEL_KINDS; ++i) {
            if (ms) ms[i] = prof_ms_[i];
            if (n) n[i] = prof_n_[i];
        }
    }

    // ---- launches ----
    // MaxDynamicSharedMemorySize is a per-device function attribute: remembered per backend
    // (one backend = one device), not in process-wide statics.
    template <class F> void ensure_smem(F* fn, size_t smem) {
        size_t& have = smem_cfg_[(const void*)fn];
        if (smem <= have) return;
        CUDA_CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        have = smem;
    }
    // CUtensorMap (in global memory) of a row-spectrum array: [nimg][nxb][rows_e * C * 2 floats],
    // box = {floats of one pair chunk, kTmaBoxBlocks, 1}.  Returns 0 when tensor maps are unavailable.
    void* make_spec_tmap(void* base, int rows_e, int nxb, int C, int nimg, int chunk_floats) {
        typedef CUresult (*encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                      const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                      CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                      CUtensorMapFloatOOBfill);
        static encode_fn encode = 0;
        if (!encode) {
            void* fn = 0;
            cudaDriverEntryPointQueryResult qres;
            if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess ||
                qres != cudaDriverEntryPointSuccess || !fn)
                return 0;
            encode = (encode_fn)fn;
        }
        CUtensorMap map;
        const cuuint64_t dims[3] = {(cuuint64_t)rows_e * C * 2, (cuuint64_t)nxb, (cuuint64_t)nimg};
        const cuuint64_t strides[2] = {(cuuint64_t)rows_e * C * 2 * sizeof(float),
                                       (cuuint64_t)nxb * rows_e * C * 2 * sizeof(float)};
        const cuuint32_t box[3] = {(cuuint32_t)chunk_floats, (cuuint32_t)lsted::kTmaBoxBlocks, 1};
        const cuuint32_t estr[3] = {1, 1, 1};
        if (encode(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base, dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                   CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return 0;
        void* d = alloc(sizeof(map));
        CUDA_CHECK(cudaMemcpyAsync(d, &map, sizeof(map), cudaMemcpyHostToDevice, stream_));
        CUDA_CHECK(cudaStreamSynchronize(stream_));
        return d;
    }
    // ---- launches: dispatch.h chooses the kernel instance, the executors below run it ----
    template <int MODE, typename T> void launch_row(int grid, const lsted::RowArgs<T>& a) {
        lsted::run_row<MODE>(*this, lsted::select_row<MODE>(grid, a, sw), a);
    }
    template <int MODE, typename T> void launch_col(int grid, const lsted::ColArgs<T>& a) {
        const lsted::DeviceShape dev = {num_sms_, g_live_backends, num_sms_};   // split up to the SM count
        lsted::run_col<MODE>(*this, lsted::select_col<MODE>(grid, a, sw, dev), a);
    }
    template <int MODE, typename T> void row_generic(const lsted::RowChoice& c, const lsted::RowArgs<T>& a) {
        const size_t smem = lsted::row_smem_bytes(a.g, (int)sizeof(lsted::cplx<T>));
        ensure_smem(row_kernel<MODE, T>, smem);
        before(c.kind);
        row_kernel<MODE, T><<<c.grid, kRowThreads, smem, stream_>>>(a);
        after();
    }
    template <int MODE, class P, class G, int TMA>
    void row_fast(const lsted::RowChoice& c, const lsted::RowArgs<typename P::T>& a) {
        const size_t smem = lsted::fast_row_smem_bytes<P>(MODE, TMA == 2);
        ensure_smem(row_fast_kernel<MODE, P, G, TMA>, smem);
        before(c.kind);
        row_fast_kernel<MODE, P, G, TMA><<<c.grid, P::ROW_THREADS, smem, stream_>>>(a);
        after();
    }
    // the two-pass and the dual-pair row kernels prefetch one wave of their own CTAs ahead
    template <int MODE, class P> void row2(const lsted::RowChoice& c, const lsted::RowArgs<float>& a) {
        const size_t smem = lsted::fast_row2_smem_bytes<P>(MODE);
        ensure_smem(row2_fast_kernel<MODE, P>, smem);
        lsted::RowArgs<float> b = a;
        if (b.prefetch_ahead > 0) b.prefetch_ahead = num_sms_ * LSTED_ROW2_CTAS;
        before(c.kind);
        row2_fast_kernel<MODE, P><<<c.grid, P::ROW_THREADS, smem, stream_>>>(b);
        after();
    }
    template <class P> void row_mid_dual(const lsted::RowChoice& c, const lsted::RowArgs<float>& a) {
        typedef lsted::RowDual<P> D;
        ensure_smem(row_mid_dual_kernel<P>, D::smem_bytes());
        lsted::RowArgs<float> b = a;
        if (b.prefetch_ahead > 0) b.prefetch_ahead = num_sms_ * 2;   // two CTAs per SM
        before(c.kind);
        row_mid_dual_kernel<P><<<c.grid, D::THREADS, D::smem_bytes(), stream_>>>(b);
        after();
    }
    template <int MODE, typename T> void col_generic(const lsted::ColChoice& c, const lsted::ColArgs<T>& a) {
        const size_t smem = lsted::col_smem_bytes(a.g, (int)sizeof(lsted::cplx<T>), MODE == lsted::COL_OTF ? 2 : 3);
        ensure_smem(col_kernel<MODE, T>, smem);
        before(c.kind);
        col_kernel<MODE, T><<<c.grid, sizeof(T) == 4 ? kColThreads32 : kColThreads64, smem, stream_>>>(a);
        after();
    }
    template <int MODE, class P, class G, bool RO>
    void col_fast(const lsted::ColChoice& c, const lsted::ColArgs<typename P::T>& a) {
        const size_t smem = lsted::fast_col_smem_bytes<P>();
        ensure_smem(col_fast_kernel<MODE, P, G, RO>, smem);
        before(c.kind);
        col_fast_kernel<MODE, P, G, RO><<<c.grid, P::COL_THREADS, smem, stream_>>>(a);
        after();
    }
    template <int MODE, class P, class G>
    void col_sub(const lsted::ColChoice& c, const lsted::ColArgs<typename P::T>& a) {
        const size_t smem = lsted::fast_col_sub_smem_bytes<P>();
        ensure_smem(col_sub_kernel<MODE, P, G>, smem);
        before(c.kind);
        col_sub_kernel<MODE, P, G><<<c.grid, P::SUB_THREADS, smem, stream_>>>(a);
        after();
    }
    // persistent: at most one CTA per SM, each walks several column blocks
    template <class P, bool RO> void col_ht_p2p(const lsted::ColChoice& c, const lsted::ColArgs<typename P::T>& a) {
        const size_t smem = lsted::fast_col_smem_bytes<P>();
        ensure_smem(col_ht_p2p_kernel<P, RO>, smem);
        before(c.kind);
        col_ht_p2p_kernel<P, RO><<<c.grid < num_sms_ ? c.grid : num_sms_, P::COL_THREADS, smem, stream_>>>(a);
        after();
    }
    template <int OP, typename T> void ew(const lsted::EwArgs<T>& a) {
        if (a.n == 0) return;
        size_t blocks = (a.n + kEwThreads - 1) / kEwThreads;
        const size_t cap = (size_t)num_sms_ * 16;
        if (blocks > cap) blocks = cap;
        before(lsted::KK_EW);
        ew_kernel<OP, T><<<(int)blocks, kEwThreads, 0, stream_>>>(a);
        after();
    }
    // record_iteration's error spectrum on sides without a Stockham plan (ew_bodies.cuh)
    template <int PASS, typename T> void dft_direct(const lsted::DftArgs<T>& a) {
        const size_t n = (size_t)a.Ny * a.Nx;
        if (n == 0) return;
        const size_t blocks = (n + kEwThreads - 1) / kEwThreads;   // one bin per thread: O(N) work each
        before(lsted::KK_EW);
        dft_direct_kernel<PASS, T><<<(unsigned)blocks, kEwThreads, 0, stream_>>>(a);
        after();
    }
    template <int OP, typename T> void launch_win(const lsted::WinArgs<T>& a) {
        const size_t n = (size_t)a.nimg * a.W * a.W;
        if (n == 0) return;
        size_t blocks = (n + kEwThreads - 1) / kEwThreads;
        const size_t cap = (size_t)num_sms_ * 16;
        if (blocks > cap) blocks = cap;
        before(lsted::KK_EW);
        win_kernel<OP, T><<<(int)blocks, kEwThreads, 0, stream_>>>(a);
        after();
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
    // generic column kernel in COL_LOGMAG mode (record_iteration's error spectrum)
    template <typename T> void launch_col_logmag(int grid, const lsted::ColArgs<T>& a) {
        const size_t smem = lsted::col_smem_bytes(a.g, (int)sizeof(lsted::cplx<T>), 2);
        ensure_smem(col_kernel<lsted::COL_LOGMAG, T>, smem);
        const int threads = sizeof(T) == 4 ? kColThreads32 : kColThreads64;
        before(lsted::KK_EW);
        col_kernel<lsted::COL_LOGMAG, T><<<grid, threads, smem, stream_>>>(a);
        after();
    }
    template <typename T> void rl_update(T* est, const T* num, const T* den, size_t n) {
        lsted::EwArgs<T> a; memset(&a, 0, sizeof(a)); a.t0 = est; a.t1 = num; a.t2 = den; a.n = n;
        ew<lsted::EW_RL_UPDATE, T>(a);
    }
    double sum(const double* x, size_t n, double* partial) {
        const int blocks = 1024;
        before(lsted::KK_EW);
        sum_partial_kernel<<<blocks, 256, 0, stream_>>>(x, n, partial);
        sum_final_kernel<<<1, 256, 0, stream_>>>(partial, blocks);
        after();
        double s = 0;
        download(&s, partial, sizeof(double));
        return s;
    }

  private:
    int device_;
    cudaStream_t stream_;
    size_t bytes_;
    // NVLS state
    CUmemGenericAllocationHandle nvls_mc_ = 0, nvls_mem_ = 0;
    CUdeviceptr nvls_uc_ = 0, nvls_mcp_ = 0;
    size_t nvls_bytes_ = 0, nvls_data_bytes_ = 0, nvls_gran_ = 0;
    int nvls_world_ = 1, nvls_rank_ = 0;
    unsigned long long nvls_epoch_ = 0;
    bool nvls_have_mc_ = false, nvls_bound_ = false;
    int nvls_ctas_ = 0, nvls_threads_ = 512;   // options "nvls_ctas" / "nvls_threads" (tuning)
    bool nvls_probe_ = false;                  // option "nvls_probe": barriers only (timing; results are wrong)
    bool profile_;
    bool graph_ = getenv("LSTED_GRAPH") ? atoi(getenv("LSTED_GRAPH")) != 0 : true;   // A/B switch, option "graph"
    std::map<void*, size_t> sizes_;   // live allocations (for lsted_deconv_info)
    std::map<const void*, size_t> smem_cfg_;   // kernels whose dynamic shared-memory limit is raised
    void* p2p_local_[3] = {0, 0, 0};
    void* p2p_recv_[lsted::kMaxPeers]; unsigned* p2p_flags_[lsted::kMaxPeers];
    void* p2p_spec_[lsted::kMaxPeers]; unsigned* p2p_done_[lsted::kMaxPeers];
    std::vector<void*> p2p_opened_;
    int p2p_rank_ = 0, p2p_world_ = 1; unsigned p2p_epoch_ = 0;
    int prefetch_quarters_ = 1;   // row-kernel L2 prefetch distance in CTAs per SM.  With per-thread
                                  // loads it was worth 14 % of row_mid; with the TMA-staged kernels
                                  // it hardly matters for row_mid (1: 0.196, 2: 0.197, 4: 0.199, 8: 0.213 ms)
    int prefetch_final_quarters_ = 6;   // ROW_FINAL (1024 CTAs, 592 resident): 2: 0.0271, 6: 0.0234 ms
    ncclComm_t comm_ = 0;
    cudaEvent_t t0_, t1_;
    int num_sms_;
    std::vector<cudaEvent_t> ev_pool_;
    struct Span { int kind; size_t e0, e1; };
    std::vector<Span> spans_;
    size_t ev_used_ = 0;
    double prof_ms_[LSTED_NUM_KERNEL_KINDS];
    long long prof_n_[LSTED_NUM_KERNEL_KINDS];

    size_t next_event() {
        if (ev_used_ == ev_pool_.size()) {
            cudaEvent_t e;
            CUDA_CHECK(cudaEventCreate(&e));
            ev_pool_.push_back(e);
        }
        return ev_used_++;
    }
    void before(int kind) {
        if (!profile_) return;
        Span s; s.kind = kind; s.e0 = next_event(); s.e1 = 0;
        CUDA_CHECK(cudaEventRecord(ev_pool_[s.e0], stream_));
        spans_.push_back(s);
    }
    void after() {
        CUDA_CHECK(cudaGetLastError());
        if (!profile_) return;
        Span& s = spans_.back();
        s.e1 = next_event();
        CUDA_CHECK(cudaEventRecord(ev_pool_[s.e1], stream_));
    }
    void profile_drain() {
        if (spans_.empty()) return;
        sync();
        for (size_t i = 0; i < spans_.size(); ++i) {
            float ms = 0;
            CUDA_CHECK(cudaEventElapsedTime(&ms, ev_pool_[spans_[i].e0], ev_pool_[spans_[i].e1]));
            prof_ms_[spans_[i].kind] += ms;
            prof_n_[spans_[i].kind] += 1;
        }
        spans_.clear();
        ev_used_ = 0;
    }
};

#define LSTED_BACKEND CudaBackend
#include "api_deconv.inl"

// ---------------------------------------------------------------------------
// Core entry points
// ---------------------------------------------------------------------------
extern "C" int lsted_version(void) { return 100; }
extern "C" const char* lsted_last_error(void) { return g_error.c_str(); }

extern "C" int lsted_device_count(int* count) {
    if (!count) return set_error(LSTED_ERR_ARG, "null pointer");
    cudaError_t err = cudaGetDeviceCount(count);
    if (err != cudaSuccess) {
        *count = 0;
        return set_error(LSTED_ERR_CUDA, std::string("cudaGetDeviceCount: ") + cudaGetErrorString(err));
    }
    return LSTED_OK;
}

extern "C" int lsted_nccl_unique_id(char* out) {
    if (!out) return set_error(LSTED_ERR_ARG, "null pointer");
    try {
        static_assert(sizeof(ncclUniqueId) == LSTED_NCCL_UNIQUE_ID_BYTES, "NCCL id size");
        ncclUniqueId id;
        NCCL_CHECK(nccl_api().GetUniqueId(&id));
        memcpy(out, id.internal, sizeof(id.internal));
        return LSTED_OK;
    } catch (const lsted::ApiError& e) { return set_error(e.code, e.msg); }
}

extern "C" int lsted_host_alloc(void** ptr, size_t bytes) {
    if (!ptr) return set_error(LSTED_ERR_ARG, "null pointer");
    cudaError_t err = cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocDefault);
    if (err != cudaSuccess)
        return set_error(LSTED_ERR_CUDA, std::string("cudaHostAlloc: ") + cudaGetErrorString(err));
    return LSTED_OK;
}
extern "C" int lsted_host_free(void* ptr) {
    if (ptr) cudaFreeHost(ptr);
    return LSTED_OK;
}

// ---------------------------------------------------------------------------
// PSF synthesis (fp64)
// ---------------------------------------------------------------------------
namespace {
void select_device(int device) {
    int count = 0;
    CUDA_CHECK(cudaGetDeviceCount(&count));
    if (device < 0 || device >= count) {
        lsted::ApiError e; e.code = LSTED_ERR_CUDA;
        e.msg = "CUDA device " + std::to_string(device) + " not available; there is no CPU fallback";
        throw e;
    }
    CUDA_CHECK(cudaSetDevice(device));
}

// psf_report is called hundreds of times in a row by tune_psf and the figure sweeps
// with kilobytes of data: per-call cudaMalloc/cudaFree and one D2H copy per array
// would dominate.  One workspace per device (device block + pinned host mirror,
// grown on demand), one H2D and one D2H per call.
struct PsfWorkspace {
    int device;
    void* dev; void* host; size_t cap;
    cudaStream_t stream;
    PsfWorkspace() : device(-1), dev(0), host(0), cap(0), stream(0) {}
    void reserve(size_t bytes) {
        if (bytes <= cap) return;
        if (dev) cudaFree(dev);
        if (host) cudaFreeHost(host);
        dev = host = 0; cap = 0;
        const size_t want = bytes + bytes / 2 + 4096;
        CUDA_CHECK(cudaMalloc(&dev, want));
        CUDA_CHECK(cudaHostAlloc(&host, want, cudaHostAllocDefault));
        cap = want;
    }
};
PsfWorkspace& psf_workspace(int device) {
    static thread_local std::map<int, PsfWorkspace> all;
    PsfWorkspace& w = all[device];
    if (w.device != device) {
        w.device = device;
        CUDA_CHECK(cudaStreamCreateWithFlags(&w.stream, cudaStreamNonBlocking));
    }
    return w;
}
inline size_t align256(size_t x) { return (x + 255) / 256 * 256; }
// dynamic shared memory above 48 KB needs the opt-in attribute (per device; cheap to repeat)
template <class F> void psf_raise_smem(F* kernel, size_t smem) {
    if (smem > 48 * 1024)
        CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
}
}  // namespace

extern "C" int lsted_psf_illumination(int device, int psf_type, int batch, int n, const double* taps,
                                      int radius, const double* excitation_brightness,
                                      const double* depletion_brightness, double* excitation,
                                      double* depletion, double* excitation_fraction,
                                      double* depletion_fraction, double* sted) {
    if (!taps || !excitation_brightness || !depletion_brightness || !excitation || !depletion ||
        !excitation_fraction || !depletion_fraction || !sted)
        return set_error(LSTED_ERR_ARG, "null pointer");
    if (batch < 1 || n < 1 || radius < 0 || (psf_type != 0 && psf_type != 1))
        return set_error(LSTED_ERR_ARG, "bad PSF arguments");
    if (n > lsted::kPsfMaxN || 2 * radius + 1 > lsted::kPsfMaxTaps)
        return set_error(LSTED_ERR_ARG, "PSF grid too large for the on-chip kernel");
    try {
        select_device(device);
        PsfWorkspace& w = psf_workspace(device);
        const size_t img = (size_t)n * n, ntap = 2 * radius + 1;
        // input block: taps | exc | dep ; output block: [batch][5][n][n]
        const size_t in_bytes = align256(sizeof(double) * (ntap + 2 * (size_t)batch));
        const size_t out_bytes = sizeof(double) * img * 5 * batch;
        w.reserve(in_bytes + out_bytes);
        double* h_in = (double*)w.host;
        memcpy(h_in, taps, sizeof(double) * ntap);
        memcpy(h_in + ntap, excitation_brightness, sizeof(double) * batch);
        memcpy(h_in + ntap + batch, depletion_brightness, sizeof(double) * batch);
        double* d_in = (double*)w.dev;
        double* d_out = (double*)((char*)w.dev + in_bytes);
        double* h_out = (double*)((char*)w.host + in_bytes);
        CUDA_CHECK(cudaMemcpyAsync(d_in, h_in, sizeof(double) * (ntap + 2 * (size_t)batch),
                                   cudaMemcpyHostToDevice, w.stream));
        lsted::PsfIlluminationArgs a;
        a.psf_type = psf_type; a.n = n; a.radius = radius;
        a.taps = d_in; a.exc_brightness = d_in + ntap; a.dep_brightness = d_in + ntap + batch;
        a.out = d_out;
        lsted::psf_illumination_kernel<<<batch, lsted::kPsfThreads, 0, w.stream>>>(a);
        CUDA_CHECK(cudaGetLastError());
        CUDA_CHECK(cudaMemcpyAsync(h_out, d_out, out_bytes, cudaMemcpyDeviceToHost, w.stream));
        CUDA_CHECK(cudaStreamSynchronize(w.stream));
        double* outs[5] = {excitation, depletion, excitation_fraction, depletion_fraction, sted};
        for (int b = 0; b < batch; ++b)
            for (int i = 0; i < 5; ++i)
                memcpy(outs[i] + img * b, h_out + img * (5 * (size_t)b + i), sizeof(double) * img);
        return LSTED_OK;
    } catch (const lsted::ApiError& e) { return set_error(e.code, e.msg); }
}

extern "C" int lsted_psf_report_batch(int device, int psf_type, int batch, const int* n, const int* radius,
                                      const double* taps, int tap_stride, const double* blur_sigma,
                                      const double* excitation_brightness,
                                      const double* depletion_brightness, double* scalars, double* psfs) {
    if (!n || !radius || !taps || !blur_sigma || !excitation_brightness || !depletion_brightness || !scalars)
        return set_error(LSTED_ERR_ARG, "null pointer");
    if (batch < 1 || tap_stride < 1 || (psf_type != 0 && psf_type != 1))
        return set_error(LSTED_ERR_ARG, "bad PSF arguments");
    int nmax = 0;
    for (int b = 0; b < batch; ++b) {
        if (n[b] < 1 || radius[b] < 0 || 2 * radius[b] + 1 > tap_stride)
            return set_error(LSTED_ERR_ARG, "bad PSF arguments");
        if (n[b] > lsted::kPsfMaxN || 2 * radius[b] + 1 > lsted::kPsfMaxTaps)
            return set_error(LSTED_ERR_ARG, "PSF grid too large for the on-chip kernel");
        nmax = n[b] > nmax ? n[b] : nmax;
    }
    try {
        select_device(device);
        PsfWorkspace& w = psf_workspace(device);
        // input block: taps[batch][tap_stride] | sigma | exc | dep | n | radius
        const size_t in_doubles = (size_t)batch * tap_stride + 3 * (size_t)batch;
        const size_t in_bytes = align256(sizeof(double) * in_doubles + 2 * sizeof(int) * batch);
        const size_t sc_bytes = align256(sizeof(double) * lsted::kPsfReportScalars * batch);
        const size_t plane = (size_t)nmax * nmax;
        const size_t psf_bytes = psfs ? sizeof(double) * plane * 7 * batch : 0;
        w.reserve(in_bytes + sc_bytes + psf_bytes);
        double* h_in = (double*)w.host;
        memcpy(h_in, taps, sizeof(double) * batch * tap_stride);
        double* h_par = h_in + (size_t)batch * tap_stride;
        memcpy(h_par, blur_sigma, sizeof(double) * batch);
        memcpy(h_par + batch, excitation_brightness, sizeof(double) * batch);
        memcpy(h_par + 2 * batch, depletion_brightness, sizeof(double) * batch);
        int* h_int = (int*)(h_in + in_doubles);
        memcpy(h_int, n, sizeof(int) * batch);
        memcpy(h_int + batch, radius, sizeof(int) * batch);
        double* d_in = (double*)w.dev;
        CUDA_CHECK(cudaMemcpyAsync(d_in, h_in, sizeof(double) * in_doubles + 2 * sizeof(int) * batch,
                                   cudaMemcpyHostToDevice, w.stream));
        lsted::PsfReportArgs a;
        a.psf_type = psf_type; a.nmax = nmax; a.tap_stride = tap_stride;
        a.taps = d_in;
        a.blur_sigma = d_in + (size_t)batch * tap_stride;
        a.exc_brightness = a.blur_sigma + batch; a.dep_brightness = a.blur_sigma + 2 * batch;
        a.n = (const int*)(d_in + in_doubles); a.radius = a.n + batch;
        a.scalars = (double*)((char*)w.dev + in_bytes);
        a.psfs = psfs ? (double*)((char*)w.dev + in_bytes + sc_bytes) : 0;
        const size_t smem = sizeof(double) * lsted::PsfReportSmem::doubles(nmax);
        psf_raise_smem(lsted::psf_report_kernel, smem);
        lsted::psf_report_kernel<<<batch, lsted::kPsfThreads, smem, w.stream>>>(a);
        CUDA_CHECK(cudaGetLastError());
        CUDA_CHECK(cudaMemcpyAsync((char*)w.host + in_bytes, (char*)w.dev + in_bytes, sc_bytes + psf_bytes,
                                   cudaMemcpyDeviceToHost, w.stream));
        CUDA_CHECK(cudaStreamSynchronize(w.stream));
        memcpy(scalars, (char*)w.host + in_bytes, sizeof(double) * lsted::kPsfReportScalars * batch);
        if (psfs) memcpy(psfs, (char*)w.host + in_bytes + sc_bytes, psf_bytes);
        return LSTED_OK;
    } catch (const lsted::ApiError& e) { return set_error(e.code, e.msg); }
}

extern "C" int lsted_gauss_fit(int device, int batch, int n, const double* rows, double* out) {
    if (!rows || !out) return set_error(LSTED_ERR_ARG, "null pointer");
    if (batch < 1 || n < 3 || n > lsted::kPsfMaxN) return set_error(LSTED_ERR_ARG, "bad fit arguments");
    try {
        select_device(device);
        PsfWorkspace& w = psf_workspace(device);
        const size_t in_bytes = align256(sizeof(double) * (size_t)n * batch);
        const size_t out_bytes = sizeof(double) * 5 * batch;
        w.reserve(in_bytes + out_bytes);
        memcpy(w.host, rows, sizeof(double) * (size_t)n * batch);
        CUDA_CHECK(cudaMemcpyAsync(w.dev, w.host, sizeof(double) * (size_t)n * batch, cudaMemcpyHostToDevice, w.stream));
        lsted::GaussFitArgs a;
        a.n = n; a.rows = (const double*)w.dev; a.out = (double*)((char*)w.dev + in_bytes);
        const size_t smem = sizeof(double) * lsted::PsfReportSmem::doubles(n);
        psf_raise_smem(lsted::gauss_fit_kernel, smem);
        lsted::gauss_fit_kernel<<<batch, lsted::kPsfThreads, smem, w.stream>>>(a);
        CUDA_CHECK(cudaGetLastError());
        CUDA_CHECK(cudaMemcpyAsync((char*)w.host + in_bytes, a.out, out_bytes, cudaMemcpyDeviceToHost, w.stream));
        CUDA_CHECK(cudaStreamSynchronize(w.stream));
        memcpy(out, (char*)w.host + in_bytes, out_bytes);
        return LSTED_OK;
    } catch (const lsted::ApiError& e) { return set_error(e.code, e.msg); }
}

extern "C" int lsted_psf_rotate(int device, int batch, int n0, int n1, const double* plane,
                               const double* xform, double clip_hi, double* out) {
    if (!plane || !xform || !out) return set_error(LSTED_ERR_ARG, "null pointer");
    if (batch < 1 || n0 < 1 || n1 < 1 || (long long)n0 * n1 > (1 << 24))
        return set_error(LSTED_ERR_ARG, "bad rotate arguments");
    try {
        select_device(device);
        PsfWorkspace& w = psf_workspace(device);
        const size_t img = (size_t)n0 * n1;
        // input block: plane | xform[batch][6]; scratch + output: 2 x [batch][n0][n1]
        const size_t in_doubles = img + 6 * (size_t)batch;
        const size_t in_bytes = align256(sizeof(double) * in_doubles);
        const size_t out_bytes = sizeof(double) * img * batch;
        w.reserve(in_bytes + 2 * out_bytes);
        double* h_in = (double*)w.host;
        memcpy(h_in, plane, sizeof(double) * img);
        memcpy(h_in + img, xform, sizeof(double) * 6 * batch);
        double* d_in = (double*)w.dev;
        double* d_out = (double*)((char*)w.dev + in_bytes);
        double* h_out = (double*)((char*)w.host + in_bytes);
        CUDA_CHECK(cudaMemcpyAsync(d_in, h_in, sizeof(double) * in_doubles, cudaMemcpyHostToDevice, w.stream));
        lsted::PsfRotateArgs a;
        a.n0 = n0; a.n1 = n1; a.plane = d_in; a.xform = d_in + img; a.clip_hi = clip_hi;
        a.out = d_out; a.coef = d_out + img * batch;
        lsted::psf_rotate_kernel<<<batch, lsted::kPsfThreads, 0, w.stream>>>(a);
        CUDA_CHECK(cudaGetLastError());
        CUDA_CHECK(cudaMemcpyAsync(h_out, d_out, out_bytes, cudaMemcpyDeviceToHost, w.stream));
        CUDA_CHECK(cudaStreamSynchronize(w.stream));
        memcpy(out, h_out, out_bytes);
        return LSTED_OK;
    } catch (const lsted::ApiError& e) { return set_error(e.code, e.msg); }
}

extern "C" int lsted_psf_rescan(int device, int batch, int n, const double* taps, int radius,
                                const double* sted_rows, const int* ratios, double* emission,
                                double* rescan, double* descan, double* wide) {
    if (!taps || !sted_rows || !ratios || !emission || !rescan || !descan)
        return set_error(LSTED_ERR_ARG, "null pointer");
    if (batch < 1 || n < 1 || radius < 0) return set_error(LSTED_ERR_ARG, "bad PSF arguments");
    if (n > lsted::kPsfMaxN || 2 * radius + 1 > lsted::kPsfMaxTaps)
        return set_error(LSTED_ERR_ARG, "PSF grid too large for the on-chip kernel");
    if (wide && batch != 1) return set_error(LSTED_ERR_ARG, "`wide` output needs batch == 1");
    for (int b = 0; b < batch; ++b)
        if (ratios[b] < 1 || (long long)ratios[b] * n > (1 << 24))
            return set_error(LSTED_ERR_ARG, "rescan ratio out of range");
    try {
        select_device(device);
        PsfWorkspace& w = psf_workspace(device);
        const size_t img = (size_t)n * n, ntap = 2 * radius + 1;
        const size_t W = wide ? (size_t)ratios[0] * n : 0;
        // input block: taps | rows[batch][n] | ratios[batch] ; output: [batch][3][n][n] | wide
        const size_t in_doubles = ntap + (size_t)n * batch;
        const size_t in_bytes = align256(sizeof(double) * in_doubles + sizeof(int) * batch);
        const size_t out_bytes = sizeof(double) * (img * 3 * batch + (size_t)n * W);
        w.reserve(in_bytes + out_bytes);
        double* h_in = (double*)w.host;
        memcpy(h_in, taps, sizeof(double) * ntap);
        memcpy(h_in + ntap, sted_rows, sizeof(double) * n * batch);
        memcpy(h_in + in_doubles, ratios, sizeof(int) * batch);
        double* d_in = (double*)w.dev;
        double* d_out = (double*)((char*)w.dev + in_bytes);
        double* h_out = (double*)((char*)w.host + in_bytes);
        CUDA_CHECK(cudaMemcpyAsync(d_in, h_in, sizeof(double) * in_doubles + sizeof(int) * batch,
                                   cudaMemcpyHostToDevice, w.stream));
        lsted::PsfRescanArgs a;
        a.n = n; a.radius = radius; a.taps = d_in;
        a.sted_rows = d_in + ntap; a.ratios = (const int*)(d_in + in_doubles);
        a.out = d_out; a.wide = wide ? d_out + img * 3 * batch : 0;
        lsted::psf_rescan_kernel<<<batch, lsted::kPsfThreads, 0, w.stream>>>(a);
        CUDA_CHECK(cudaGetLastError());
        CUDA_CHECK(cudaMemcpyAsync(h_out, d_out, out_bytes, cudaMemcpyDeviceToHost, w.stream));
        CUDA_CHECK(cudaStreamSynchronize(w.stream));
        double* outs[3] = {emission, rescan, descan};
        for (int b = 0; b < batch; ++b)
            for (int i = 0; i < 3; ++i)
                memcpy(outs[i] + img * b, h_out + img * (3 * (size_t)b + i), sizeof(double) * img);
        if (wide) memcpy(wide, h_out + img * 3 * batch, sizeof(double) * (size_t)n * W);
        return LSTED_OK;
    } catch (const lsted::ApiError& e) { return set_error(e.code, e.msg); }
}

// ---------------------------------------------------------------------------
// Figure-3 scan-position engine and the spline / Gaussian plane operators (fp64)
// ---------------------------------------------------------------------------
#include "scan_kernels.cuh"

namespace lsted {
// every scan kernel is an element functor (scan_kernels.cuh) under one grid-stride shell
template <class F> __global__ void __launch_bounds__(256) scan_for_each_kernel(const F f, size_t n) {
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n;
         e += (size_t)gridDim.x * blockDim.x)
        f(e);
}
}  // namespace lsted

namespace {
struct ScanCudaBackend {
    int device;
    cudaStream_t stream;
    cudaEvent_t ev0, ev1;
    int sm_count;
    std::vector<void*> live;
    explicit ScanCudaBackend(int dev) : device(dev), stream(0), ev0(0), ev1(0), sm_count(148) {
        select_device(dev);
        CUDA_CHECK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        CUDA_CHECK(cudaEventCreate(&ev0));
        CUDA_CHECK(cudaEventCreate(&ev1));
        cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev);
    }
    ~ScanCudaBackend() {
        cudaSetDevice(device);
        if (stream) cudaStreamSynchronize(stream);
        for (void* p : live) cudaFree(p);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (stream) cudaStreamDestroy(stream);
    }
    void activate() { CUDA_CHECK(cudaSetDevice(device)); }
    template <class T> T* alloc(size_t n) {
        void* p = 0;
        CUDA_CHECK(cudaMalloc(&p, (n ? n : 1) * sizeof(T)));
        live.push_back(p);
        return (T*)p;
    }
    void free(void* p) {
        for (size_t i = 0; i < live.size(); ++i)
            if (live[i] == p) { live[i] = live.back(); live.pop_back(); break; }
        CUDA_CHECK(cudaStreamSynchronize(stream));
        CUDA_CHECK(cudaFree(p));
    }
    void upload(void* d, const void* h, size_t bytes) {
        CUDA_CHECK(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, stream));
        CUDA_CHECK(cudaStreamSynchronize(stream));
    }
    void download(void* h, const void* d, size_t bytes) {
        CUDA_CHECK(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, stream));
        CUDA_CHECK(cudaStreamSynchronize(stream));
    }
    void copy(void* d, const void* s, size_t bytes) {
        CUDA_CHECK(cudaMemcpyAsync(d, s, bytes, cudaMemcpyDeviceToDevice, stream));
    }
    void zero(void* d, size_t bytes) { CUDA_CHECK(cudaMemsetAsync(d, 0, bytes, stream)); }
    void sync() { CUDA_CHECK(cudaStreamSynchronize(stream)); }
    void timer_start() { CUDA_CHECK(cudaEventRecord(ev0, stream)); }
    double timer_stop() {
        CUDA_CHECK(cudaEventRecord(ev1, stream));
        CUDA_CHECK(cudaEventSynchronize(ev1));
        float ms = 0.f;
        CUDA_CHECK(cudaEventElapsedTime(&ms, ev0, ev1));
        return ms;
    }
    template <class F> void for_each(size_t n, const F& f) {
        if (!n) return;
        const size_t want = (n + 255) / 256, cap = (size_t)sm_count * 32;
        lsted::scan_for_each_kernel<F><<<(unsigned)(want < cap ? want : cap), 256, 0, stream>>>(f, n);
        CUDA_CHECK(cudaGetLastError());
    }
};
}  // namespace

#define LSTED_SCAN_BACKEND ScanCudaBackend
#include "api_scan.inl"
