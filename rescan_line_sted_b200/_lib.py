"""ctypes binding of liblsted.so (the C ABI declared in include/lsted.h).

There is no CPU fallback: `get()` raises if the CUDA library has not been
built (`python -c "import __graft_entry__ as g; g.build()"`), and every call
raises RuntimeError with the library's message when CUDA fails.
"""
import ctypes
import os
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# LSTED_LIBRARY selects another build of the same C ABI (the debug build with in-kernel checks)
LIBRARY_PATH = os.environ.get('LSTED_LIBRARY') or os.path.join(_HERE, 'liblsted.so')

c_double_p = ctypes.POINTER(ctypes.c_double)
c_int_p = ctypes.POINTER(ctypes.c_int)
NUM_KERNEL_KINDS = 9
KERNEL_KINDS = ('row_fwd', 'row_inv_store', 'row_inv_sim', 'row_mid',
                'row_final', 'col_otf', 'col_h', 'col_ht', 'elementwise')

TRUE_OBJECT, NOISELESS, NOISY, ESTIMATE, NORMALIZATION = range(5)


class DeconvInfo(ctypes.Structure):
    _fields_ = [('K', ctypes.c_int), ('ny', ctypes.c_int), ('nx', ctypes.c_int),
                ('Ny', ctypes.c_int), ('Nx', ctypes.c_int),
                ('Ly', ctypes.c_int), ('Lx', ctypes.c_int),
                ('cols_per_cta', ctypes.c_int),
                ('row_pairs_per_cta', ctypes.c_int),
                ('precision', ctypes.c_int),
                ('iterations_done', ctypes.c_int),
                ('device', ctypes.c_int),
                ('row_smem_bytes', ctypes.c_size_t),
                ('col_smem_bytes', ctypes.c_size_t),
                ('device_bytes', ctypes.c_size_t),
                ('bytes_forward', ctypes.c_double),
                ('bytes_normalization', ctypes.c_double),
                ('bytes_iteration', ctypes.c_double),
                ('tiles_y', ctypes.c_int), ('tiles_x', ctypes.c_int),
                ('tile_out_y', ctypes.c_int), ('tile_out_x', ctypes.c_int),
                ('band_y0', ctypes.c_int), ('band_y1', ctypes.c_int),
                ('band_x0', ctypes.c_int), ('band_x1', ctypes.c_int)]


class ScanParams(ctypes.Structure):
    """lsted_scan_params_t of include/lsted.h"""
    _fields_ = [('imaging_type', ctypes.c_int),
                ('n_y', ctypes.c_int), ('n_x', ctypes.c_int), ('pad', ctypes.c_int),
                ('step', ctypes.c_int), ('exc_sep', ctypes.c_int),
                ('num_positions', ctypes.c_int),
                ('zoom_factor', ctypes.c_double),
                ('blur_radius', ctypes.c_int), ('exc_radius', ctypes.c_int),
                ('chunk_bytes', ctypes.c_size_t)]


# name -> (argtypes); all return int status except the two noted below
_DECONV_SIGNATURES = {
    'lsted_deconv_create': [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int,
                            c_double_p, ctypes.c_int, ctypes.c_int,
                            ctypes.c_int, ctypes.c_int, ctypes.c_int,
                            ctypes.c_int],
    'lsted_deconv_create_tiled': [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int,
                                  c_double_p, ctypes.c_int, ctypes.c_int,
                                  ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                  ctypes.c_int, ctypes.c_int],
    'lsted_deconv_destroy': [ctypes.c_void_p],
    'lsted_deconv_info': [ctypes.c_void_p, ctypes.POINTER(DeconvInfo)],
    'lsted_deconv_set_option': [ctypes.c_void_p, ctypes.c_char_p,
                                ctypes.c_double],
    'lsted_deconv_create_data': [ctypes.c_void_p, c_double_p, ctypes.c_double,
                                 ctypes.c_int, ctypes.c_uint64],
    'lsted_deconv_upload_object': [ctypes.c_void_p, c_double_p],
    'lsted_deconv_simulate': [ctypes.c_void_p, ctypes.c_double, ctypes.c_int,
                              ctypes.c_uint64],
    'lsted_deconv_shard': [ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                           ctypes.c_int, ctypes.c_char_p],
    'lsted_deconv_p2p_export': [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int],
    'lsted_deconv_p2p_attach': [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int],
    'lsted_deconv_nvls_create': [ctypes.c_void_p, ctypes.c_int, c_int_p],
    'lsted_deconv_nvls_import': [ctypes.c_void_p, ctypes.c_int, ctypes.c_int],
    'lsted_deconv_nvls_add_device': [ctypes.c_void_p],
    'lsted_deconv_nvls_bind': [ctypes.c_void_p],
    'lsted_deconv_iterate': [ctypes.c_void_p, ctypes.c_int],
    'lsted_deconv_get': [ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                         c_double_p],
    'lsted_deconv_set': [ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                         c_double_p],
    'lsted_deconv_ft_error': [ctypes.c_void_p, c_double_p, c_double_p, c_int_p],
    'lsted_deconv_H': [ctypes.c_void_p, c_double_p, c_double_p],
    'lsted_deconv_Ht': [ctypes.c_void_p, c_double_p, c_double_p, ctypes.c_int],
    # device-buffer twins: (..., pointer(s), dtype 32 | 64, [normalize,] cudaStream_t)
    'lsted_deconv_get_dev': [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                             ctypes.c_int, ctypes.c_void_p],
    'lsted_deconv_set_dev': [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                             ctypes.c_int, ctypes.c_void_p],
    'lsted_deconv_upload_object_dev': [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                       ctypes.c_void_p],
    'lsted_deconv_H_dev': [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                           ctypes.c_void_p],
    'lsted_deconv_Ht_dev': [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                            ctypes.c_int, ctypes.c_void_p],
    'lsted_deconv_sync': [ctypes.c_void_p],
    'lsted_deconv_timer_start': [ctypes.c_void_p],
    'lsted_deconv_timer_stop': [ctypes.c_void_p,
                                ctypes.POINTER(ctypes.c_float)],
    'lsted_deconv_profile': [ctypes.c_void_p, ctypes.c_int, c_double_p,
                             ctypes.POINTER(ctypes.c_longlong)],
}

_CORE_SIGNATURES = {
    'lsted_version': [],
    'lsted_device_count': [c_int_p],
    'lsted_host_alloc': [ctypes.POINTER(ctypes.c_void_p), ctypes.c_size_t],
    'lsted_host_free': [ctypes.c_void_p],
    'lsted_nccl_unique_id': [ctypes.c_char_p],
    'lsted_deconv_nvls_supported': [ctypes.c_int, c_int_p],
    'lsted_psf_illumination': [ctypes.c_int, ctypes.c_int, ctypes.c_int,
                               ctypes.c_int, c_double_p, ctypes.c_int,
                               c_double_p, c_double_p, c_double_p, c_double_p,
                               c_double_p, c_double_p, c_double_p],
    'lsted_psf_rescan': [ctypes.c_int, ctypes.c_int, ctypes.c_int, c_double_p,
                         ctypes.c_int, c_double_p, c_int_p, c_double_p,
                         c_double_p, c_double_p, c_double_p],
    'lsted_psf_report_batch': [ctypes.c_int, ctypes.c_int, ctypes.c_int, c_int_p,
                               c_int_p, c_double_p, ctypes.c_int, c_double_p,
                               c_double_p, c_double_p, c_double_p, c_double_p],
    'lsted_gauss_fit': [ctypes.c_int, ctypes.c_int, ctypes.c_int, c_double_p,
                        c_double_p],
    'lsted_psf_rotate': [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                         c_double_p, c_double_p, ctypes.c_double, c_double_p],
}

# figure-3 scan-position engine and the plane operators it is built from
_SCAN_SIGNATURES = {
    'lsted_scan_create': [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int,
                          ctypes.POINTER(ScanParams), c_int_p, c_double_p, c_double_p],
    'lsted_scan_destroy': [ctypes.c_void_p],
    'lsted_scan_excitation': [ctypes.c_void_p, c_double_p],
    'lsted_scan_run': [ctypes.c_void_p, c_double_p, c_double_p, c_int_p, ctypes.c_int,
                       c_double_p, c_double_p, c_double_p, c_double_p],
    'lsted_scan_frames': [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, c_double_p,
                          c_double_p, c_double_p],
    'lsted_img_spline': [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_double_p,
                         c_double_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                         c_double_p],
    'lsted_img_gauss': [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_double_p,
                        c_double_p, ctypes.c_int, c_double_p, ctypes.c_int, c_double_p],
}

# every symbol include/lsted.h declares (checked by tests/test_cabi_symbols.py)
EXPORTED_SYMBOLS = (['lsted_last_error'] + sorted(_CORE_SIGNATURES) +
                    sorted(_DECONV_SIGNATURES) + sorted(_SCAN_SIGNATURES))


class Library:
    """A loaded C-ABI library with typed entry points and error mapping."""

    def __init__(self, path, signatures):
        self.path = path
        self.cdll = ctypes.CDLL(path)
        self.cdll.lsted_last_error.restype = ctypes.c_char_p
        self.cdll.lsted_last_error.argtypes = []
        for name, argtypes in signatures.items():
            fn = getattr(self.cdll, name)
            fn.argtypes = argtypes
            fn.restype = ctypes.c_int

    def last_error(self):
        msg = self.cdll.lsted_last_error()
        return msg.decode('utf-8', 'replace') if msg else ''

    def call(self, name, *args):
        status = getattr(self.cdll, name)(*args)
        if status != 0:
            raise RuntimeError('%s failed (status %d): %s'
                               % (name, status, self.last_error()))


def as_f64(a):
    """C-contiguous float64 view/copy + its ctypes pointer."""
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, a.ctypes.data_as(c_double_p)


def is_tensor(x):
    """True for a torch.Tensor.  torch is never imported here: a caller that
    holds a tensor has imported it already."""
    torch = sys.modules.get('torch')
    return torch is not None and isinstance(x, torch.Tensor)


def check_tensor(t, shape, device, what):
    """Raise TypeError / ValueError unless `t` is a C-contiguous float32 or
    float64 CUDA tensor of `shape` (None: any extent) on CUDA device `device`.
    Everything but the device is checked first, so a CPU tensor shows its other
    faults too."""
    import torch
    if not isinstance(t, torch.Tensor):
        raise TypeError('%s must be a torch.Tensor, got %s' % (what, type(t).__name__))
    if t.dtype not in (torch.float32, torch.float64):
        raise TypeError('%s must be float32 or float64, got %s' % (what, t.dtype))
    if t.dim() != len(shape) or any(s is not None and s != n for s, n in zip(shape, t.shape)):
        want = '(%s)' % ', '.join('n' if s is None else str(s) for s in shape)
        raise ValueError('%s must have shape %s, got %s' % (what, want, tuple(t.shape)))
    if not t.is_contiguous():
        raise ValueError('%s must be C-contiguous' % what)
    if t.device.type != 'cuda':
        raise ValueError('%s must be a CUDA tensor, got one on %s' % (what, t.device))
    if t.device.index != device:
        raise ValueError('%s is on %s, the handle on cuda:%d' % (what, t.device, device))
    return t


_library = None


def get():
    """The product library.  Raises when liblsted.so is missing."""
    global _library
    if _library is None:
        if not os.path.isfile(LIBRARY_PATH):
            raise RuntimeError(
                'liblsted.so is not built (%s). Build it with '
                '`python -c "import __graft_entry__ as g; g.build()"` or '
                '`make -C rescan_line_sted_b200/csrc`. There is no CPU '
                'fallback.' % LIBRARY_PATH)
        sigs = dict(_CORE_SIGNATURES)
        sigs.update(_DECONV_SIGNATURES)
        sigs.update(_SCAN_SIGNATURES)
        _library = Library(LIBRARY_PATH, sigs)
    return _library


def bind_deconv_only(path):
    """Bind a library that exports just the Deconvolver subset (used by the
    CPU tests on the host replay of the kernel bodies)."""
    return Library(path, dict(_DECONV_SIGNATURES))


class DeconvHandle:
    """Thin RAII wrapper over lsted_deconv_* for one Deconvolver."""

    def __init__(self, lib, psfs, image_shape, precision=32, device=0,
                 tile_fft_len=0):
        self.lib = lib
        psfs = np.ascontiguousarray(psfs, dtype=np.float64)
        assert psfs.ndim == 3
        self.K, self.ny, self.nx = psfs.shape
        self.Ny, self.Nx = int(image_shape[0]), int(image_shape[1])
        self.precision = precision
        self.device = int(device)
        self._h = ctypes.c_void_p()
        lib.call('lsted_deconv_create_tiled', ctypes.byref(self._h), device,
                 psfs.ctypes.data_as(c_double_p), self.K, self.ny, self.nx,
                 self.Ny, self.Nx, precision, int(tile_fft_len))

    def close(self):
        if self._h:
            self.lib.cdll.lsted_deconv_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self):
        info = DeconvInfo()
        self.lib.call('lsted_deconv_info', self._h, ctypes.byref(info))
        return info

    def set_option(self, name, value):
        self.lib.call('lsted_deconv_set_option', self._h, name.encode(),
                      float(value))

    def create_data(self, obj, total_brightness, seed, reset_estimate=True):
        """Forward model + noise.  `reset_estimate` (default): the next iterate() starts
        from ones; the library itself leaves the estimate alone, like ref:496-512."""
        obj, p = as_f64(obj)
        assert obj.size == self.Ny * self.Nx
        rescale = total_brightness is not None
        if reset_estimate:
            self.set_option('reset_estimate', 1)
        self.lib.call('lsted_deconv_create_data', self._h, p,
                      float(total_brightness or 0.0), int(rescale),
                      ctypes.c_uint64(seed))

    def upload_object(self, obj):
        """Stage an object (async H2D when `obj` lives in pinned memory)."""
        assert obj.dtype == np.float64 and obj.flags.c_contiguous
        assert obj.size == self.Ny * self.Nx
        self.lib.call('lsted_deconv_upload_object', self._h,
                      obj.ctypes.data_as(c_double_p))

    def simulate(self, total_brightness, seed, reset_estimate=True):
        rescale = total_brightness is not None
        if reset_estimate:
            self.set_option('reset_estimate', 1)
        self.lib.call('lsted_deconv_simulate', self._h,
                      float(total_brightness or 0.0), int(rescale),
                      ctypes.c_uint64(seed))

    def shard(self, rank, world, k_offset, unique_id):
        """Orientation sharding: this handle holds PSFs k_offset..k_offset+K-1."""
        self.lib.call('lsted_deconv_shard', self._h, int(rank), int(world),
                      int(k_offset), unique_id)

    P2P_HANDLE_BYTES = 192

    def p2p_export(self):
        """CUDA-IPC handles of this rank's peer-memory reduction buffers (bytes)."""
        buf = ctypes.create_string_buffer(self.P2P_HANDLE_BYTES)
        self.lib.call('lsted_deconv_p2p_export', self._h, buf, self.P2P_HANDLE_BYTES)
        return buf.raw

    def p2p_attach(self, all_handles, world):
        """all_handles: the exports of ranks 0..world-1, concatenated."""
        assert len(all_handles) == world * self.P2P_HANDLE_BYTES
        self.lib.call('lsted_deconv_p2p_attach', self._h, all_handles, int(world))

    # NVLS (multicast) reduction of orientation shards: see include/lsted.h
    def nvls_create(self, world):
        fd = ctypes.c_int(-1)
        self.lib.call('lsted_deconv_nvls_create', self._h, int(world), ctypes.byref(fd))
        return fd.value

    def nvls_import(self, world, fd):
        self.lib.call('lsted_deconv_nvls_import', self._h, int(world), int(fd))

    def nvls_add_device(self):
        self.lib.call('lsted_deconv_nvls_add_device', self._h)

    def nvls_bind(self):
        self.lib.call('lsted_deconv_nvls_bind', self._h)

    def iterate(self, n=1):
        self.lib.call('lsted_deconv_iterate', self._h, int(n))

    def get(self, which, k=0):
        # large results land in recycled page-locked buffers (DMA at PCIe speed straight into
        # the array the caller gets; a fresh pageable array costs page faults + a staged copy)
        out = pooled_pinned_empty((1, self.Ny, self.Nx), lib=self.lib)
        self.lib.call('lsted_deconv_get', self._h, which, k,
                      out.ctypes.data_as(c_double_p))
        return out

    def get_into(self, which, k, out):
        self.lib.call('lsted_deconv_get', self._h, which, k,
                      out.ctypes.data_as(c_double_p))

    def set(self, which, k, arr):
        arr, p = as_f64(arr)
        assert arr.size == self.Ny * self.Nx
        self.lib.call('lsted_deconv_set', self._h, which, k, p)

    def ft_error(self, image=None):
        """log(1 + |fftshift(fft2(image - true_object))|), image = the estimate in HBM when
        None; (1, Ny, Nx) float64.  None only on a rank of a sharded tiled object asked for its
        own estimate (it holds a region of it): pass the gathered image instead."""
        out = pooled_pinned_empty((1, self.Ny, self.Nx), lib=self.lib)
        done = ctypes.c_int(0)
        if image is None:
            p = None
        else:
            image, p = as_f64(image)
            assert image.size == self.Ny * self.Nx
        self.lib.call('lsted_deconv_ft_error', self._h, p, out.ctypes.data_as(c_double_p),
                      ctypes.byref(done))
        return out if done.value else None

    def H(self, x):
        x, p = as_f64(x)
        assert x.size == self.Ny * self.Nx
        out = np.empty((self.K, self.Ny, self.Nx), dtype=np.float64)
        self.lib.call('lsted_deconv_H', self._h, p,
                      out.ctypes.data_as(c_double_p))
        return out

    def Ht(self, y, normalize=True):
        y, p = as_f64(y)
        assert y.size == self.K * self.Ny * self.Nx
        out = np.empty((1, self.Ny, self.Nx), dtype=np.float64)
        self.lib.call('lsted_deconv_Ht', self._h, p,
                      out.ctypes.data_as(c_double_p), int(bool(normalize)))
        return out

    # -- torch.Tensor forms (the _dev entry points): CUDA tensors on the handle's device,
    # float32 or float64, C-contiguous; ordered on the current torch stream, no host round trip
    def _stream(self):
        import torch
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _image(self, t, nimg, what):
        return check_tensor(t, (nimg, self.Ny, self.Nx), self.device, what)

    @staticmethod
    def _dtype_bits(t):
        return 32 if t.element_size() == 4 else 64

    def get_tensor(self, which, k=0, dtype=None, out=None):
        """Attribute `which` (PSF k) as a (1, Ny, Nx) tensor of `dtype` (float64 by
        default), or into `out`."""
        import torch
        if out is None:
            out = torch.empty((1, self.Ny, self.Nx), dtype=dtype or torch.float64,
                              device=torch.device('cuda', self.device))
        self._image(out, 1, 'out')
        self.lib.call('lsted_deconv_get_dev', self._h, which, k, out.data_ptr(),
                      self._dtype_bits(out), self._stream())
        return out

    def set_tensor(self, which, k, t):
        self._image(t, 1, 'the image')
        self.lib.call('lsted_deconv_set_dev', self._h, which, k, t.data_ptr(),
                      self._dtype_bits(t), self._stream())

    def upload_object_tensor(self, obj):
        """Stage an object from a tensor (then simulate(): the device form of create_data)."""
        self._image(obj, 1, 'the object')
        self.lib.call('lsted_deconv_upload_object_dev', self._h, obj.data_ptr(),
                      self._dtype_bits(obj), self._stream())

    def H_tensor(self, x):
        """(1, Ny, Nx) -> (K, Ny, Nx), dtype of x."""
        import torch
        self._image(x, 1, 'x')
        out = torch.empty((self.K, self.Ny, self.Nx), dtype=x.dtype, device=x.device)
        self.lib.call('lsted_deconv_H_dev', self._h, x.data_ptr(), out.data_ptr(),
                      self._dtype_bits(x), self._stream())
        return out

    def Ht_tensor(self, y, normalize=True):
        """(K, Ny, Nx) -> (1, Ny, Nx), dtype of y."""
        import torch
        self._image(y, self.K, 'y')
        out = torch.empty((1, self.Ny, self.Nx), dtype=y.dtype, device=y.device)
        self.lib.call('lsted_deconv_Ht_dev', self._h, y.data_ptr(), out.data_ptr(),
                      self._dtype_bits(y), int(bool(normalize)), self._stream())
        return out

    def sync(self):
        self.lib.call('lsted_deconv_sync', self._h)

    def timer_start(self):
        self.lib.call('lsted_deconv_timer_start', self._h)

    def timer_stop(self):
        ms = ctypes.c_float()
        self.lib.call('lsted_deconv_timer_stop', self._h, ctypes.byref(ms))
        return ms.value

    def profile(self, reset=False):
        ms = (ctypes.c_double * NUM_KERNEL_KINDS)()
        n = (ctypes.c_longlong * NUM_KERNEL_KINDS)()
        self.lib.call('lsted_deconv_profile', self._h, int(reset), ms, n)
        return {kind: (ms[i], n[i]) for i, kind in enumerate(KERNEL_KINDS)}


def pinned_empty(shape, dtype=np.float64):
    """numpy array over page-locked host memory (cudaHostAlloc); keep the
    returned array alive while transfers are in flight."""
    lib = get()
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    ptr = ctypes.c_void_p()
    lib.call('lsted_host_alloc', ctypes.byref(ptr), n)
    buf = (ctypes.c_char * n).from_address(ptr.value)
    arr = np.frombuffer(buf, dtype=dtype).reshape(shape)
    _pinned_keepalive[arr.ctypes.data] = ptr
    return arr


class _PinnedBlock:
    """Owner of one page-locked buffer handed out as a numpy array (through the array
    interface, so every view keeps it alive); when the last view dies the buffer goes back
    to the pool instead of to cudaFreeHost."""

    def __init__(self, lib, ptr, nbytes, shape, dtype):
        self._lib, self._ptr, self._nbytes = lib, ptr, nbytes
        self.__array_interface__ = {'shape': tuple(shape), 'typestr': np.dtype(dtype).str,
                                    'data': (ptr.value, False), 'version': 3}

    def __del__(self):
        try:
            _pinned_pool_release(self._lib, self._ptr, self._nbytes)
        except Exception:   # interpreter shutdown
            pass


_pinned_pool = {}                 # nbytes -> [free c_void_p, ...]
_pinned_pool_stats = {'outstanding': 0, 'pooled': 0}
PINNED_POOL_MIN_BYTES = 1 << 20   # smaller results: plain numpy arrays
PINNED_POOL_MAX_BYTES = 2 << 30   # page-locked bytes handed out + kept; beyond: plain arrays


def _pinned_pool_release(lib, ptr, nbytes):
    _pinned_pool_stats['outstanding'] -= nbytes
    if _pinned_pool_stats['pooled'] + nbytes <= PINNED_POOL_MAX_BYTES // 2:
        _pinned_pool.setdefault((id(lib), nbytes), []).append(ptr)
        _pinned_pool_stats['pooled'] += nbytes
    else:
        lib.cdll.lsted_host_free(ptr)


def pooled_pinned_empty(shape, dtype=np.float64, lib=None):
    """Fresh numpy array for a result read back from the GPU.  At least 1 MB: page-locked
    memory from a recycling pool (returned to it when the array is garbage-collected)."""
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    st = _pinned_pool_stats
    lib = lib or get()
    if (nbytes < PINNED_POOL_MIN_BYTES or st['outstanding'] + nbytes > PINNED_POOL_MAX_BYTES
            or not hasattr(lib.cdll, 'lsted_host_alloc')):   # (the CPU replay has none)
        return np.empty(shape, dtype=dtype)
    free = _pinned_pool.get((id(lib), nbytes))
    if free:
        ptr = free.pop()
        st['pooled'] -= nbytes
    else:
        ptr = ctypes.c_void_p()
        try:
            lib.call('lsted_host_alloc', ctypes.byref(ptr), nbytes)
        except RuntimeError:
            return np.empty(shape, dtype=dtype)
    st['outstanding'] += nbytes
    return np.asarray(_PinnedBlock(lib, ptr, nbytes, shape, dtype))


def pinned_free(arr):
    ptr = _pinned_keepalive.pop(arr.ctypes.data, None)
    if ptr is not None:
        get().cdll.lsted_host_free(ptr)


_pinned_keepalive = {}


NCCL_UNIQUE_ID_BYTES = 128


def nccl_unique_id(lib=None):
    """128-byte NCCL id (call on rank 0, broadcast to the other ranks).  A
    library without NCCL (the CPU replay used by the gloo tests) gets zeros."""
    lib = lib or get()
    buf = ctypes.create_string_buffer(NCCL_UNIQUE_ID_BYTES)
    if hasattr(lib.cdll, 'lsted_nccl_unique_id'):
        lib.call('lsted_nccl_unique_id', buf)
    return buf.raw
