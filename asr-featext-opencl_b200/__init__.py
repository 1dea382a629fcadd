"""ctypes binding of libafe_cuda.so (include/afe_cuda.h) — plumbing for tests and bench.py.

The product is the C-ABI library (hand-written sm_100a kernels) and the C++ mirror classes in host/; this module only
forwards to the C ABI, keeping the reference's verb set (ParamBase: set_window / set_input / flush / apply /
get_output_data_width / get_output_data, parambase.h:23-32). There is no CPU fallback: if the library is missing or no
CUDA device is usable, construction raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libafe_cuda.so")
ABI_VERSION = 3

NORM_NONE, NORM_CMN, NORM_CVN, NORM_MINMAX = 0, 1, 2, 3
DYN_NONE, DYN_DELTA, DYN_ACC = 0, 1, 2
STATS_REFERENCE_BLOCK, STATS_UTTERANCE, STATS_CORPUS = 0, 1, 2
BATCH_Q1_EXACT, BATCH_NO_TMA, BATCH_UNFUSED_NORM, BATCH_NO_CLUSTER = 1, 2, 8, 32
OPT_FIX_FLUSH_STATICS, OPT_STAGED_KERNELS = 1, 2

# every symbol include/afe_cuda.h declares (tests/test_abi.py checks the header against this list and the .so)
SYMBOLS = """
afe_last_error afe_abi_version afe_build_flags afe_device_count afe_estimated_window_count afe_output_width afe_fft_size
afe_make_window afe_build_filters afe_build_dct
afe_mfcc_create afe_mfcc_destroy afe_mfcc_set_window afe_mfcc_set_alpha afe_mfcc_input_buffer_size
afe_mfcc_estimated_window_count afe_mfcc_output_width afe_mfcc_set_input afe_mfcc_flush afe_mfcc_apply
afe_mfcc_get_output afe_mfcc_reset afe_mfcc_set_option afe_mfcc_set_preemphasis afe_mfcc_uses_fused_kernel
afe_mfcc_kernel_launches
afe_segmenter_create afe_segmenter_destroy afe_segmenter_set_window afe_segmenter_set_preemphasis afe_segmenter_set_input
afe_segmenter_flush
afe_segmenter_remaining_samples afe_segmenter_samples afe_segmenter_is_flushed afe_segmenter_was_flushed
afe_delta_create afe_delta_destroy afe_delta_apply afe_delta_output
afe_normalizer_create afe_normalizer_destroy afe_normalizer_normalize afe_normalizer_stats_len afe_normalizer_reset
afe_normalizer_accumulate afe_normalizer_allreduce afe_normalizer_finalize afe_normalizer_apply afe_normalizer_get_stats
afe_normalizer_set_stats
afe_device_malloc afe_device_free afe_memcpy_h2d afe_memcpy_d2h
afe_batch_create afe_batch_destroy afe_batch_set_window afe_batch_set_alpha afe_batch_set_preemphasis afe_batch_set_options
afe_batch_set_stream
afe_batch_plan afe_batch_plan_segments afe_batch_frame_offsets afe_batch_num_tiles afe_batch_kernel_launches afe_batch_kernel_name afe_batch_run_device
afe_batch_extract_device afe_batch_corpus_stats afe_batch_normalizer afe_batch_set_corpus_stats
afe_batch_normalize_device afe_batch_synchronize afe_batch_run_host
afe_cmvn_finalize_host afe_shard_utterances afe_shard_stream afe_nccl_get_unique_id afe_nccl_comm_init afe_nccl_comm_destroy
""".split()


class AfeParams(C.Structure):
    _fields_ = [("input_buffer_size", C.c_int), ("window_size", C.c_int), ("shift", C.c_int), ("num_banks", C.c_int),
                ("sample_rate", C.c_float), ("low_freq", C.c_float), ("high_freq", C.c_float),
                ("ceps_len", C.c_int), ("want_c0", C.c_int), ("lift_coef", C.c_float),
                ("norm", C.c_int), ("dyn", C.c_int), ("delta_l1", C.c_int), ("delta_l2", C.c_int),
                ("norm_after_dyn", C.c_int)]


def make_params(input_buffer_size=10_000_000, window_size=400, shift=160, num_banks=23, sample_rate=16000.0,
                low_freq=64.0, high_freq=8000.0, ceps_len=12, want_c0=1, lift_coef=22.0, norm=0, dyn=0,
                delta_l1=3, delta_l2=3, norm_after_dyn=1, alpha=None):
    """Defaults follow the reference driver's SConfig (ASR_OCL.cpp:560) except norm/dyn = none. `alpha` is accepted
    and ignored so that the oracle's parameter dicts can be splatted in."""
    return AfeParams(int(input_buffer_size), int(window_size), int(shift), int(num_banks), float(sample_rate),
                     float(low_freq), float(high_freq), int(ceps_len), int(want_c0), float(lift_coef), int(norm),
                     int(dyn), int(delta_l1), int(delta_l2), int(norm_after_dyn))


_lib = None


def lib():
    """Load libafe_cuda.so (fails loudly when it was not built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        vp, ip, fp = C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_float)
        i16p, i64p, dp = C.POINTER(C.c_short), C.POINTER(C.c_longlong), C.POINTER(C.c_double)
        pp = C.POINTER(AfeParams)
        sig = {
            "afe_last_error": (C.c_char_p, []),
            "afe_abi_version": (C.c_int, []),
            "afe_build_flags": (C.c_int, []),
            "afe_device_count": (C.c_int, []),
            "afe_estimated_window_count": (C.c_int, [C.c_int] * 3),
            "afe_output_width": (C.c_int, [pp]),
            "afe_fft_size": (C.c_int, [C.c_int]),
            "afe_make_window": (None, [fp, C.c_int]),
            "afe_build_filters": (C.c_int, [pp, C.c_float, ip, fp]),
            "afe_build_dct": (C.c_int, [pp, fp]),
            "afe_mfcc_create": (C.c_int, [pp, C.c_int, C.POINTER(vp)]),
            "afe_mfcc_destroy": (None, [vp]),
            "afe_mfcc_set_window": (C.c_int, [vp, fp]),
            "afe_mfcc_set_alpha": (C.c_int, [vp, C.c_float]),
            "afe_mfcc_input_buffer_size": (C.c_int, [vp]),
            "afe_mfcc_estimated_window_count": (C.c_int, [vp, C.c_int]),
            "afe_mfcc_output_width": (C.c_int, [vp]),
            "afe_mfcc_set_input": (C.c_int, [vp, i16p, C.c_int, ip]),
            "afe_mfcc_flush": (C.c_int, [vp, ip]),
            "afe_mfcc_apply": (C.c_int, [vp]),
            "afe_mfcc_get_output": (C.c_int, [vp, fp, C.c_int]),
            "afe_mfcc_reset": (C.c_int, [vp]),
            "afe_mfcc_set_option": (C.c_int, [vp, C.c_int, C.c_int]),
            "afe_mfcc_set_preemphasis": (C.c_int, [vp, C.c_float]),
            "afe_mfcc_uses_fused_kernel": (C.c_int, [vp]),
            "afe_mfcc_kernel_launches": (C.c_int, [vp]),
            "afe_segmenter_set_preemphasis": (C.c_int, [vp, C.c_float]),
            "afe_segmenter_create": (C.c_int, [C.c_int] * 5 + [C.POINTER(vp)]),
            "afe_segmenter_destroy": (None, [vp]),
            "afe_segmenter_set_window": (C.c_int, [vp, fp]),
            "afe_segmenter_set_input": (C.c_int, [vp, i16p, vp, C.c_int, ip, ip]),
            "afe_segmenter_flush": (C.c_int, [vp, vp, ip, ip]),
            "afe_segmenter_remaining_samples": (C.c_int, [vp]),
            "afe_segmenter_samples": (C.c_int, [vp]),
            "afe_segmenter_is_flushed": (C.c_int, [vp]),
            "afe_segmenter_was_flushed": (C.c_int, [vp]),
            "afe_delta_create": (C.c_int, [C.c_int] * 4 + [C.POINTER(vp)]),
            "afe_delta_destroy": (None, [vp]),
            "afe_delta_apply": (C.c_int, [vp, vp, C.c_int]),
            "afe_delta_output": (vp, [vp]),
            "afe_normalizer_create": (C.c_int, [C.c_int] * 3 + [C.POINTER(vp)]),
            "afe_normalizer_destroy": (None, [vp]),
            "afe_normalizer_normalize": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int]),
            "afe_normalizer_stats_len": (C.c_int, [vp]),
            "afe_normalizer_reset": (C.c_int, [vp]),
            "afe_normalizer_accumulate": (C.c_int, [vp, vp, C.c_int, C.c_int]),
            "afe_normalizer_allreduce": (C.c_int, [vp, vp]),
            "afe_normalizer_finalize": (C.c_int, [vp]),
            "afe_normalizer_apply": (C.c_int, [vp, vp, C.c_int, C.c_int]),
            "afe_normalizer_get_stats": (C.c_int, [vp, dp]),
            "afe_normalizer_set_stats": (C.c_int, [vp, dp]),
            "afe_device_malloc": (C.c_int, [C.c_int, C.c_size_t, C.POINTER(vp)]),
            "afe_device_free": (C.c_int, [C.c_int, vp]),
            "afe_memcpy_h2d": (C.c_int, [C.c_int, vp, vp, C.c_size_t]),
            "afe_memcpy_d2h": (C.c_int, [C.c_int, vp, vp, C.c_size_t]),
            "afe_batch_create": (C.c_int, [pp, C.c_int, C.POINTER(vp)]),
            "afe_batch_destroy": (None, [vp]),
            "afe_batch_set_window": (C.c_int, [vp, fp]),
            "afe_batch_set_alpha": (C.c_int, [vp, C.c_float]),
            "afe_batch_set_preemphasis": (C.c_int, [vp, C.c_float]),
            "afe_batch_set_options": (C.c_int, [vp, C.c_int, C.c_int]),
            "afe_batch_set_stream": (C.c_int, [vp, vp]),
            "afe_batch_plan": (C.c_int, [vp, i64p, i64p, C.c_int, i64p]),
            "afe_batch_plan_segments": (C.c_int, [vp, i64p, i64p, ip, ip, C.c_int, i64p]),
            "afe_shard_stream": (C.c_int, [C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int, i64p, i64p, i64p, ip, ip]),
            "afe_batch_frame_offsets": (C.c_int, [vp, i64p]),
            "afe_batch_num_tiles": (C.c_int, [vp]),
            "afe_batch_kernel_launches": (C.c_int, [vp]),
            "afe_batch_kernel_name": (C.c_char_p, [vp]),
            "afe_batch_run_device": (C.c_int, [vp, vp, vp]),
            "afe_batch_extract_device": (C.c_int, [vp, vp, vp]),
            "afe_batch_corpus_stats": (C.c_int, [vp, C.POINTER(vp), ip]),
            "afe_batch_normalizer": (vp, [vp]),
            "afe_batch_set_corpus_stats": (C.c_int, [vp, dp, C.c_int]),
            "afe_batch_normalize_device": (C.c_int, [vp, vp]),
            "afe_batch_synchronize": (C.c_int, [vp]),
            "afe_batch_run_host": (C.c_int, [vp, vp, vp]),
            "afe_cmvn_finalize_host": (C.c_int, [C.c_int, C.c_int, dp, fp, fp]),
            "afe_shard_utterances": (C.c_int, [i64p, C.c_int, C.c_int, ip]),
            "afe_nccl_get_unique_id": (C.c_int, [vp]),
            "afe_nccl_comm_init": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]),
            "afe_nccl_comm_destroy": (C.c_int, [vp]),
        }
        for name, (res, args) in sig.items():
            f = getattr(L, name)
            f.restype, f.argtypes = res, args
        _lib = L
    return _lib


class AfeError(RuntimeError):
    pass


def _check(rc):
    if rc != 0:
        raise AfeError((lib().afe_last_error() or b"unknown error").decode())


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def make_window(window_size):
    """The reference driver's window (ASR_OCL.cpp:149-152)."""
    w = np.empty(window_size, np.float32)
    lib().afe_make_window(_fp(w), window_size)
    return w


def estimated_window_count(samples, window_size, shift):
    return lib().afe_estimated_window_count(int(samples), int(window_size), int(shift))


def build_filters(params, alpha=1.0):
    n2 = lib().afe_fft_size(params.window_size)
    edges = np.zeros(params.num_banks + 2, np.int32)
    filt = np.zeros(2 * n2, np.float32)
    _check(lib().afe_build_filters(C.byref(params), float(alpha), edges.ctypes.data_as(C.POINTER(C.c_int)), _fp(filt)))
    return edges, filt.reshape(2, n2)


def build_dct(params):
    dl = params.ceps_len + (1 if params.want_c0 else 0)
    m = np.zeros((params.num_banks, dl), np.float32)
    _check(lib().afe_build_dct(C.byref(params), _fp(m)))
    return m


def shard_utterances(sample_lengths, n_ranks):
    off = np.ascontiguousarray(sample_lengths, np.int64)
    starts = np.zeros(n_ranks + 1, np.int32)
    _check(lib().afe_shard_utterances(off.ctypes.data_as(C.POINTER(C.c_longlong)), len(off), n_ranks,
                                      starts.ctypes.data_as(C.POINTER(C.c_int))))
    return starts


def shard_stream(total_samples, window_size, shift, delta_frames, n_ranks):
    """-> dict of arrays: sample_begin, sample_count, first, count, local_first (afe_shard_stream)."""
    sb, sc, fi = (np.zeros(n_ranks, np.int64) for _ in range(3))
    cnt, lf = np.zeros(n_ranks, np.int32), np.zeros(n_ranks, np.int32)
    i64p, ip = C.POINTER(C.c_longlong), C.POINTER(C.c_int)
    _check(lib().afe_shard_stream(int(total_samples), int(window_size), int(shift), int(delta_frames), int(n_ranks),
                                  sb.ctypes.data_as(i64p), sc.ctypes.data_as(i64p), fi.ctypes.data_as(i64p),
                                  cnt.ctypes.data_as(ip), lf.ctypes.data_as(ip)))
    return dict(sample_begin=sb, sample_count=sc, first=fi, count=cnt, local_first=lf)


def cmvn_finalize_host(norm, width, stats):
    stats = np.ascontiguousarray(stats, np.float64)
    mean = np.zeros(width, np.float32)
    scale = np.zeros(width, np.float32)
    _check(lib().afe_cmvn_finalize_host(int(norm), int(width), stats.ctypes.data_as(C.POINTER(C.c_double)), _fp(mean), _fp(scale)))
    return mean, scale


class MfccCuda:
    """Accelerator variant of the Mfcc stage object: same 15 constructor arguments as MfccOpenCL plus the CUDA device
    (mfccopencl.h:45-60), same verbs as ParamBase."""

    def __init__(self, params, cuda_device=0):
        self._h = C.c_void_p()
        self.params = params
        _check(lib().afe_mfcc_create(C.byref(params), cuda_device, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            lib().afe_mfcc_destroy(self._h)
            self._h = None

    __del__ = close

    def set_window(self, window):
        w = np.ascontiguousarray(window, np.float32)
        assert len(w) == self.params.window_size
        _check(lib().afe_mfcc_set_window(self._h, _fp(w)))

    def set_alpha(self, alpha):
        _check(lib().afe_mfcc_set_alpha(self._h, float(alpha)))

    def set_preemphasis(self, coefficient):
        _check(lib().afe_mfcc_set_preemphasis(self._h, float(coefficient)))

    @property
    def uses_fused_kernel(self):
        return bool(lib().afe_mfcc_uses_fused_kernel(self._h))

    @property
    def kernel_launches(self):
        return lib().afe_mfcc_kernel_launches(self._h)

    def get_input_buffer_size(self):
        return lib().afe_mfcc_input_buffer_size(self._h)

    def estimated_window_count(self, samples):
        return lib().afe_mfcc_estimated_window_count(self._h, int(samples))

    def get_output_data_width(self):
        return lib().afe_mfcc_output_width(self._h)

    def set_input(self, data):
        d = np.ascontiguousarray(data, np.int16)
        n = C.c_int(0)
        _check(lib().afe_mfcc_set_input(self._h, d.ctypes.data_as(C.POINTER(C.c_short)), len(d), C.byref(n)))
        return n.value

    def flush(self):
        n = C.c_int(0)
        _check(lib().afe_mfcc_flush(self._h, C.byref(n)))
        return n.value

    def apply(self):
        _check(lib().afe_mfcc_apply(self._h))

    def get_output_data(self, window_count):
        out = np.zeros((window_count, self.get_output_data_width()), np.float32)
        _check(lib().afe_mfcc_get_output(self._h, _fp(out), int(window_count)))
        return out

    def reset(self):
        _check(lib().afe_mfcc_reset(self._h))

    def set_option(self, option, value):
        _check(lib().afe_mfcc_set_option(self._h, int(option), int(value)))


def extract_stream(params, pcm, alpha=1.0, window=None, cuda_device=0, fix_flush_statics=False, preemphasis=0.0,
                   staged=False):
    """The reference driver's block loop (ASR_OCL.cpp:227-301) over one utterance, through the streaming object."""
    m = MfccCuda(params, cuda_device)
    try:
        if staged:
            m.set_option(OPT_STAGED_KERNELS, 1)
        m.set_window(make_window(params.window_size) if window is None else window)
        m.set_alpha(alpha)
        if preemphasis:
            m.set_preemphasis(preemphasis)
        if fix_flush_statics:
            m.set_option(OPT_FIX_FLUSH_STATICS, 1)
        limit = m.get_input_buffer_size()
        rows, pos = [], 0
        while pos < len(pcm):
            n = min(limit, len(pcm) - pos)
            wc = m.set_input(pcm[pos:pos + n])
            m.apply()
            if wc > 0:
                rows.append(m.get_output_data(wc))
            pos += n
        wc = m.flush()
        if wc > 0:
            m.apply()
            rows.append(m.get_output_data(wc))
        return np.concatenate(rows) if rows else np.zeros((0, m.get_output_data_width()), np.float32)
    finally:
        m.close()


class DeviceBuffer:
    def __init__(self, nbytes, cuda_device=0):
        self.dev, self.nbytes = cuda_device, int(nbytes)
        self.ptr = C.c_void_p()
        _check(lib().afe_device_malloc(cuda_device, self.nbytes, C.byref(self.ptr)))

    def upload(self, arr):
        arr = np.ascontiguousarray(arr)
        assert arr.nbytes <= self.nbytes
        _check(lib().afe_memcpy_h2d(self.dev, self.ptr, arr.ctypes.data_as(C.c_void_p), arr.nbytes))

    def download(self, shape, dtype):
        out = np.zeros(shape, dtype)
        assert out.nbytes <= self.nbytes
        _check(lib().afe_memcpy_d2h(self.dev, out.ctypes.data_as(C.c_void_p), self.ptr, out.nbytes))
        return out

    def free(self):
        if self.ptr:
            lib().afe_device_free(self.dev, self.ptr)
            self.ptr = None

    __del__ = free


class SegmenterCuda:
    """SegmenterOpenCL counterpart (segmenteropencl.h:27-42); frames land in a device buffer."""

    def __init__(self, window_size, shift, window_limit, deltasize, cuda_device=0):
        self._h = C.c_void_p()
        self.W, self.S, self.limit = window_size, shift, window_limit
        self.N2 = lib().afe_fft_size(window_size)
        _check(lib().afe_segmenter_create(window_size, shift, window_limit, deltasize, cuda_device, C.byref(self._h)))
        self.out = DeviceBuffer(4 * self.N2 * max(window_limit, 1), cuda_device)

    def close(self):
        if getattr(self, "_h", None):
            lib().afe_segmenter_destroy(self._h)
            self._h = None
            self.out.free()

    __del__ = close

    def set_window(self, w):
        w = np.ascontiguousarray(w, np.float32)
        _check(lib().afe_segmenter_set_window(self._h, _fp(w)))

    def set_input(self, data):
        d = np.ascontiguousarray(data, np.int16)
        wc, nd = C.c_int(0), C.c_int(0)
        _check(lib().afe_segmenter_set_input(self._h, d.ctypes.data_as(C.POINTER(C.c_short)), self.out.ptr, len(d),
                                             C.byref(wc), C.byref(nd)))
        return wc.value, nd.value

    def flush(self):
        wc, nd = C.c_int(0), C.c_int(0)
        _check(lib().afe_segmenter_flush(self._h, self.out.ptr, C.byref(wc), C.byref(nd)))
        return wc.value, nd.value

    def frames(self, n):
        return self.out.download((n, self.N2), np.float32)

    def get_remaining_samples(self):
        return lib().afe_segmenter_remaining_samples(self._h)

    def get_samples(self):
        return lib().afe_segmenter_samples(self._h)

    def is_flushed(self):
        return bool(lib().afe_segmenter_is_flushed(self._h))

    def was_flushed(self):
        return bool(lib().afe_segmenter_was_flushed(self._h))


class DeltaCuda:
    """DeltaOpenCL counterpart (deltaopencl.h:17-22)."""

    def __init__(self, dim, window_limit, delta_size, cuda_device=0):
        self._h = C.c_void_p()
        self.dim, self.limit, self.L, self.dev = dim, window_limit, delta_size, cuda_device
        _check(lib().afe_delta_create(dim, window_limit, delta_size, cuda_device, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            lib().afe_delta_destroy(self._h)
            self._h = None

    __del__ = close

    def apply(self, data, window_count):
        """data: host [window_count + 2L, dim] (uploaded here for convenience) -> host [window_count, dim]"""
        data = np.ascontiguousarray(data, np.float32)
        buf = DeviceBuffer(data.nbytes, self.dev)
        buf.upload(data)
        _check(lib().afe_delta_apply(self._h, buf.ptr, int(window_count)))
        out = np.zeros((window_count, self.dim), np.float32)
        _check(lib().afe_memcpy_d2h(self.dev, out.ctypes.data_as(C.c_void_p), lib().afe_delta_output(self._h), out.nbytes))
        buf.free()
        return out


class NormalizerCuda:
    """NormalizerOpenCL counterpart (normalizeropencl.h:25-28); statistics in double like NormalizerCPU."""

    def __init__(self, norm_type, dim, cuda_device=0):
        self._h = C.c_void_p()
        self.dim, self.dev = dim, cuda_device
        _check(lib().afe_normalizer_create(int(norm_type), dim, cuda_device, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            lib().afe_normalizer_destroy(self._h)
            self._h = None

    __del__ = close

    def normalize(self, data, use_last_stats=False):
        data = np.ascontiguousarray(data, np.float32)
        buf = DeviceBuffer(max(data.nbytes, 4), self.dev)
        buf.upload(data)
        _check(lib().afe_normalizer_normalize(self._h, buf.ptr, 0, data.shape[0], int(use_last_stats)))
        out = buf.download(data.shape, np.float32)
        buf.free()
        return out

    # ---- corpus-level verbs on the running record (sum | sumsq | count | min | max): reset -> accumulate* -> allreduce ->
    #      finalize -> apply*. Host arrays are uploaded here for convenience; the C ABI takes device pointers.
    @property
    def stats_len(self):
        return lib().afe_normalizer_stats_len(self._h)

    def reset(self):
        _check(lib().afe_normalizer_reset(self._h))

    def accumulate(self, data):
        data = np.ascontiguousarray(data, np.float32)
        buf = DeviceBuffer(max(data.nbytes, 4), self.dev)
        buf.upload(data)
        _check(lib().afe_normalizer_accumulate(self._h, buf.ptr, 0, data.shape[0]))
        self.get_stats()          # drains the stream before the buffer goes away
        buf.free()

    def allreduce(self, nccl_comm):
        _check(lib().afe_normalizer_allreduce(self._h, C.c_void_p(nccl_comm)))

    def finalize(self):
        _check(lib().afe_normalizer_finalize(self._h))

    def apply(self, data):
        data = np.ascontiguousarray(data, np.float32)
        buf = DeviceBuffer(max(data.nbytes, 4), self.dev)
        buf.upload(data)
        _check(lib().afe_normalizer_apply(self._h, buf.ptr, 0, data.shape[0]))
        out = buf.download(data.shape, np.float32)
        buf.free()
        return out

    def get_stats(self):
        s = np.zeros(self.stats_len, np.float64)
        _check(lib().afe_normalizer_get_stats(self._h, s.ctypes.data_as(C.POINTER(C.c_double))))
        return s

    def set_stats(self, stats):
        s = np.ascontiguousarray(stats, np.float64)
        assert len(s) == self.stats_len
        _check(lib().afe_normalizer_set_stats(self._h, s.ctypes.data_as(C.POINTER(C.c_double))))


class BatchMfcc:
    """Fused batch extractor (afe_batch_*): whole utterances, one fused kernel + a light normalise pass."""

    def __init__(self, params, cuda_device=0, stats_scope=STATS_REFERENCE_BLOCK, flags=0, window=None, alpha=1.0,
                 preemphasis=0.0):
        self._h = C.c_void_p()
        self.params, self.dev = params, cuda_device
        _check(lib().afe_batch_create(C.byref(params), cuda_device, C.byref(self._h)))
        self.width = lib().afe_output_width(C.byref(params))
        _check(lib().afe_batch_set_options(self._h, stats_scope, flags))
        w = make_window(params.window_size) if window is None else np.ascontiguousarray(window, np.float32)
        _check(lib().afe_batch_set_window(self._h, _fp(w)))
        _check(lib().afe_batch_set_alpha(self._h, float(alpha)))
        if preemphasis:
            _check(lib().afe_batch_set_preemphasis(self._h, float(preemphasis)))
        self.frame_offsets = None

    def close(self):
        if getattr(self, "_h", None):
            lib().afe_batch_destroy(self._h)
            self._h = None

    __del__ = close

    def set_alpha(self, alpha):
        _check(lib().afe_batch_set_alpha(self._h, float(alpha)))

    def set_options(self, stats_scope, flags):
        _check(lib().afe_batch_set_options(self._h, stats_scope, flags))

    def set_stream(self, cuda_stream):
        _check(lib().afe_batch_set_stream(self._h, C.c_void_p(cuda_stream)))

    def plan(self, sample_offsets, sample_lengths):
        off = np.ascontiguousarray(sample_offsets, np.int64)
        ln = np.ascontiguousarray(sample_lengths, np.int64)
        assert len(off) == len(ln)
        total = C.c_longlong(0)
        i64p = C.POINTER(C.c_longlong)
        _check(lib().afe_batch_plan(self._h, off.ctypes.data_as(i64p), ln.ctypes.data_as(i64p), len(off), C.byref(total)))
        fo = np.zeros(len(off) + 1, np.int64)
        lib().afe_batch_frame_offsets(self._h, fo.ctypes.data_as(i64p))
        self.frame_offsets, self.sample_offsets, self.sample_lengths = fo, off, ln
        self.pcm_extent = int((off + ln).max()) if len(off) else 0
        return int(total.value)

    def plan_segments(self, sample_offsets, sample_lengths, first_frame, n_frames):
        """Segments of longer streams: entry u outputs the rows of its frames [first_frame[u], first_frame[u] + n_frames[u])."""
        off = np.ascontiguousarray(sample_offsets, np.int64)
        ln = np.ascontiguousarray(sample_lengths, np.int64)
        ff = np.ascontiguousarray(first_frame, np.int32)
        nf = np.ascontiguousarray(n_frames, np.int32)
        total = C.c_longlong(0)
        i64p, ip = C.POINTER(C.c_longlong), C.POINTER(C.c_int)
        _check(lib().afe_batch_plan_segments(self._h, off.ctypes.data_as(i64p), ln.ctypes.data_as(i64p), ff.ctypes.data_as(ip),
                                             nf.ctypes.data_as(ip), len(off), C.byref(total)))
        fo = np.zeros(len(off) + 1, np.int64)
        lib().afe_batch_frame_offsets(self._h, fo.ctypes.data_as(i64p))
        self.frame_offsets, self.sample_offsets, self.sample_lengths = fo, off, ln
        self.pcm_extent = int((off + ln).max()) if len(off) else 0
        return int(total.value)

    @property
    def num_tiles(self):
        return lib().afe_batch_num_tiles(self._h)

    @property
    def kernel_launches(self):
        return lib().afe_batch_kernel_launches(self._h)

    @property
    def kernel_name(self):
        return lib().afe_batch_kernel_name(self._h).decode()

    def run_device(self, d_pcm_ptr, d_out_ptr):
        _check(lib().afe_batch_run_device(self._h, C.c_void_p(d_pcm_ptr), C.c_void_p(d_out_ptr)))

    def extract_device(self, d_pcm_ptr, d_out_ptr):
        _check(lib().afe_batch_extract_device(self._h, C.c_void_p(d_pcm_ptr), C.c_void_p(d_out_ptr)))

    def corpus_stats(self):
        p, n = C.c_void_p(), C.c_int(0)
        _check(lib().afe_batch_corpus_stats(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    @property
    def normalizer(self):
        """afe_normalizer* that owns the corpus record (scope CORPUS, after plan)."""
        h = lib().afe_batch_normalizer(self._h)
        if not h:
            raise AfeError("the batch has no corpus Normalizer (scope != CORPUS, norm == NONE or not planned)")
        return h

    def allreduce(self, nccl_comm):
        """The one collective of the path, inside the Normalizer subsystem."""
        _check(lib().afe_normalizer_allreduce(C.c_void_p(self.normalizer), C.c_void_p(nccl_comm)))

    def corpus_record(self):
        """HOST copy of the corpus record (after corpus_stats / allreduce)."""
        n = C.c_void_p(self.normalizer)
        s = np.zeros(lib().afe_normalizer_stats_len(n), np.float64)
        _check(lib().afe_normalizer_get_stats(n, s.ctypes.data_as(C.POINTER(C.c_double))))
        return s

    def set_corpus_stats(self, stats):
        s = np.ascontiguousarray(stats, np.float64)
        _check(lib().afe_batch_set_corpus_stats(self._h, s.ctypes.data_as(C.POINTER(C.c_double)), len(s)))

    def normalize_device(self, d_out_ptr):
        _check(lib().afe_batch_normalize_device(self._h, C.c_void_p(d_out_ptr)))

    def synchronize(self):
        _check(lib().afe_batch_synchronize(self._h))

    def run_host(self, pcm, out=None):
        """pcm: host int16 packed per self.sample_offsets; returns host [total_frames, width]."""
        pcm = np.ascontiguousarray(pcm, np.int16)
        assert self.frame_offsets is not None and len(pcm) >= self.pcm_extent
        if out is None:
            out = np.zeros((int(self.frame_offsets[-1]), self.width), np.float32)
        _check(lib().afe_batch_run_host(self._h, pcm.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)))
        return out


def pack_utterances(utts, align=8):
    """Concatenate int16 utterances with every start aligned to `align` samples (16 B for the TMA staging path).
    -> (pcm, offsets[n], lengths[n])"""
    offs, lens, chunks, pos = [], [], [], 0
    for u in utts:
        u = np.ascontiguousarray(u, np.int16)
        offs.append(pos)
        lens.append(len(u))
        chunks.append(u)
        pad = (-len(u)) % align
        if pad:
            chunks.append(np.zeros(pad, np.int16))
        pos += len(u) + pad
    pcm = np.concatenate(chunks) if chunks else np.zeros(0, np.int16)
    return pcm, np.array(offs, np.int64), np.array(lens, np.int64)
