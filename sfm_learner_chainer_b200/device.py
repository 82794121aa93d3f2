"""Device-array plumbing.  The library exchanges raw device pointers; any array type that owns CUDA
memory works as a carrier: CuPy arrays (what the reference's Chainer code holds) or torch CUDA tensors
(what this image has).  Nothing here computes."""
import numpy as np

_NP2TORCH = {}


def _torch():
    import torch
    if not _NP2TORCH:
        _NP2TORCH.update({np.dtype('float32'): torch.float32, np.dtype('int32'): torch.int32,
                          np.dtype('uint8'): torch.uint8, np.dtype('float64'): torch.float64,
                          np.dtype('int8'): torch.int8})
    return torch


def is_torch(a):
    return type(a).__module__.startswith('torch')


def is_cupy(a):
    return type(a).__module__.startswith('cupy')


def ptr(a):
    if a is None:
        return None
    if is_torch(a):
        return a.data_ptr()
    if is_cupy(a):
        return a.data.ptr
    return a.__cuda_array_interface__['data'][0]


def check_array(a, name, shape=None, dtype='float32'):
    """Mirror of the reference's type checks (spational_transformer_sampler_interp.py:11-24):
    dtype 'f', expected shape, C-contiguous device memory."""
    if is_torch(a):
        if not a.is_cuda:
            raise TypeError('%s must live on a CUDA device (there is no CPU fallback)' % name)
        dt = str(a.dtype).replace('torch.', '')
        contiguous = a.is_contiguous()
    elif is_cupy(a) or hasattr(a, '__cuda_array_interface__'):
        dt = str(np.dtype(a.dtype))
        contiguous = bool(getattr(a, 'flags', None) is None or a.flags.c_contiguous)
    else:
        raise TypeError('%s must be a CUDA device array (cupy.ndarray or torch.cuda tensor), got %s '
                        '(there is no CPU fallback)' % (name, type(a)))
    if dt != dtype:
        raise TypeError('%s: expected dtype %s, got %s' % (name, dtype, dt))
    if not contiguous:
        raise ValueError('%s must be C-contiguous' % name)
    if shape is not None and tuple(a.shape) != tuple(shape):
        raise ValueError('%s: expected shape %s, got %s' % (name, tuple(shape), tuple(a.shape)))
    return a


def empty(like, shape, dtype='float32'):
    """Allocate through the caller's own allocator (CuPy memory pool / torch caching allocator)."""
    if is_torch(like):
        torch = _torch()
        return torch.empty(tuple(shape), dtype=_NP2TORCH[np.dtype(dtype)], device=like.device)
    if is_cupy(like):
        import cupy
        return cupy.empty(tuple(shape), dtype=dtype)
    raise TypeError('cannot allocate like %s' % type(like))


def current_stream(like):
    if is_torch(like):
        return _torch().cuda.current_stream(like.device).cuda_stream
    if is_cupy(like):
        import cupy
        return cupy.cuda.get_current_stream().ptr
    return 0


def record_event(like):
    """Event recorded on the caller's current stream (None for carriers without a stream API)."""
    if is_torch(like):
        ev = _torch().cuda.Event()
        ev.record(_torch().cuda.current_stream(like.device))
        return ev
    if is_cupy(like):
        import cupy
        ev = cupy.cuda.Event()
        ev.record(cupy.cuda.get_current_stream())
        return ev
    return None


def wait_event(like, ev):
    """Makes the caller's current stream wait for `ev` (no host synchronisation)."""
    if ev is None:
        return
    if is_torch(like):
        _torch().cuda.current_stream(like.device).wait_event(ev)
    elif is_cupy(like):
        import cupy
        cupy.cuda.get_current_stream().wait_event(ev)


def to_numpy(a):
    if is_torch(a):
        return a.detach().cpu().numpy()
    if is_cupy(a):
        return a.get()
    return np.asarray(a)


def from_host_bytes(like, buf):
    """Device uint8 array holding the bytes of `buf` (small parameter blocks), through the caller's allocator."""
    raw = np.frombuffer(bytes(buf), dtype=np.uint8).copy()
    if is_torch(like):
        return _torch().from_numpy(raw).to(like.device)
    if is_cupy(like):
        import cupy
        return cupy.asarray(raw)
    raise TypeError('cannot allocate like %s' % type(like))
