"""B200-native multi-label anisotropic Euclidean distance transform.

Host-side mirror of the reference's Python API (seung-lab/euclidean-distance-transform-3d,
``src/edt.pyx``): same function names, positional/keyword arguments, dtype handling, C/F
order handling and error behaviour, so that ``import edt_b200 as edt`` is a drop-in for
``import edt`` on the distance-transform path.  All arithmetic happens in hand-written
sm_100a CUDA kernels reached through the C ABI of ``include/edt_b200.h`` (ctypes); there is
no CPU implementation in this package -- if ``libedt_b200.so`` is missing or no CUDA device
is usable the calls raise.

Reference entry points mirrored here (file:line in the reference):
  edt      src/edt.pyx:205-242      edtsq    src/edt.pyx:245-310
  sdf      src/edt.pyx:121-158      sdfsq    src/edt.pyx:161-202
  edt1d/edt1dsq  src/edt.pyx:312-399   edt2d/edt2dsq  src/edt.pyx:401-512
  edt3d/edt3dsq  src/edt.pyx:622-734

Differences, all additive: ``parallel`` is accepted and ignored (the CUDA grid replaces the
thread pool); keyword-only ``device=`` selects the GPU; ``sdf``/``sdfsq`` run ONE fused
transform (background treated as a label, sign applied in the last store) instead of two;
``voxel_graph=`` (2-D / 3-D, src/edt.pyx:514-620, 736-844) draws the doubled grid and runs
the transform on the device.
``edt_cuda`` transforms a torch CUDA tensor without touching host memory, and every function
above accepts device-resident input directly (a torch CUDA tensor or any object exposing
``__cuda_array_interface__``) and then returns a torch CUDA tensor.
"""
import ctypes
import os

import numpy as np

__version__ = "0.1.0"
__all__ = [
  "edt", "edtsq", "sdf", "sdfsq",
  "edt1d", "edt1dsq", "edt2d", "edt2dsq", "edt3d", "edt3dsq",
  "edt_cuda", "transform_batch", "each", "each_cuda", "label_stats_cuda", "device_count", "library_path", "EDTError",
]

FLAG_SQRT = 1
FLAG_SIGNED = 2
FLAG_LABELS_ON_DEVICE = 4
FLAG_OUT_ON_DEVICE = 8
FLAG_LABELS_FLOAT = 16

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class EDTError(RuntimeError):
  """A C-ABI call failed (CUDA error, no device, unsupported size...)."""


def library_path():
  """The CUDA library built in-tree by __graft_entry__.build().  EDTB200_LIBRARY overrides the
  path (A/B measurements of two builds on the same box); it is still this library, never a
  CPU substitute."""
  return os.environ.get("EDTB200_LIBRARY") or os.path.join(_HERE, "libedt_b200.so")


def _lib():
  """Load libedt_b200.so (built in-tree by __graft_entry__.build()); fail loudly if absent."""
  global _LIB
  if _LIB is not None:
    return _LIB
  path = library_path()
  if not os.path.exists(path):
    raise ImportError(
      "edt_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
      "There is no CPU fallback." % path)
  lib = ctypes.CDLL(path)
  i64, f32, vp, ci = ctypes.c_int64, ctypes.c_float, ctypes.c_void_p, ctypes.c_int
  lib.edtb200_version.restype = ci
  lib.edtb200_last_error.restype = ctypes.c_char_p
  lib.edtb200_device_count.restype = ci
  lib.edtb200_transform.argtypes = [vp, ci, ci, i64, i64, i64, f32, f32, f32, ci, ci, vp, ci, vp]
  lib.edtb200_transform.restype = ci
  lib.edtb200_transform_multi.argtypes = [vp, ci, ci, i64, i64, i64, f32, f32, f32, ci, ci, vp, vp, ci]
  lib.edtb200_transform_multi.restype = ci
  lib.edtb200_transform_batch.argtypes = [vp, vp, ci, ci, ci, i64, i64, i64, f32, f32, f32, ci, ci, ci]
  lib.edtb200_transform_batch.restype = ci
  lib.edtb200_transform_voxel_graph.argtypes = [vp, ci, vp, ci, i64, i64, i64, f32, f32, f32, ci, ci, vp, ci, vp]
  lib.edtb200_transform_voxel_graph.restype = ci
  lib.edtb200_pass_first.argtypes = [vp, ci, i64, i64, i64, f32, ci, ci, vp, ci, vp]
  lib.edtb200_pass_first.restype = ci
  lib.edtb200_pass_later.argtypes = [vp, ci, ci, i64, i64, i64, f32, ci, ci, ci, vp, ci, vp]
  lib.edtb200_pass_later.restype = ci
  lib.edtb200_slab_pack.argtypes = [vp, vp, i64, i64, i64, ci, ctypes.POINTER(ctypes.c_int64), ci, ci, vp]
  lib.edtb200_slab_pack.restype = ci
  lib.edtb200_slab_face_runs.argtypes = [vp, ci, i64, i64, i64, ci, ci, ci, vp, vp, ci, vp]
  lib.edtb200_slab_face_runs.restype = ci
  lib.edtb200_slab_face_fixup.argtypes = [vp, ci, i64, i64, i64, ci, ci, f32, ci, vp, vp, vp, vp, vp, ci, vp]
  lib.edtb200_slab_face_fixup.restype = ci
  lib.edtb200_profile_passes.argtypes = [ci]
  lib.edtb200_profile_passes.restype = ci
  lib.edtb200_pass_ms.argtypes = [ci, vp]
  lib.edtb200_pass_ms.restype = ci
  lib.edtb200_slab_stage_bytes.argtypes = [i64, i64, ci, ci]
  lib.edtb200_slab_stage_bytes.restype = i64
  lib.edtb200_slab_step.argtypes = [vp, ci, i64, i64, i64, f32, f32, f32, ci, ci, ci, ci, vp, ci, vp, vp, vp,
                                    ctypes.c_uint64, vp, ci, vp]
  lib.edtb200_slab_step.restype = ci
  lib.edtb200_label_stats.argtypes = [vp, ci, vp, i64, i64, i64, ci, vp, vp, vp, vp, vp, vp, ci, vp]
  lib.edtb200_label_stats.restype = ci
  lib.edtb200_label_extract.argtypes = [vp, ci, vp, i64, i64, i64, ctypes.c_uint64, vp, ci, vp, ci, vp]
  lib.edtb200_label_extract.restype = ci
  lib.edtb200_host_alloc.argtypes = [ctypes.c_size_t]
  lib.edtb200_host_alloc.restype = vp
  lib.edtb200_host_free.argtypes = [vp]
  lib.edtb200_host_free.restype = None
  lib.edtb200_release.restype = ci
  _LIB = lib
  return lib


def _check(rc):
  if rc != 0:
    msg = _lib().edtb200_last_error()
    raise EDTError("edt_b200 error %d: %s" % (rc, msg.decode("utf-8", "replace") if msg else "?"))


def device_count():
  return int(_lib().edtb200_device_count())


def nvl(val, default_val):
  return default_val if val is None else val


# ---------------------------------------------------------------------------------------
# host-side logic mirrored from the reference's Cython layer
# ---------------------------------------------------------------------------------------

def _label_view(data, voxel_graph=False):
  """Labels as raw unsigned integers (src/edt.pyx:670-732): signed ints are reinterpreted,
  bool is one byte, floats are compared by value (so -0.0 is folded onto +0.0 first).
  With a voxel graph the labels only say foreground (> 0) or background
  (src/edt_voxel_graph.hpp:76, 151), so floats are kept as they are and `_run` marks them
  EDTB200_LABELS_FLOAT.  Returns None for dtypes the reference does not dispatch on (it then
  returns zeros)."""
  dt = data.dtype
  if dt == np.bool_:
    return data.view(np.uint8)
  if dt.kind in "iu" and dt.itemsize in (1, 2, 4, 8):
    return data.view(np.dtype("u%d" % dt.itemsize))
  if dt == np.float32 or dt == np.float64:
    return data if voxel_graph else (data + dt.type(0)).view(np.dtype("u%d" % dt.itemsize))
  return None


def _check_dims(dims, voxel_graph=None):
  """The reference's dimension checks (src/edt.pyx:291-292, 310)."""
  if voxel_graph is not None and dims not in (2, 3):
    raise TypeError("Voxel connectivity graph is only supported for 2D and 3D. Got {}.".format(dims))
  if dims < 1 or dims > 3:
    raise TypeError("Multi-Label EDT library only supports up to 3 dimensions got {}.".format(dims))


def _anisotropy(anisotropy, dims):
  """Weights of an array of `dims` dimensions, in array axis order (src/edt.pyx:276-310): None
  means ones, and a 1-D array takes a scalar or the first entry of a sequence.  Anything else is
  passed on for _x_fastest to check (a scalar raises TypeError, a wrong length ValueError) once
  the label dtype is known to be supported: for the others the reference returns zeros."""
  if anisotropy is None:
    return (1.0,) * dims
  if dims == 1:
    return (float(np.asarray(anisotropy).reshape(-1)[0]),)
  return anisotropy


def _x_fastest(shape, anisotropy, f_contiguous):
  """(sx, sy, sz), (wx, wy, wz) for an array of `shape`: Fortran order keeps the axes,
  C order reverses them (src/edt.pyx:429-440, 651-664)."""
  dims = [int(s) for s in shape]
  weights = [float(a) for a in anisotropy]
  if len(weights) != len(dims):
    raise ValueError("anisotropy must have one entry per dimension")
  if not f_contiguous:
    dims.reverse()
    weights.reverse()
  while len(dims) < 3:
    dims.append(1)
    weights.append(1.0)
  return dims, weights


# ---------------------------------------------------------------------------------------
# result arrays backed by recycled page-locked memory
# ---------------------------------------------------------------------------------------
# A fresh 512 MiB numpy array costs ~130 000 page faults while the result is copied into it, and
# pageable memory has to be staged through pinned buffers on the way back from the GPU.  Large
# results are therefore placed in page-locked blocks (edtb200_host_alloc) that return to a small
# pool when the array that wraps them is garbage collected: from the second call of a loop on, the
# download is ONE direct DMA into memory that is already mapped.  The pool holds at most
# EDTB200_PINNED_POOL_MB (default 2048) of idle blocks and hands out at most twice that in total;
# beyond it, and for arrays below 4 MiB, plain numpy memory is used.  EDTB200_PINNED_POOL_MB=0
# turns the pool off.

import threading as _threading
import weakref as _weakref

_POOL_LOCK = _threading.Lock()
_POOL_FREE = {}            # nbytes -> [ptr, ...]
_POOL_IDLE = 0             # bytes sitting in _POOL_FREE
_POOL_OUT = 0              # bytes currently behind live arrays
_POOL_MIN = 4 << 20


def _pool_cap():
  try:
    return int(os.environ.get("EDTB200_PINNED_POOL_MB", "2048")) << 20
  except ValueError:
    return 2048 << 20


def _pool_release(ptr, nbytes):
  global _POOL_IDLE, _POOL_OUT
  with _POOL_LOCK:
    _POOL_OUT -= nbytes
    if _POOL_IDLE + nbytes <= _pool_cap():
      _POOL_FREE.setdefault(nbytes, []).append(ptr)
      _POOL_IDLE += nbytes
      return
  try:
    _lib().edtb200_host_free(ctypes.c_void_p(ptr))
  except Exception:        # interpreter shutdown
    pass


def _result_buffer(count):
  """float32[count] for a result: page-locked and recycled when the pool allows, else np.empty."""
  global _POOL_IDLE, _POOL_OUT
  nbytes = int(count) * 4
  cap = _pool_cap()
  if nbytes < _POOL_MIN or cap <= 0:
    return np.empty(count, dtype=np.float32)
  ptr = None
  with _POOL_LOCK:
    free = _POOL_FREE.get(nbytes)
    if free:
      ptr = free.pop()
      _POOL_IDLE -= nbytes
      _POOL_OUT += nbytes
    elif _POOL_OUT + nbytes > 2 * cap:
      return np.empty(count, dtype=np.float32)
  if ptr is None:
    lib = _lib()
    if _POOL_IDLE:                              # make room: drop idle blocks of other sizes
      with _POOL_LOCK:
        for size in list(_POOL_FREE):
          while _POOL_FREE[size] and _POOL_IDLE + nbytes > cap:
            lib.edtb200_host_free(ctypes.c_void_p(_POOL_FREE[size].pop()))
            _POOL_IDLE -= size
    ptr = lib.edtb200_host_alloc(ctypes.c_size_t(nbytes))
    if not ptr:
      return np.empty(count, dtype=np.float32)
    with _POOL_LOCK:
      _POOL_OUT += nbytes
  block = (ctypes.c_char * nbytes).from_address(ptr)
  _weakref.finalize(block, _pool_release, ptr, nbytes)
  return np.frombuffer(block, dtype=np.float32, count=count)


def _run(labels, graph, dims, weights, black_border, flags, out, device=None):
  """The one Python call site of edtb200_transform and, with a `graph`, of
  edtb200_transform_voxel_graph.  `labels`, `graph` and `out` are numpy arrays, transformed on GPU
  `device` before the call returns, or torch CUDA tensors, transformed asynchronously on their own
  device and its current stream.  `dims` and `weights` are _x_fastest's."""
  if isinstance(labels, np.ndarray):
    def ptr(a):
      return a.ctypes.data
    stream, floating = None, labels.dtype.kind == "f"
  else:
    import torch

    def ptr(a):
      return a.data_ptr()
    flags |= FLAG_LABELS_ON_DEVICE | FLAG_OUT_ON_DEVICE
    device, floating = labels.device.index, labels.is_floating_point()
    stream = ctypes.c_void_p(torch.cuda.current_stream(labels.device).cuda_stream)
  if floating:                     # only with a graph: the labels are compared as floats (> 0)
    flags |= FLAG_LABELS_FLOAT
  (sx, sy, sz), (wx, wy, wz) = dims, weights
  rest = (sx, sy, sz, wx, wy, wz, int(bool(black_border)), int(flags), ptr(out), int(device), stream)
  if graph is None:
    _check(_lib().edtb200_transform(ptr(labels), labels.itemsize, labels.ndim, *rest))
  else:
    _check(_lib().edtb200_transform_voxel_graph(ptr(labels), labels.itemsize, ptr(graph), labels.ndim, *rest))


def _graph_bytes(voxel_graph, order):
  """The graph as uint8 in the data's memory order (src/edt.pyx:294-298, 527-530)."""
  g = np.asarray(voxel_graph)
  g = np.ascontiguousarray(g) if order == "C" else np.asfortranarray(g)
  return g.view(np.uint8) if g.dtype in (np.uint8, np.int8) else g.astype(np.uint8)


def _transform_host(data, voxel_graph, anisotropy, black_border, flags, device):
  """A numpy array, answered in its memory order: Fortran order keeps the axes, anything else is
  read in C order (src/edt.pyx:651-664), strided input after a copy.  With a voxel graph this is
  __edt2dsq_voxel_graph / __edt3dsq_voxel_graph, src/edt.pyx:514-620, 736-844."""
  order = "F" if data.flags.f_contiguous else "C"
  if not data.flags.c_contiguous and not data.flags.f_contiguous:
    data = np.ascontiguousarray(data)
  graph = None
  if voxel_graph is not None:
    graph = _graph_bytes(voxel_graph, order)
    if graph.shape != data.shape:
      raise ValueError("voxel_graph must have the shape of data")
  labels = _label_view(data, voxel_graph=graph is not None)
  if labels is None:
    return np.zeros(data.shape, dtype=np.float32, order=order)
  dims, weights = _x_fastest(data.shape, anisotropy, order == "F")
  out = _result_buffer(data.size) if graph is None else np.empty(data.size, dtype=np.float32)
  if graph is None and (isinstance(device, (list, tuple, range))
                        or (isinstance(device, np.ndarray) and device.ndim == 1)):
    # several GPUs of this process share ONE host volume (edtb200_transform_multi): Z slabs for the
    # X / Y passes, Y slabs for the Z pass, re-partitioned over NVLink; exact for any input
    devs = [int(d) for d in device]
    _check(_lib().edtb200_transform_multi(
      labels.ctypes.data, labels.itemsize, data.ndim, *dims, *weights, int(bool(black_border)), int(flags),
      out.ctypes.data, (ctypes.c_int * len(devs))(*devs), len(devs)))
  else:
    if isinstance(device, (list, tuple)):
      device = device[0]                      # the graph transform runs on one GPU
    _run(labels, graph, dims, weights, black_border, flags, out, device)
  return out.reshape(data.shape, order=order)


def _device_array(data):
  """torch CUDA tensor view of `data` if it already lives on a GPU (a torch CUDA tensor, or any
  object exposing `__cuda_array_interface__`: CuPy, Numba, ...), else None.  Zero-copy."""
  if isinstance(data, (np.ndarray, list, tuple)) or np.isscalar(data):
    return None
  mod = type(data).__module__
  if mod.startswith("torch"):
    return data if getattr(data, "is_cuda", False) else None
  if hasattr(data, "__cuda_array_interface__"):
    import torch
    t = torch.as_tensor(data, device="cuda")
    # interface v3: "stream" names the stream the producer's work was queued on (1 = legacy
    # default, 2 = per-thread default, else a cudaStream_t); order torch's current stream after it
    stream = data.__cuda_array_interface__.get("stream")
    if stream is not None and stream != 0:
      cur = torch.cuda.current_stream(t.device)
      if stream in (1, 2):
        torch.cuda.synchronize(t.device)
      elif int(stream) != cur.cuda_stream:
        ev = torch.cuda.Event()
        ev.record(torch.cuda.ExternalStream(int(stream), device=t.device))
        cur.wait_event(ev)
    return t
  return None


def _transform_device(t, voxel_graph, anisotropy, black_border, flags, device=None):
  """A torch CUDA tensor, transformed on its own device (`device` is not used) and current stream,
  answered as a torch CUDA tensor in its memory order (which itself exports DLPack and
  `__cuda_array_interface__`).  As on the host, Fortran order keeps the axes and anything else is
  read in C order (src/edt.pyx:651-664), so a Fortran-ordered tensor is not copied."""
  import torch
  graph = None
  if voxel_graph is not None:
    graph = _device_array(voxel_graph)
    if graph is None:
      graph = torch.as_tensor(np.ascontiguousarray(voxel_graph), device=t.device)
    if graph.shape != t.shape or graph.device != t.device:
      raise ValueError("voxel_graph must have the shape and device of data")
    if graph.dtype not in (torch.uint8, torch.int8):
      graph = graph.to(torch.uint8)
  labels = _torch_label_view(t, voxel_graph=graph is not None)
  if labels is None:
    return torch.zeros(t.shape, dtype=torch.float32, device=t.device)
  rev = tuple(reversed(range(labels.dim())))
  fortran = labels.dim() > 1 and not labels.is_contiguous() and labels.permute(rev).is_contiguous()
  if fortran:
    graph = None if graph is None else graph.permute(rev).contiguous().permute(rev)
  else:
    labels = labels.contiguous()
    graph = None if graph is None else graph.contiguous()
  dims, weights = _x_fastest(labels.shape, anisotropy, fortran)
  out = torch.empty_like(labels, dtype=torch.float32)        # same strides as the labels
  _run(labels, graph, dims, weights, black_border, flags, out)
  return out


def _front_door(data, anisotropy, black_border, voxel_graph, flags, device, fixed_dims=None):
  """Argument handling of edtsq(), src/edt.pyx:276-310, for host arrays and device-resident input
  alike; the result is a numpy array or a torch CUDA tensor, as the input is."""
  on_device = _device_array(data)
  data = np.asarray(data) if on_device is None else on_device
  dims = data.ndim
  if fixed_dims is not None and dims != fixed_dims:
    raise ValueError("expected a %d-D array, got %d-D" % (fixed_dims, dims))
  if 0 in data.shape:
    if on_device is None:
      return np.zeros(shape=data.shape, dtype=np.float32)
    import torch
    return torch.zeros(data.shape, dtype=torch.float32, device=data.device)
  _check_dims(dims, voxel_graph)
  anisotropy = _anisotropy(anisotropy, dims)
  transform = _transform_host if on_device is None else _transform_device
  if voxel_graph is not None and flags & FLAG_SIGNED:
    # sdf / sdfsq with a graph: f(data) - f(data == 0), both under the graph (src/edt.pyx:147-158)
    flags &= ~FLAG_SIGNED
    dt = transform(data, voxel_graph, anisotropy, black_border, flags, device)
    dt -= transform(data == 0, voxel_graph, anisotropy, black_border, flags, device)
    return dt
  return transform(data, voxel_graph, anisotropy, black_border, flags, device)


# ---------------------------------------------------------------------------------------
# public API (signatures follow src/edt.pyx; `device` is keyword-only and additive)
# ---------------------------------------------------------------------------------------

def _pick(device, devices):
  """`devices` (a sequence of GPU ordinals: one host volume spread over them) wins over `device`."""
  if devices is None:
    return device
  devs = [int(d) for d in devices]
  if not devs:
    raise ValueError("devices must name at least one GPU")
  return devs if len(devs) > 1 else devs[0]


def edtsq(data, anisotropy=None, black_border=False, parallel=1, voxel_graph=None, order=None,
          *, device=0, devices=None):
  """Squared anisotropic multi-label EDT of a 1-D, 2-D or 3-D array (src/edt.pyx:245-310).
  `devices=[0, 1, ...]` spreads one host volume over several GPUs (see _transform_host)."""
  return _front_door(data, anisotropy, black_border, voxel_graph, 0, _pick(device, devices))


def edt(data, anisotropy=None, black_border=False, parallel=1, voxel_graph=None, order=None,
        *, device=0, devices=None):
  """Anisotropic multi-label EDT (src/edt.pyx:205-242); the sqrt is fused into the last pass."""
  return _front_door(data, anisotropy, black_border, voxel_graph, FLAG_SQRT, _pick(device, devices))


def sdf(data, anisotropy=None, black_border=False, parallel=1, voxel_graph=None, order=None,
        *, device=0, devices=None):
  """Signed distance function, edt(data) - edt(data == 0) (src/edt.pyx:121-158), computed as
  one transform with background as a label and the sign applied in the last store."""
  return _front_door(data, anisotropy, black_border, voxel_graph, FLAG_SQRT | FLAG_SIGNED, _pick(device, devices))


def sdfsq(data, anisotropy=None, black_border=False, parallel=1, voxel_graph=None, *, device=0, devices=None):
  """Squared signed distance function (src/edt.pyx:161-202)."""
  return _front_door(data, anisotropy, black_border, voxel_graph, FLAG_SIGNED, _pick(device, devices))


def edt1dsq(data, anisotropy=1.0, black_border=False, *, device=0):
  return _front_door(data, anisotropy, black_border, None, 0, device, fixed_dims=1)


def edt1d(data, anisotropy=1.0, black_border=False, *, device=0):
  return _front_door(data, anisotropy, black_border, None, FLAG_SQRT, device, fixed_dims=1)


def edt2dsq(data, anisotropy=(1.0, 1.0), black_border=False, parallel=1, voxel_graph=None,
            *, device=0):
  return _front_door(data, anisotropy, black_border, voxel_graph, 0, device, fixed_dims=2)


def edt2d(data, anisotropy=(1.0, 1.0), black_border=False, parallel=1, voxel_graph=None,
          *, device=0):
  return _front_door(data, anisotropy, black_border, voxel_graph, FLAG_SQRT, device, fixed_dims=2)


def edt3dsq(data, anisotropy=(1.0, 1.0, 1.0), black_border=False, parallel=1, voxel_graph=None,
            *, device=0):
  return _front_door(data, anisotropy, black_border, voxel_graph, 0, device, fixed_dims=3)


def edt3d(data, anisotropy=(1.0, 1.0, 1.0), black_border=False, parallel=1, voxel_graph=None,
          *, device=0):
  return _front_door(data, anisotropy, black_border, voxel_graph, FLAG_SQRT, device, fixed_dims=3)


# ---------------------------------------------------------------------------------------
# device-resident entry (zero-copy): torch CUDA tensor in, torch CUDA tensor out
# ---------------------------------------------------------------------------------------

_TORCH_LABEL_BYTES = None


def _torch_label_bytes(torch):
  global _TORCH_LABEL_BYTES
  if _TORCH_LABEL_BYTES is None:
    table = {torch.bool: 1, torch.uint8: 1, torch.int8: 1, torch.int16: 2, torch.int32: 4,
             torch.int64: 8}
    for name, size in (("uint16", 2), ("uint32", 4), ("uint64", 8)):
      if hasattr(torch, name):
        table[getattr(torch, name)] = size
    _TORCH_LABEL_BYTES = table
  return _TORCH_LABEL_BYTES


def _torch_label_view(t, voxel_graph=False):
  """The torch counterpart of _label_view: `t` itself for integer and bool labels, whose raw bits
  are the labels; floats compared by value (-0.0 folded onto +0.0) as their raw bits, or, with a
  voxel graph, kept as they are; None for dtypes the reference does not dispatch on."""
  import torch
  if t.dtype in _torch_label_bytes(torch):
    return t
  if t.dtype == torch.float32 or t.dtype == torch.float64:
    return t if voxel_graph else (t + 0).view(torch.int32 if t.dtype == torch.float32 else torch.int64)
  return None


def edt_cuda(labels, anisotropy=None, black_border=False, *, sqrt=False, signed=False, out=None,
             voxel_graph=None):
  """Transform a C-contiguous integer/bool torch CUDA tensor of 1-3 dims on its own device
  and current stream, asynchronously; returns a float32 CUDA tensor of the same shape
  (`out` may be passed to reuse a buffer).  Same semantics as edtsq/edt/sdfsq/sdf.
  `voxel_graph` (a uint8/int8 CUDA tensor of the same shape, 2-D / 3-D only, not with `signed`)
  selects the connectivity-graph transform."""
  import torch
  if not (isinstance(labels, torch.Tensor) and labels.is_cuda):
    raise TypeError("edt_cuda expects a torch CUDA tensor")
  nd = labels.dim()
  _check_dims(nd)
  if not labels.is_contiguous():
    labels = labels.contiguous()
  if labels.dtype not in _torch_label_bytes(torch):
    raise TypeError("edt_cuda: unsupported label dtype %s" % labels.dtype)
  if out is None:
    out = torch.empty(labels.shape, dtype=torch.float32, device=labels.device)
  elif not (out.is_cuda and out.dtype == torch.float32 and out.is_contiguous()
            and out.shape == labels.shape and out.device == labels.device):
    raise ValueError("edt_cuda: `out` must be a contiguous float32 CUDA tensor of the same shape/device")
  if labels.numel() == 0:
    return out
  dims, weights = _x_fastest(labels.shape, _anisotropy(anisotropy, nd), False)
  flags = (FLAG_SQRT if sqrt else 0) | (FLAG_SIGNED if signed else 0)
  if voxel_graph is not None:
    _check_dims(nd, voxel_graph)
    if signed:
      raise ValueError("edt_cuda: with voxel_graph, form f(labels) - f(labels == 0) from two calls")
    if not (isinstance(voxel_graph, torch.Tensor) and voxel_graph.device == labels.device
            and voxel_graph.dtype in (torch.uint8, torch.int8) and voxel_graph.shape == labels.shape):
      raise ValueError("edt_cuda: voxel_graph must be a uint8/int8 CUDA tensor shaped like labels")
    voxel_graph = voxel_graph.contiguous()
  _run(labels, voxel_graph, dims, weights, black_border, flags, out)
  return out


def transform_batch(volumes, anisotropy=None, black_border=False, *, sqrt=False, signed=False, outs=None,
                    device=0):
  """edtsq (or edt / sdfsq / sdf via `sqrt` / `signed`) of many arrays of ONE shape, dtype and
  memory order -- e.g. the chunks of a dataset -- pipelined through the GPU: the upload of chunk
  k+1 and the download of chunk k-1 overlap the transform of chunk k (`edtb200_transform_batch`).
  Returns a list of float32 arrays (the arrays of `outs`, if given: same shape and order as the
  inputs, float32; pass pinned buffers, e.g. `torch.empty(..., pin_memory=True).numpy()`, to let
  the copies run at the PCIe rate).  Each result equals the single-call function's."""
  vols = [np.asarray(v) for v in volumes]
  if not vols:
    return []
  first = vols[0]
  _check_dims(first.ndim)
  order = "F" if first.flags.f_contiguous else "C"
  fixed = []
  for v in vols:
    if v.shape != first.shape or v.dtype != first.dtype:
      raise ValueError("transform_batch: all volumes must share one shape and dtype")
    if order == "F" and not v.flags.f_contiguous:
      v = np.asfortranarray(v)
    elif order == "C" and not v.flags.c_contiguous:
      v = np.ascontiguousarray(v)
    fixed.append(v)
  if outs is None:
    outs = [np.empty(first.shape, dtype=np.float32, order=order) for _ in fixed]
  else:
    outs = list(outs)
    if len(outs) != len(fixed):
      raise ValueError("transform_batch: one output array per volume")
    for o in outs:
      ok = isinstance(o, np.ndarray) and o.dtype == np.float32 and o.shape == first.shape and \
          (o.flags.f_contiguous if order == "F" else o.flags.c_contiguous) and o.flags.writeable
      if not ok:
        raise ValueError("transform_batch: outs must be writable float32 arrays shaped and ordered like the volumes")
  if first.size == 0:
    for o in outs:
      o[...] = 0
    return outs
  views = [_label_view(v) for v in fixed]
  if views[0] is None:                      # dtype the reference does not dispatch on: zeros
    for o in outs:
      o[...] = 0
    return outs
  nd = first.ndim
  (sx, sy, sz), (wx, wy, wz) = _x_fastest(first.shape, _anisotropy(anisotropy, nd), order == "F")
  n = len(views)
  lab_ptrs = (ctypes.c_void_p * n)(*[v.ctypes.data for v in views])
  out_ptrs = (ctypes.c_void_p * n)(*[o.ctypes.data for o in outs])
  flags = (FLAG_SQRT if sqrt else 0) | (FLAG_SIGNED if signed else 0)
  _check(_lib().edtb200_transform_batch(lab_ptrs, out_ptrs, n, views[0].dtype.itemsize, nd, sx, sy, sz,
                                        wx, wy, wz, int(bool(black_border)), flags, int(device)))
  return outs


# ---------------------------------------------------------------------------------------
# downstream helper of the reference's headline use case: one multi-label transform, then one
# masked image per label (src/edt.pyx:951-994; README.md:23, 204)
# ---------------------------------------------------------------------------------------

def label_stats_cuda(labels, dt):
  """Per-label statistics of a finished transform in ONE pass on the device: a dict of torch CUDA
  tensors sorted by label -- "labels" (int64, background 0 skipped), "count" (voxels), "max"
  (largest distance), "argmax" (smallest C-order linear index where it is attained), "box"
  (n x 6: inclusive bounding box, low corner then high corner, in ARRAY axis order).
  `labels` and `dt` are C-contiguous CUDA tensors of the same 1-3 dim shape (kernels:
  csrc/edt_each.cuh; the reference builds the same information from run lists,
  src/edt_voxel_graph.hpp:238-275)."""
  import torch
  if not (isinstance(labels, torch.Tensor) and labels.is_cuda and isinstance(dt, torch.Tensor) and dt.is_cuda):
    raise TypeError("label_stats_cuda expects torch CUDA tensors")
  if labels.shape != dt.shape or labels.device != dt.device:
    raise ValueError("labels and dt must have the same shape and device")
  nbytes = _torch_label_bytes(torch).get(labels.dtype)
  if nbytes is None:
    raise TypeError("label_stats_cuda: unsupported label dtype %s" % labels.dtype)
  labels = labels.contiguous()
  dt = dt.contiguous().to(torch.float32)
  nd = labels.dim()
  (sx, sy, sz), _ = _x_fastest(labels.shape, (1.0,) * nd, False)
  dev = labels.device
  stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
  capacity = 1024
  while True:
    keys = torch.empty(capacity, dtype=torch.int64, device=dev)
    count = torch.empty(capacity, dtype=torch.int64, device=dev)
    mx = torch.empty(capacity, dtype=torch.float32, device=dev)
    argmax = torch.empty(capacity, dtype=torch.int64, device=dev)
    box = torch.empty((capacity, 6), dtype=torch.int32, device=dev)
    overflow = torch.zeros(1, dtype=torch.int32, device=dev)
    _check(_lib().edtb200_label_stats(labels.data_ptr(), nbytes, dt.data_ptr(), sx, sy, sz, capacity,
                                      keys.data_ptr(), count.data_ptr(), mx.data_ptr(), argmax.data_ptr(),
                                      box.data_ptr(), overflow.data_ptr(), dev.index, stream))
    used = int((keys != 0).sum().item())
    if int(overflow.item()) == 0 and 2 * used <= capacity:
      break
    capacity *= 4                                    # table too full (or full): again with more room
  sel = torch.nonzero(keys != 0).flatten()
  order = sel[torch.argsort(_unsigned_sort_key(torch, keys[sel], nbytes))]
  b = box[order].to(torch.int64)
  lo = b[:, :nd].flip(1)                             # x0 y0 z0 -> array axis order
  hi = b[:, 3:3 + nd].flip(1)
  return {"labels": keys[order], "count": count[order], "max": mx[order], "argmax": argmax[order],
          "box": torch.cat([lo, hi], dim=1)}


def _unsigned_sort_key(torch, keys, nbytes):
  """Sort key that orders int64-held label bits as the unsigned integers they are."""
  if nbytes < 8:
    return keys
  return keys ^ torch.tensor(-0x8000000000000000, dtype=torch.int64, device=keys.device)


def _label_scalar(key, dtype):
  """The label of numpy `dtype` that a table key (the label's raw bits, zero-extended) stands for."""
  raw = np.array([key & ((1 << (8 * dtype.itemsize)) - 1)], dtype=np.dtype("u%d" % dtype.itemsize))
  return raw.view(dtype)[0]


def each_cuda(labels, dt, in_place=False, *, _stats=None):
  """Device-resident `each` (reference: edt.each, src/edt.pyx:951-994): iterator over
  (label, dt masked to that label) as torch CUDA tensors, labels in ascending order of their raw
  bits (the reference's order is that of a hash map), background skipped.
  One pass of `label_stats_cuda` finds every label's bounding box; each image is then drawn by a
  kernel that touches only that box (the device equivalent of the reference's run-list
  transfer).  in_place=True reuses ONE image: the previous label's box is erased, the next one
  drawn -- do not keep references to it between iterations (the reference marks it read-only)."""
  import torch
  stats = _stats if _stats is not None else label_stats_cuda(labels, dt)
  labels = labels.contiguous()
  dt = dt.contiguous().to(torch.float32)
  nbytes = _torch_label_bytes(torch)[labels.dtype]
  # labels are reported as Python values: bool, uint8 unsigned, torch's other integer types signed
  value_type = np.dtype(bool if labels.dtype == torch.bool else "u1" if labels.dtype == torch.uint8 else
                        "i%d" % nbytes)
  nd = labels.dim()
  (sx, sy, sz), _ = _x_fastest(labels.shape, (1.0,) * nd, False)
  dev = labels.device
  keys = stats["labels"].tolist()
  boxes = stats["box"].tolist()
  lib = _lib()

  class DeviceImageIterator:
    def __len__(self):
      return len(keys)

    def __iter__(self):
      img = torch.zeros(labels.shape, dtype=torch.float32, device=dev) if in_place else None
      prev = None
      for key, bx in zip(keys, boxes):
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        lo, hi = bx[:nd][::-1] + [0] * (3 - nd), bx[nd:][::-1] + [0] * (3 - nd)      # -> x y z order
        cbox = (ctypes.c_int * 6)(*(lo + hi))
        out = img if in_place else torch.zeros(labels.shape, dtype=torch.float32, device=dev)
        if in_place and prev is not None:
          _check(lib.edtb200_label_extract(labels.data_ptr(), nbytes, dt.data_ptr(), sx, sy, sz,
                                           ctypes.c_uint64(0), prev, 1, out.data_ptr(), dev.index, stream))
        _check(lib.edtb200_label_extract(labels.data_ptr(), nbytes, dt.data_ptr(), sx, sy, sz,
                                         ctypes.c_uint64(key & 0xffffffffffffffff), cbox, 0, out.data_ptr(),
                                         dev.index, stream))
        prev = cbox
        yield (_label_scalar(key, value_type).item(), out)

  return DeviceImageIterator()


def each(labels, dt, in_place=False, *, device=0):
  """Iterator over (label, distance transform of that label alone), labels in ascending order,
  background skipped -- same contract as the reference's edt.each (src/edt.pyx:951-994), which
  builds it from run lists (src/edt_voxel_graph.hpp:238-310).  Here labels and dt are uploaded
  ONCE, every label's bounding box comes from one device pass (`label_stats_cuda`), each masked
  image is drawn on the device inside that box, and only the box travels back to be pasted into
  the host image.  in_place=True reuses one read-only image between iterations, as the reference
  does.  Device-resident input (torch CUDA tensors) is handed to `each_cuda`."""
  try:
    import torch
  except ImportError:          # pragma: no cover
    torch = None
  if torch is not None and isinstance(labels, torch.Tensor) and labels.is_cuda:
    return each_cuda(labels, dt, in_place)
  labels = np.asarray(labels)
  dt = np.asarray(dt)
  if labels.shape != dt.shape:
    raise ValueError("labels and dt must have the same shape")
  _check_dims(labels.ndim)
  order = "F" if labels.flags.f_contiguous else "C"
  view = _label_view(labels)
  if view is None or torch is None:
    raise TypeError("each: unsupported label dtype %s" % labels.dtype)
  # memory order decides the axis roles on the device; the images are pasted back in array order
  mem = view.T if order == "F" else view
  dmem = dt.T if order == "F" else dt
  dev = torch.device("cuda", int(device))
  lab_t = torch.from_numpy(np.ascontiguousarray(mem)).to(dev)
  dt_t = torch.from_numpy(np.ascontiguousarray(dmem, dtype=np.float32)).to(dev)
  stats = label_stats_cuda(lab_t, dt_t)
  keys = stats["labels"].tolist()
  boxes = stats["box"].tolist()
  nd = labels.ndim
  inner = each_cuda(lab_t, dt_t, in_place=True, _stats=stats)

  class ImageIterator:
    def __len__(self):
      return len(keys)

    def __iter__(self):
      img = np.zeros(labels.shape, dtype=np.float32, order=order) if in_place else None
      prev = None
      for (key, dimg), bx in zip(inner, boxes):
        sl = tuple(slice(bx[a], bx[nd + a] + 1) for a in range(nd))          # box in device-array axis order
        sub = dimg[sl].cpu().numpy()
        host_sl, host_sub = (sl[::-1], sub.T) if order == "F" else (sl, sub)
        if in_place:
          img.setflags(write=1)
          if prev is not None:
            img[prev] = 0
          img[host_sl] = host_sub
          img.setflags(write=0)
          prev = host_sl
          yield (_label_scalar(key, labels.dtype), img)
        else:
          out = np.zeros(labels.shape, dtype=np.float32, order=order)
          out[host_sl] = host_sub
          yield (_label_scalar(key, labels.dtype), out)

  return ImageIterator()


def release():
  """Free cached device buffers held by the library, and the idle page-locked result blocks."""
  global _POOL_IDLE
  lib = _lib()
  with _POOL_LOCK:
    for size, ptrs in _POOL_FREE.items():
      while ptrs:
        lib.edtb200_host_free(ctypes.c_void_p(ptrs.pop()))
        _POOL_IDLE -= size
  _check(lib.edtb200_release())
