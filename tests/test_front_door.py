"""The Python front door: every input kind reaches the C ABI through the same decisions.

CPU part: the C library is replaced by a recording fake, so these tests need neither a GPU nor
the built library.  For each host input the test states the C calls the reference's rules ask for
(label bytes in memory order, x-fastest sizes and weights, flags, device) and the result's type,
shape, dtype and memory order, or the exception.

GPU part: device-resident input (torch CUDA tensors and `__cuda_array_interface__` objects) must
answer exactly as the same input on the host does.
"""
import ctypes
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)
import edt_b200  # noqa: E402

SQRT, SIGNED, LABELS_FLOAT = 1, 2, 16


class RecordingLib:
  """Stands in for libedt_b200.so: every transform entry point returns 0 and records its arguments,
  with the host bytes it would read (labels, voxel graph) taken while the call runs."""

  def __init__(self):
    self.calls = []

  def _common(self, fn, nbytes, ndim, sx, sy, sz, wx, wy, wz, black_border, flags):
    return dict(fn=fn, label_bytes=nbytes, ndim=ndim, sizes=(sx, sy, sz), weights=(wx, wy, wz),
                border=black_border, flags=flags)

  def edtb200_transform(self, labels, nbytes, ndim, sx, sy, sz, wx, wy, wz, black_border, flags, out, device,
                        stream):
    rec = self._common("transform", nbytes, ndim, sx, sy, sz, wx, wy, wz, black_border, flags)
    rec.update(labels=ctypes.string_at(labels, sx * sy * sz * nbytes), device=device, stream=stream)
    self.calls.append(rec)
    return 0

  def edtb200_transform_voxel_graph(self, labels, nbytes, graph, ndim, sx, sy, sz, wx, wy, wz, black_border, flags,
                                    out, device, stream):
    rec = self._common("transform_voxel_graph", nbytes, ndim, sx, sy, sz, wx, wy, wz, black_border, flags)
    rec.update(labels=ctypes.string_at(labels, sx * sy * sz * nbytes), graph=ctypes.string_at(graph, sx * sy * sz),
               device=device, stream=stream)
    self.calls.append(rec)
    return 0

  def edtb200_transform_multi(self, labels, nbytes, ndim, sx, sy, sz, wx, wy, wz, black_border, flags, out, devices,
                              count):
    rec = self._common("transform_multi", nbytes, ndim, sx, sy, sz, wx, wy, wz, black_border, flags)
    rec.update(labels=ctypes.string_at(labels, sx * sy * sz * nbytes), devices=list(devices)[:count])
    self.calls.append(rec)
    return 0

  def edtb200_transform_batch(self, labels, outs, count, nbytes, ndim, sx, sy, sz, wx, wy, wz, black_border, flags,
                              device):
    rec = self._common("transform_batch", nbytes, ndim, sx, sy, sz, wx, wy, wz, black_border, flags)
    rec.update(labels=[ctypes.string_at(labels[k], sx * sy * sz * nbytes) for k in range(count)], device=device)
    self.calls.append(rec)
    return 0


@pytest.fixture
def fake(monkeypatch):
  lib = RecordingLib()
  monkeypatch.setattr(edt_b200, "_LIB", lib)
  return lib


# ---- what the reference's rules ask for -------------------------------------------------------

def memory_order(data):
  """Fortran-ordered arrays keep their axes, everything else (C order, strided views, lists) is
  read in C order with the axes reversed (src/edt.pyx:651-664)."""
  return "F" if data.flags.f_contiguous else "C"


def x_fastest(data, anisotropy):
  sizes, weights = list(data.shape), [float(a) for a in anisotropy]
  if memory_order(data) == "C":
    sizes.reverse()
    weights.reverse()
  return tuple(sizes + [1] * (3 - data.ndim)), tuple(weights + [1.0] * (3 - data.ndim))


def call(data, flags=0, anisotropy=None, border=False, device=0, graph=None, devices=None):
  """The one C call for `data`: labels by value as raw bits (src/edt.pyx:670-732), -0.0 folded onto
  +0.0; with a voxel graph float labels go as they are, marked EDTB200_LABELS_FLOAT."""
  data = np.asarray(data)
  order = memory_order(data)
  sizes, weights = x_fastest(data, anisotropy if anisotropy is not None else (1.0,) * data.ndim)
  if data.dtype.kind == "f" and graph is None:
    labels = np.where(data == 0, np.zeros((), data.dtype), data)
  else:
    labels = data
  if data.dtype.kind == "f" and graph is not None:
    flags |= LABELS_FLOAT
  rec = dict(label_bytes=data.dtype.itemsize, ndim=data.ndim, sizes=sizes, weights=weights, border=int(border),
             flags=flags, labels=labels.tobytes(order))
  if devices is not None:
    rec.update(fn="transform_multi", devices=devices)
  elif graph is not None:
    rec.update(fn="transform_voxel_graph", graph=np.asarray(graph).astype(np.uint8).tobytes(order), device=device,
               stream=None)
  else:
    rec.update(fn="transform", device=device, stream=None)
  return rec


def gives(calls, shape, order):
  return ("gives", calls, tuple(shape), order)


CASES = []


def case(name, run, expect):
  CASES.append(pytest.param(run, expect, id=name))


rng = np.random.default_rng(5)
BASE = rng.integers(0, 4, (3, 4, 5))
FLAGS = {"edtsq": 0, "edt": SQRT, "sdfsq": SIGNED, "sdf": SQRT | SIGNED}
DTYPES = [np.bool_, np.uint8, np.int8, np.uint16, np.int16, np.uint32, np.int32, np.uint64, np.int64,
          np.float32, np.float64, np.float16]
FLOATS = np.array([[-2.5, -0.0, 0.0, 1.0], [np.nan, 3.5, -0.0, 2.0], [0.0, 1.0, -1.0, 1.0]], np.float32)


def labels_of(dtype):
  """(3, 4, 5) labels of `dtype`, with negative values and -0.0 where the dtype has them."""
  if dtype == np.bool_:
    return BASE != 0
  if np.dtype(dtype).kind == "i":
    return np.where(BASE == 3, -1, BASE).astype(dtype)
  if np.dtype(dtype).kind == "f":
    return np.where(BASE == 0, -0.0, np.where(BASE == 3, -1.5, BASE)).astype(dtype)
  return BASE.astype(dtype)


# every label dtype, C and F order, through every reference-named function of any dimension
for dt in DTYPES:
  for order in "CF":
    lab = np.asarray(labels_of(dt), order=order)
    name = "%s-%s" % (np.dtype(dt).name, order)
    supported = np.dtype(dt) != np.float16
    for fn, flags in FLAGS.items():
      case("%s-%s" % (fn, name), lambda m, fn=fn, lab=lab: getattr(m, fn)(lab),
           gives([call(lab, flags)] if supported else [], lab.shape, order))
    case("edt3dsq-" + name, lambda m, lab=lab: m.edt3dsq(lab, (2.0, 3.0, 4.0), True),
         gives([call(lab, 0, (2.0, 3.0, 4.0), True)] if supported else [], lab.shape, order))
    plane = np.asarray(lab[1], order=order)
    case("edt2d-" + name, lambda m, plane=plane: m.edt2d(plane, (2.0, 3.0)),
         gives([call(plane, SQRT, (2.0, 3.0))] if supported else [], plane.shape, memory_order(plane)))
    line = np.ascontiguousarray(lab[1, 2])
    case("edt1dsq-" + name, lambda m, line=line: m.edt1dsq(line, 2.0),
         gives([call(line, 0, (2.0,))] if supported else [], line.shape, "F"))
    # with a voxel graph: floats keep their value (foreground iff > 0), sdf is f(data) - f(data == 0)
    graph = np.asarray(rng.integers(0, 64, lab.shape).astype(np.uint8), order=order)
    for fn, flags in FLAGS.items():
      want = [call(lab, flags & SQRT, graph=graph)] if supported else []      # unsupported: f(data) is zeros
      if flags & SIGNED:
        want.append(call(lab == 0, flags & SQRT, graph=graph))
      elif supported:
        want = [call(lab, flags, graph=graph)]
      case("%s-graph-%s" % (fn, name), lambda m, fn=fn, lab=lab, graph=graph: getattr(m, fn)(lab, voxel_graph=graph),
           gives(want, lab.shape, order))

# float labels with negative values, -0.0 and NaN
for fn, flags in FLAGS.items():
  g = rng.integers(0, 64, FLOATS.shape).astype(np.uint8)
  case("%s-floats" % fn, lambda m, fn=fn: getattr(m, fn)(FLOATS), gives([call(FLOATS, flags)], FLOATS.shape, "C"))
  want = ([call(FLOATS, flags & SQRT, graph=g), call(FLOATS == 0, flags & SQRT, graph=g)] if flags & SIGNED
          else [call(FLOATS, flags, graph=g)])
  case("%s-floats-graph" % fn, lambda m, fn=fn, g=g: getattr(m, fn)(FLOATS, voxel_graph=g),
       gives(want, FLOATS.shape, "C"))

# memory layouts: strided views and lists are read in C order
big = rng.integers(0, 3, (6, 8, 5)).astype(np.uint16)
view = big[::2, 1:-1, ::-1]
case("strided", lambda m: m.edt(view, (1.0, 2.0, 3.0)),
     gives([call(np.ascontiguousarray(view), SQRT, (1.0, 2.0, 3.0))], view.shape, "C"))
fview = np.asfortranarray(big)[::2, 1:-1]
case("strided-from-F", lambda m: m.edtsq(fview), gives([call(np.ascontiguousarray(fview))], fview.shape, "C"))
sgraph = rng.integers(0, 64, big.shape).astype(np.uint8)[::2, 1:-1, ::-1]
case("strided-graph", lambda m: m.edtsq(view, voxel_graph=sgraph),
     gives([call(np.ascontiguousarray(view), graph=sgraph)], view.shape, "C"))
case("list-2d", lambda m: m.edtsq([[1, 1, 0], [1, 2, 2]]),
     gives([call(np.array([[1, 1, 0], [1, 2, 2]]))], (2, 3), "C"))
case("list-1d", lambda m: m.edt([0, 1, 1, 0]), gives([call(np.array([0, 1, 1, 0]), SQRT)], (4,), "F"))
case("list-graph", lambda m: m.edtsq([[1, 1], [0, 1]], voxel_graph=[[63, 63], [63, 63]]),
     gives([call(np.array([[1, 1], [0, 1]]), graph=np.full((2, 2), 63))], (2, 2), "C"))
cgraph = np.ascontiguousarray(rng.integers(0, 64, (3, 4, 5)).astype(np.int8))
flab = np.asfortranarray(labels_of(np.uint32))
case("graph-other-order-int8", lambda m: m.edtsq(flab, voxel_graph=cgraph),
     gives([call(flab, graph=cgraph)], flab.shape, "F"))
bgraph = rng.random((3, 4, 5)) < 0.5
case("graph-bool", lambda m: m.edt(flab, voxel_graph=bgraph), gives([call(flab, SQRT, graph=bgraph)], flab.shape, "F"))
case("graph-shape", lambda m: m.edtsq(flab, voxel_graph=bgraph[:2]), ValueError)
case("graph-shape-float16", lambda m: m.edtsq(labels_of(np.float16), voxel_graph=bgraph[:2]), ValueError)

# dimensions and empty input
case("0d", lambda m: m.edtsq(np.uint8(3)), TypeError)
case("0d-array", lambda m: m.edt(np.array(1, np.uint32)), TypeError)
case("4d", lambda m: m.edtsq(np.ones((2, 2, 2, 2), np.uint8)), TypeError)
case("4d-graph", lambda m: m.edtsq(np.ones((2, 2, 2, 2), np.uint8), voxel_graph=np.ones((2, 2, 2, 2), np.uint8)),
     TypeError)
case("1d-graph", lambda m: m.edtsq(np.ones(4, np.uint8), voxel_graph=np.ones(4, np.uint8)), TypeError)
case("empty-2d", lambda m: m.edtsq(np.zeros((0, 3), np.uint8)), gives([], (0, 3), "C"))
case("empty-list", lambda m: m.edt([]), gives([], (0,), "C"))
case("empty-F", lambda m: m.sdf(np.zeros((4, 0, 2), np.uint32, order="F")), gives([], (4, 0, 2), "C"))
case("empty-4d", lambda m: m.edtsq(np.zeros((2, 0, 2, 2), np.uint8)), gives([], (2, 0, 2, 2), "C"))
case("empty-graph", lambda m: m.sdf(np.zeros((0, 3), np.uint8), voxel_graph=np.zeros((0, 3), np.uint8)),
     gives([], (0, 3), "C"))
case("empty-1d-graph", lambda m: m.edtsq(np.zeros(0, np.uint8), voxel_graph=np.zeros(0, np.uint8)),
     gives([], (0,), "C"))
case("edt2d-on-3d", lambda m: m.edt2d(labels_of(np.uint8)), ValueError)
case("edt1d-on-2d", lambda m: m.edt1d(np.ones((2, 2), np.uint8)), ValueError)
case("edt3d-on-empty-2d", lambda m: m.edt3d(np.zeros((0, 2), np.uint8)), ValueError)

# anisotropy: None -> ones; 1-D takes a scalar or the first element of a sequence; 2-D / 3-D take
# exactly one weight per axis (wrong length: ValueError, scalar: TypeError)
line = np.array([1, 0, 2, 2, 0], np.int32)
img = np.asfortranarray(labels_of(np.int32)[0])
vol = labels_of(np.int32)
for an, want in ((None, 1.0), (2.5, 2.5), ((2.0, 3.0), 2.0), ([4.0], 4.0), (np.array([5.0, 6.0]), 5.0),
                 (np.float32(1.5), 1.5)):
  case("aniso-1d-%r" % (an,), lambda m, an=an: m.edtsq(line, an), gives([call(line, 0, (want,))], line.shape, "F"))
case("aniso-1d-empty-seq", lambda m: m.edtsq(line, ()), IndexError)
case("aniso-2d-default", lambda m: m.edtsq(img), gives([call(img, 0, (1.0, 1.0))], img.shape, "F"))
case("aniso-2d-list", lambda m: m.edtsq(img, [2, 3]), gives([call(img, 0, (2.0, 3.0))], img.shape, "F"))
case("aniso-2d-scalar", lambda m: m.edtsq(img, 2.0), TypeError)
case("aniso-2d-long", lambda m: m.edtsq(img, (1.0, 2.0, 3.0)), ValueError)
case("aniso-3d-array", lambda m: m.sdf(vol, np.array([4, 4, 40])),
     gives([call(vol, SQRT | SIGNED, (4.0, 4.0, 40.0))], vol.shape, "C"))
case("aniso-3d-short", lambda m: m.edt3d(vol, (1.0, 2.0)), ValueError)
case("aniso-3d-scalar", lambda m: m.edt(vol, 3.0), TypeError)
case("aniso-3d-scalar-graph", lambda m: m.edt(vol, 3.0, voxel_graph=np.ones(vol.shape, np.uint8)), TypeError)
case("aniso-3d-short-graph", lambda m: m.edt(vol, (1.0, 2.0), voxel_graph=np.ones(vol.shape, np.uint8)), ValueError)
case("aniso-3d-graph", lambda m: m.edt(vol, (1, 2, 3), voxel_graph=np.ones(vol.shape, np.uint8)),
     gives([call(vol, SQRT, (1.0, 2.0, 3.0), graph=np.ones(vol.shape))], vol.shape, "C"))
# the reference returns zeros for label dtypes it does not dispatch on, whatever the anisotropy
f16 = labels_of(np.float16)
case("aniso-3d-scalar-float16", lambda m: m.edt(f16, 3.0), gives([], f16.shape, "C"))
case("aniso-3d-scalar-float16-graph", lambda m: m.edt(f16, 3.0, voxel_graph=np.ones(f16.shape, np.uint8)),
     gives([], f16.shape, "C"))

# devices
case("device", lambda m: m.edt(vol, device=2), gives([call(vol, SQRT, device=2)], vol.shape, "C"))
case("devices-empty", lambda m: m.edtsq(vol, devices=[]), ValueError)
case("devices-one", lambda m: m.edtsq(vol, devices=[3], device=1), gives([call(vol, device=3)], vol.shape, "C"))
case("devices-two", lambda m: m.sdf(vol, devices=(0, 1)),
     gives([call(vol, SQRT | SIGNED, devices=[0, 1])], vol.shape, "C"))
case("devices-range", lambda m: m.edtsq(np.asfortranarray(vol), device=range(3)),
     gives([call(np.asfortranarray(vol), devices=[0, 1, 2])], vol.shape, "F"))
case("devices-graph", lambda m: m.sdfsq(vol, voxel_graph=np.ones(vol.shape, np.uint8), devices=[1, 2]),
     gives([call(vol, graph=np.ones(vol.shape), device=1), call(vol == 0, graph=np.ones(vol.shape), device=1)],
           vol.shape, "C"))
case("devices-float16", lambda m: m.edtsq(f16, devices=[0, 1]), gives([], f16.shape, "C"))


def batch_call(vols, flags=0, anisotropy=None, border=False, device=0):
  one = call(vols[0], flags, anisotropy, border, device)
  one.update(fn="transform_batch", labels=[call(v, flags, anisotropy, border, device)["labels"] for v in vols])
  del one["stream"]
  return one


# transform_batch and each: argument checks and the batch call
vols = [labels_of(np.int16), labels_of(np.int16)[::-1]]
fvols = [np.asfortranarray(v) for v in vols]
case("batch", lambda m: m.transform_batch(vols, (1.0, 2.0, 3.0), True, sqrt=True),
     ("batch", [batch_call([np.ascontiguousarray(v) for v in vols], SQRT, (1.0, 2.0, 3.0), True)], vol.shape, "C"))
case("batch-F-mixed", lambda m: m.transform_batch([fvols[0], vols[1]], signed=True, device=1),
     ("batch", [batch_call(fvols, SIGNED, device=1)], vol.shape, "F"))
case("batch-1d-scalar", lambda m: m.transform_batch([line, line], 2.0),
     ("batch", [batch_call([line, line], 0, (2.0,))], line.shape, "F"))
case("batch-1d-sequence", lambda m: m.transform_batch([line], (2.0, 3.0)),
     ("batch", [batch_call([line], 0, (2.0,))], line.shape, "F"))
case("batch-3d-scalar", lambda m: m.transform_batch(vols, 2.0), TypeError)
case("batch-3d-short", lambda m: m.transform_batch(vols, (2.0, 3.0)), ValueError)
case("batch-float16", lambda m: m.transform_batch([f16, f16]), ("batch", [], f16.shape, "C"))
case("batch-empty-volumes", lambda m: m.transform_batch([np.zeros((0, 2), np.uint8)] * 2),
     ("batch", [], (0, 2), "C"))
case("batch-none", lambda m: m.transform_batch([]), ("batch", [], None, None))
case("batch-4d", lambda m: m.transform_batch([np.ones((2, 2, 2, 2), np.uint8)]), TypeError)
case("batch-0d", lambda m: m.transform_batch([np.uint8(1)]), TypeError)
case("batch-shapes", lambda m: m.transform_batch([vols[0], vols[0][:2]]), ValueError)
case("batch-dtypes", lambda m: m.transform_batch([vols[0], vols[0].astype(np.int32)]), ValueError)
case("batch-outs-count", lambda m: m.transform_batch(vols, outs=[np.empty(vol.shape, np.float32)]), ValueError)
case("batch-outs-order", lambda m: m.transform_batch(vols, outs=[np.empty(vol.shape, np.float32, order="F")] * 2),
     ValueError)
case("each-shapes", lambda m: m.each(vol, np.zeros((3, 4, 4), np.float32)), ValueError)
case("each-4d", lambda m: m.each(np.ones((2, 2, 2, 2), np.uint8), np.ones((2, 2, 2, 2), np.float32)), TypeError)
case("each-0d", lambda m: m.each(np.uint8(1), np.float32(1)), TypeError)
case("each-float16", lambda m: m.each(f16, np.zeros(f16.shape, np.float32)), TypeError)
case("edt_cuda-host-array", lambda m: m.edt_cuda(vol), TypeError)


def _same_call(got, want):
  assert got.keys() == want.keys()
  for key in want:
    assert got[key] == want[key], key


@pytest.mark.parametrize("run, expect", CASES)
def test_host_input(fake, run, expect):
  if isinstance(expect, type):
    with pytest.raises(expect):
      run(edt_b200)
    return
  kind, calls, shape, order = expect
  result = run(edt_b200)
  assert len(fake.calls) == len(calls)
  for got, want in zip(fake.calls, calls):
    _same_call(got, want)
  results = result if kind == "batch" else [result]
  if shape is None:
    assert results == []
  for res in results:
    assert type(res) is np.ndarray and res.dtype == np.float32 and res.shape == shape
    assert res.flags.f_contiguous if order == "F" else res.flags.c_contiguous


# ---- device-resident input answers as the host does ----------------------------------------

class Foreign:
  """Exposes only `__cuda_array_interface__`, as a CuPy or Numba array does."""

  def __init__(self, tensor):
    self.keep = tensor
    self.__cuda_array_interface__ = tensor.__cuda_array_interface__


def _bits_equal(dev, host):
  got = dev.cpu().numpy()
  assert got.shape == host.shape and got.dtype == host.dtype
  nan = np.isnan(host)
  assert np.array_equal(np.isnan(got), nan)
  assert np.array_equal(got[~nan].view(np.uint32), host[~nan].view(np.uint32))


def _device_forms(host):
  """The host array as a torch CUDA tensor of the same strides, and as a foreign device array."""
  import torch
  t = torch.from_numpy(host).cuda() if host.flags.c_contiguous else \
      torch.from_numpy(np.ascontiguousarray(host.T)).cuda().T
  assert t.stride() == tuple(s // host.itemsize for s in host.strides)
  return [t, Foreign(t)]


@pytest.mark.gpu
@pytest.mark.parametrize("order", ["C", "F"])
def test_device_signed_graph_matches_host(order):
  """sdf / sdfsq with a voxel graph are f(data) - f(data == 0) on the caller's labels: negative
  values and NaN are background for f(data) and foreground for f(data == 0), -0.0 is zero."""
  import torch
  rng = np.random.default_rng(22)
  lab = rng.choice(np.array([-2.5, -0.0, 0.0, 1.0, 3.5, np.nan], np.float32), size=(12, 17, 9))
  lab = np.asarray(lab, order=order)
  graph = np.asarray(rng.integers(0, 64, lab.shape).astype(np.uint8), order=order)
  for fn in ("sdf", "sdfsq"):
    for bb in (False, True):
      with np.errstate(invalid="ignore"):
        host = getattr(edt_b200, fn)(lab, (1.0, 2.0, 1.5), bb, voxel_graph=graph)
      for dev_lab in _device_forms(lab):
        for dev_graph in (graph, torch.from_numpy(np.ascontiguousarray(graph)).cuda()):
          got = getattr(edt_b200, fn)(dev_lab, (1.0, 2.0, 1.5), bb, voxel_graph=dev_graph)
          assert isinstance(got, torch.Tensor) and got.is_cuda
          if order == "F":
            assert got.stride() == tuple(s // 4 for s in lab.strides)
          _bits_equal(got, host)


@pytest.mark.gpu
def test_device_1d_sequence_anisotropy():
  """A 1-D array takes the first entry of a sequence anisotropy, on the device as on the host."""
  import torch
  line = np.random.default_rng(23).integers(0, 3, 300).astype(np.int32)
  for dev_line in _device_forms(line):
    for fn in ("edtsq", "edt", "sdf"):
      _bits_equal(getattr(edt_b200, fn)(dev_line, (2.0, 3.0)), getattr(edt_b200, fn)(line, (2.0, 3.0)))
  _bits_equal(edt_b200.edt_cuda(torch.from_numpy(line).cuda(), (2.0, 3.0)), edt_b200.edtsq(line, 2.0))


@pytest.mark.gpu
def test_device_scalar_anisotropy_and_4d_graph_raise_type_error():
  import torch
  vol = np.asfortranarray(np.random.default_rng(24).integers(0, 3, (9, 8, 7)).astype(np.uint16))
  for dev_vol in _device_forms(vol):
    with pytest.raises(TypeError):
      edt_b200.edtsq(dev_vol, 2.0)
    with pytest.raises(TypeError):
      edt_b200.edt2dsq(edt_b200._device_array(dev_vol)[0], 2.0)
  ones = torch.ones((2, 2, 2, 2), dtype=torch.uint8, device="cuda")
  with pytest.raises(TypeError, match="Voxel connectivity"):
    edt_b200.edtsq(ones, voxel_graph=ones)


@pytest.mark.gpu
def test_device_unsupported_label_dtype_gives_zeros():
  """The reference returns zeros for label dtypes it does not dispatch on (float16, ...)."""
  import torch
  half = np.asfortranarray(np.random.default_rng(25).integers(0, 3, (9, 8, 7))).astype(np.float16)
  assert np.all(edt_b200.edtsq(half) == 0)
  for dev_half in _device_forms(half):
    for kw in ({}, {"voxel_graph": np.ones(half.shape, np.uint8)}):
      got = edt_b200.edt(dev_half, (1.0, 2.0, 3.0), **kw)
      assert isinstance(got, torch.Tensor) and got.is_cuda and got.dtype == torch.float32
      assert got.shape == half.shape and not bool(got.any())
