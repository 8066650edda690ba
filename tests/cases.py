"""Shared test data.

KNOWN_ANSWERS restates the golden vectors of the reference's own test-suite for the
distance-transform path (reference automated_test.py, cited per block).  They are plain
data: (labels, kwargs, expected edtsq, dtypes).  Both the oracle (CPU) and the CUDA path are
checked against them with exact equality, as the reference does (`np.all(result == ans)`).

random_volume()/RANDOM_SPECS drive the randomized differential tests (CUDA vs oracle) and the
committed fixtures under tests/golden/ (compiled reference -> oracle, see make_golden.py).
"""
import hashlib

import numpy as np

I = np.inf
INTS = [np.uint8, np.uint16, np.uint32, np.uint64]
NO_BOOL = INTS + [np.float32]
ALL = NO_BOOL + [bool]

ONES5 = [[1] * 5 for _ in range(5)]
HOLE5 = [r[:] for r in ONES5]; HOLE5[2][2] = 0
ISLE5 = [r[:] for r in ONES5]; ISLE5[2][2] = 2
TWO66 = [[1] * 6] * 3 + [[2] * 6] * 3

_seven = np.ones((7, 7), dtype=np.int64)
_seven[0, :] = 0
_seven[3:, :] = 2
_seven[5, 5] = 3

ONES333 = [[[1] * 3] * 3] * 3
_c = [[[1] * 3] * 3, [[1, 1, 1], [1, 4, 1], [1, 1, 1]], [[1] * 3] * 3]


KNOWN_ANSWERS = [
  # ---- 1-D, black border (automated_test.py:62-97) ----
  ("1d_bb_single", [1], dict(black_border=True), [1], ALL),
  ("1d_bb_single5", [5], dict(black_border=True), [1], NO_BOOL),
  ("1d_bb_01110", [0, 1, 1, 1, 0], dict(black_border=True), [0, 1, 4, 1, 0], ALL),
  ("1d_bb_1111", [1, 1, 1, 1], dict(black_border=True), [1, 4, 4, 1], ALL),
  ("1d_bb_1111_w2", [1, 1, 1, 1], dict(black_border=True, anisotropy=2.0), [4, 16, 16, 4], ALL),
  ("1d_bb_multi", [1, 1, 1, 1, 1, 0, 2, 2, 2, 2, 2, 1, 1, 1, 1, 3], dict(black_border=True),
   [1, 4, 9, 4, 1, 0, 1, 4, 9, 4, 1, 1, 4, 4, 1, 1], NO_BOOL),
  # ---- 1-D, no border (automated_test.py:99-146) ----
  ("1d_single", [1], dict(), [I], ALL),
  ("1d_single5", [5], dict(), [I], NO_BOOL),
  ("1d_01110", [0, 1, 1, 1, 0], dict(), [0, 1, 4, 1, 0], ALL),
  ("1d_01111", [0, 1, 1, 1, 1], dict(), [0, 1, 4, 9, 16], ALL),
  ("1d_11110", [1, 1, 1, 1, 0], dict(), [16, 9, 4, 1, 0], ALL),
  ("1d_1111", [1, 1, 1, 1], dict(), [I, I, I, I], ALL),
  ("1d_1111_w2", [1, 1, 1, 1], dict(anisotropy=2.0), [I, I, I, I], ALL),
  ("1d_multi", [1, 1, 1, 1, 1, 0, 2, 2, 2, 2, 2, 1, 1, 1, 1, 3], dict(),
   [25, 16, 9, 4, 1, 0, 1, 4, 9, 4, 1, 1, 4, 4, 1, 1], NO_BOOL),
  # ---- 2-D identities (automated_test.py:188-230) ----
  ("2d_0", [[0]], dict(), [[0]], ALL),
  ("2d_1", [[1]], dict(), [[I]], ALL),
  ("2d_diag", [[1, 0], [0, 1]], dict(), [[1, 0], [0, 1]], ALL),
  ("2d_11_11", [[1, 1], [1, 1]], dict(), [[I, I], [I, I]], ALL),
  ("2d_2x5", [[1] * 5] * 2, dict(), [[I] * 5] * 2, ALL),
  ("2d_bb_0", [[0]], dict(black_border=True), [[0]], ALL),
  ("2d_bb_1", [[1]], dict(black_border=True), [[1]], ALL),
  ("2d_bb_11_11", [[1, 1], [1, 1]], dict(black_border=True), [[1, 1], [1, 1]], ALL),
  ("2d_bb_diag", [[1, 0], [0, 1]], dict(black_border=True), [[1, 0], [0, 1]], ALL),
  ("2d_bb_2x5", [[1] * 5] * 2, dict(black_border=True), [[1] * 5] * 2, ALL),
  # ---- 2-D black border (automated_test.py:232-381) ----
  ("2d_bb_ones5", ONES5, dict(black_border=True),
   [[1, 1, 1, 1, 1], [1, 4, 4, 4, 1], [1, 4, 9, 4, 1], [1, 4, 4, 4, 1], [1, 1, 1, 1, 1]], ALL),
  ("2d_bb_ones5_w56", ONES5, dict(black_border=True, anisotropy=(5.0, 6.0)),
   [[25, 25, 25, 25, 25], [36, 100, 100, 100, 36], [36, 144, 225, 144, 36],
    [36, 100, 100, 100, 36], [25, 25, 25, 25, 25]], ALL),
  ("2d_bb_hole", HOLE5, dict(black_border=True),
   [[1, 1, 1, 1, 1], [1, 2, 1, 2, 1], [1, 1, 0, 1, 1], [1, 2, 1, 2, 1], [1, 1, 1, 1, 1]], ALL),
  ("2d_bb_island", ISLE5, dict(black_border=True),
   [[1, 1, 1, 1, 1], [1, 2, 1, 2, 1], [1, 1, 1, 1, 1], [1, 2, 1, 2, 1], [1, 1, 1, 1, 1]], NO_BOOL),
  ("2d_bb_two66", TWO66, dict(black_border=True),
   [[1] * 6, [1, 4, 4, 4, 4, 1], [1] * 6, [1] * 6, [1, 4, 4, 4, 4, 1], [1] * 6], NO_BOOL),
  ("2d_bb_two65", [[1] * 5] * 3 + [[2] * 5] * 3, dict(black_border=True),
   [[1] * 5, [1, 4, 4, 4, 1], [1] * 5, [1] * 5, [1, 4, 4, 4, 1], [1] * 5], NO_BOOL),
  ("2d_bb_two56", [[1] * 6] * 3 + [[2] * 6] * 2, dict(black_border=True),
   [[1] * 6, [1, 4, 4, 4, 4, 1], [1] * 6, [1] * 6, [1] * 6], NO_BOOL),
  ("2d_bb_seven", _seven.tolist(), dict(black_border=True),
   [[0] * 7, [1] * 7, [1] * 7, [1] * 7, [1, 4, 4, 4, 2, 1, 1], [1, 4, 4, 4, 1, 1, 1], [1] * 7], NO_BOOL),
  # ---- 3-D (automated_test.py:426-551; written transposed there, symmetric here) ----
  ("3d_bb_0", [[[0]]], dict(black_border=True), [[[0]]], ALL),
  ("3d_bb_1", [[[1]]], dict(black_border=True), [[[1]]], ALL),
  ("3d_bb_5", [[[5]]], dict(black_border=True), [[[1]]], NO_BOOL),
  ("3d_bb_ones", ONES333, dict(black_border=True), _c, ALL),
  ("3d_bb_ones_w444", ONES333, dict(black_border=True, anisotropy=(4, 4, 4)),
   [[[16] * 3] * 3, [[16, 16, 16], [16, 64, 16], [16, 16, 16]], [[16] * 3] * 3], ALL),
  # ---- regressions ----
  # automated_test.py:858-877 (3-D shaped 1x6x4, trailing zeros)
  ("3d_trailing_zero",
   [[[1, 1, 1, 0], [1, 1, 1, 1], [1, 1, 1, 1], [0, 0, 0, 0], [0, 0, 0, 0], [0, 0, 0, 0]]], dict(),
   [[[9, 4, 1, 0], [4, 4, 2, 1], [1, 1, 1, 1], [0, 0, 0, 0], [0, 0, 0, 0], [0, 0, 0, 0]]], [np.uint8]),
  # automated_test.py:825-829 (values are edt^2 of [[1, 1.41421], [1, 1]])
  ("2d_column_off_by_one", [[1, 1], [2, 1]], dict(), [[1, 2], [1, 1]], [np.int64]),
]


def known_answer_arrays(case, dtype):
  name, labels, kwargs, expected, _ = case
  return np.array(labels, dtype=dtype), dict(kwargs), np.array(expected, dtype=np.float32)


ANISOTROPIES = [
  (1.0, 1.0, 1.0), (6.0, 6.0, 30.0), (4.0, 4.0, 40.0), (1.0, 2.0, 3.0),
  (0.7, 1.3, 2.9), (3.3, 3.3, 40.7), (0.1, 0.1, 0.1), (1e6, 1.2e6, 40.0),
]
INTEGER_ANISOTROPIES = ANISOTROPIES[:4]
KINDS = ["iid", "few", "blocks", "sparse_zero", "ones", "zeros", "wide", "balls"]


def random_volume(rng, shape, kind, dtype):
  """Seeded synthetic label volumes covering the structures that matter to the algorithm:
  run length ~1 (iid), long runs (ones / sparse_zero, inf-rich without a border), blocky
  segmentation, labels that only differ in the high bits (wide), smooth binary shapes."""
  shape = tuple(int(s) for s in shape)
  nd = len(shape)
  if kind == "iid":
    a = rng.integers(0, 256, shape)
  elif kind == "few":
    a = rng.integers(0, 3, shape)
  elif kind == "blocks":
    b = int(rng.integers(2, 9))
    small = rng.integers(0, 6, tuple((s + b - 1) // b for s in shape))
    a = small
    for ax in range(nd):
      a = np.repeat(a, b, axis=ax)
    a = a[tuple(slice(0, s) for s in shape)]
  elif kind == "sparse_zero":
    a = np.ones(shape, dtype=np.int64)
    for _ in range(int(rng.integers(1, 4))):
      a[tuple(int(rng.integers(0, s)) for s in shape)] = 0
  elif kind == "ones":
    a = np.ones(shape, dtype=np.int64)
  elif kind == "zeros":
    a = np.zeros(shape, dtype=np.int64)
  elif kind == "wide":
    a = rng.integers(0, 3, shape)
  elif kind == "balls":
    grid = np.stack(np.meshgrid(*[np.arange(s) for s in shape], indexing="ij"), axis=-1)
    a = np.zeros(shape, dtype=np.int64)
    for k in range(int(rng.integers(1, 5))):
      c = np.array([rng.uniform(0, s) for s in shape])
      r = rng.uniform(1.0, max(2.0, 0.45 * max(shape)))
      a[((grid - c) ** 2).sum(-1) <= r * r] = k + 1
  else:
    raise ValueError(kind)
  dt = np.dtype(dtype)
  if dt == np.bool_:
    return a != 0
  if kind == "wide" and dt.kind in "iu":
    hi = np.array(1, dtype=np.uint64) << np.uint64(dt.itemsize * 8 - 1)
    a = (a.astype(np.uint64) * (hi + np.uint64(5))).astype(np.dtype("u%d" % dt.itemsize)).view(dt)
    return a
  return a.astype(dt)


def random_case(seed):
  """Deterministic (labels, kwargs) for a seed: dims 1-3, odd sizes, every dtype, both orders."""
  rng = np.random.default_rng(seed)
  nd = int(rng.integers(1, 4))
  hi = {1: 700, 2: 90, 3: 40}[nd]
  shape = tuple(int(rng.integers(1, hi)) for _ in range(nd))
  kind = KINDS[seed % len(KINDS)]
  dtypes = [np.uint8, np.uint16, np.uint32, np.uint64, np.int8, np.int16, np.int32, np.int64,
            bool, np.float32, np.float64]
  dtype = dtypes[(seed // len(KINDS)) % len(dtypes)]
  labels = random_volume(rng, shape, kind, dtype)
  if (seed // 3) % 2:
    labels = np.asfortranarray(labels)
  an = ANISOTROPIES[(seed // 5) % len(ANISOTROPIES)][:nd]
  kwargs = dict(anisotropy=an[0] if nd == 1 else an, black_border=bool((seed // 2) % 2))
  return labels, kwargs


def random_graph_case(seed):
  """Deterministic (labels, graph, kwargs) for the voxel_graph path: 2-D / 3-D, every dtype, both
  memory orders, graph bytes from 'everything allowed' to random bit fields of several dtypes."""
  rng = np.random.default_rng(7000 + seed)
  nd = 2 + seed % 2
  hi = {2: 60, 3: 24}[nd]
  shape = tuple(int(rng.integers(1, hi)) for _ in range(nd))
  dtypes = [np.uint8, np.uint16, np.uint32, np.uint64, np.int8, np.int16, np.int32, np.int64,
            bool, np.float32, np.float64]
  dtype = dtypes[(seed // 2) % len(dtypes)]
  density = [0.97, 0.8, 1.0][seed % 3]
  mask = rng.random(shape) < density
  if dtype is bool:
    labels = mask
  elif np.dtype(dtype).kind == "f":
    labels = (rng.integers(-1, 4, shape) * mask).astype(dtype)     # negatives are background here
  else:
    labels = (rng.integers(1, 5, shape) * mask).astype(dtype)
  gdtype = [np.uint8, np.int8, np.uint32][(seed // 3) % 3]
  graph = rng.integers(0, 64, shape)
  allow_all = rng.random(shape) < [0.9, 0.5, 0.0][(seed // 4) % 3]
  graph = np.where(allow_all, 63, graph).astype(gdtype)
  if (seed // 3) % 2:
    labels = np.asfortranarray(labels)
  if (seed // 5) % 2:
    graph = np.asfortranarray(graph)
  an = ANISOTROPIES[(seed // 5) % len(ANISOTROPIES)][:nd]
  kwargs = dict(anisotropy=an, black_border=bool((seed // 2) % 2))
  return labels, graph, kwargs


# cases whose reference outputs are stored as digests (tests/golden/reference_digests.json)
DIGEST_SEEDS = range(300)                 # random_case: edtsq of each, edt and sdf of every third
DIGEST_GRAPH_SEEDS = range(100, 160)      # random_graph_case: edtsq and sdf


def cfg2_volume():
  """BASELINE.json configs[1]: 512^3 uint32 iid labels 0..255, Fortran order."""
  rng = np.random.default_rng(0)
  return np.asfortranarray(rng.integers(0, 256, (512, 512, 512), dtype=np.uint32))


def digest(a):
  """SHA-256 of an array's dtype, shape and values in C order, with -0.0 folded onto +0.0 and one
  NaN for every NaN, so that two float arrays of one dtype have the same digest exactly when
  np.array_equal(a, b, equal_nan=True) holds for them."""
  a = np.asarray(a)
  if a.dtype.kind == "f":
    a = np.where(np.isnan(a), a.dtype.type(np.nan), a + a.dtype.type(0))
  h = hashlib.sha256(("%s %s " % (a.dtype.str, a.shape)).encode())
  h.update(np.ascontiguousarray(a).tobytes())
  return h.hexdigest()
