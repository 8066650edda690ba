"""Every kernel variant the axis-pass launchers can choose, against the oracle and the definition.

The launchers in csrc/edt_passes.cuh pick one of many separately compiled kernels from the line
geometry, the pointer alignment, the weights and the run statistics of the previous transform.
`dispatch()` below restates the predicates of plan_first / plan_later (naming the functions and
plan fields it mirrors) and names the branch each pass takes; CASES is a table of inputs chosen so that every reachable branch is taken at least
once, which test_case_table_covers_every_branch checks without a GPU.  The GPU tests then compare
each case bit for bit with the oracle, compare small volumes bit for bit and large-magnitude ones
within 2 ULP with the exact definition (nearest voxel of another label, from scipy's feature
transform and float64 integer offsets), and exercise misaligned device buffers, the forced tile
variants, asymmetric slab borders and the label-statistics hash table.

Branches the table cannot reach on a device with 232 448 bytes of opt-in shared memory:
  - TX = 16 or TX = 8 without `wide`: those widths are chosen only for n >= 1597, i.e. >= 25 warps;
  - the noise variant or the integer hull with TX < 32 or without TMA staging (not instantiated);
  - `too many line tiles` / `too many lines` (> 2^31 tiles) and the first-axis ELIMIT (sx > 1.8M).
"""
import ctypes
import json
import os
import subprocess
import sys
import zlib
from collections import namedtuple

import numpy as np
import pytest

import cases

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SMEM_B200 = 232448                 # cudaDevAttrMaxSharedMemoryPerBlockOptin of a B200
INT_LIMIT = 2147483000.0           # integer_bound (edt_capi.cu), LaterPlan.int_hull (plan_later)
MODES = {"edtsq": (0, 0), "edt": (1, 0), "sdfsq": (0, 1), "sdf": (1, 1)}      # (sqrt, signed)


# ---- dispatch mirror --------------------------------------------------------------------------

def f32_square(w):
  """w * w as the kernels form it: a float32 product (w2 of launch_later, integer_bound)."""
  w = np.float32(w)
  return float(w * w)


def integer_bound(ws, ns):
  """integer_bound (edt_capi.cu): bound of the earlier passes' values when they are exact integers, else -1."""
  bound = 0.0
  for i, (w, n) in enumerate(zip(ws, ns)):
    w2 = f32_square(w)
    if w2 != np.floor(w2) or w2 < 1.0:
      return -1.0
    w0 = float(np.float32(ws[0]))
    if i == 0 and not (w0 == np.floor(w0) and w0 * n < 16777216.0):
      return -1.0
    bound += w2 * float(n) * float(n)
  return bound if bound < INT_LIMIT else -1.0


def tile_boxes(n):
  """tile_boxes (edt_passes.cuh): (nboxes, box_rows) of the TMA staging, LaterPlan.tb."""
  nboxes = (n + 255) // 256
  rows = (n + nboxes - 1) // nboxes
  if nboxes > 1:
    rows = (rows + 3) & ~3
  return nboxes, rows


def tile_smem_bytes(n, tx, rows_alloc):
  """tile_smem_bytes (edt_passes.cuh)."""
  nchunks = (n + 31) >> 5
  return rows_alloc * tx * 4 + nchunks * tx * 12 + ((n + 3) & ~1) * 4 + 16 + nchunks * tx + tx * 4 + 4


def tile_warps(n, tx):
  """plan_later: LaterPlan.warps of one tile before the cap at 32."""
  subs = 32 // tx
  return (((n + 31) >> 5) + subs - 1) // subs


def tile_width(n, smem):
  """plan_later: LaterPlan.tx, the widest of TX = 32, 16, 8 whose tile fits, or 0."""
  nboxes, rows = tile_boxes(n)
  return next((c for c in (32, 16, 8) if tile_smem_bytes(n, c, rows * nboxes) <= smem), 0)


def first_key(sx, label_bytes, flags, lab_addr, f_addr):
  """plan_first: `vecK` (FirstPlan.vec_k = 1, 2, 4, 8 blocks of 128) or `general`; `+epi` when the
  pass has flags (FirstPlan.epilogue: the vector kernel is then the non-Plain instantiation)."""
  epi = "+epi" if flags else ""
  if sx % 4 == 0 and sx <= 1024 and lab_addr % (4 * label_bytes) == 0 and f_addr % 16 == 0:
    kk = 1 if sx <= 128 else 2 if sx <= 256 else 4 if sx <= 512 else 8
    return "vec%d%s" % (kk, epi)
  return "general" + epi


def later_key(n, inner, line_stride, outer_count, outer_stride, w, flags, f_addr, fmax, noise, smem,
              no_int_hull=False):
  """plan_later: ("tile", TX, tma, variant, int_hull, epi) for LaterPlan.tile, or ("long",)."""
  fits32 = n * line_stride + 64 < (1 << 32)                                   # fits32
  if fits32 and n <= 4096 and inner < (1 << 31):
    aligned = f_addr % 16 == 0 and line_stride % 4 == 0 and (outer_count <= 1 or outer_stride % 4 == 0)  # aligned
    tx = tile_width(n, smem)                                                  # LaterPlan.tx
    if tx:
      tma = aligned and inner >= tx                                           # LaterPlan.tma
      w2 = f32_square(w)
      int_hull = (fmax >= 0 and w2 == np.floor(w2) and 1.0 <= w2 < 1048576.0 and
                  fmax + w2 * float(n) * float(n) < INT_LIMIT)
      wide = tile_warps(n, tx) > 16                                           # LaterPlan.wide
      ih = int_hull and not no_int_hull and tx == 32 and tma                  # LaterPlan.int_hull
      if tx == 32 and tma:                                                    # LaterPlan.ctas, tile_variant
        variant = "wide" if wide else "noise" if noise else "normal"
      else:
        variant = "wide" if wide else "normal"
      return ("tile", tx, bool(tma), variant, bool(ih), bool(flags))         # LaterPlan.epilogue
  return ("long",)                                                            # later_axis_long_kernel


def x_fastest(shape, anisotropy, order):
  """(sx, sy, sz), (wx, wy, wz) as edt_b200._x_fastest forms them."""
  dims, ws = list(shape), [float(a) for a in anisotropy]
  if order == "C":
    dims, ws = dims[::-1], ws[::-1]
  while len(dims) < 3:
    dims.append(1)
    ws.append(1.0)
  return dims, ws


def dispatch(shape, order, label_bytes, anisotropy, mode, lab_addr=0, f_addr=0, smem=SMEM_B200, noise=False,
             no_int_hull=False):
  """Branch key of every pass of one transform (run_passes in edt_capi.cu)."""
  nd = len(shape)
  (sx, sy, sz), (wx, wy, wz) = x_fastest(shape, anisotropy, order)
  sqrt, signed = MODES[mode]
  epi = sqrt or signed                                                        # epilogue_flags
  keys = {"x": first_key(sx, label_bytes, signed or (nd == 1 and epi), lab_addr, f_addr)}   # zero_label_flags
  if nd >= 2:                                                                 # later_pass, geom_for_axis
    keys["y"] = later_key(sy, sx, sx, sz, sx * sy, wy, nd == 2 and epi, f_addr,
                          integer_bound([wx], [sx]), noise, smem, no_int_hull)
  if nd >= 3:
    keys["z"] = later_key(sz, sx * sy, sx * sy, 1, 0, wz, epi, f_addr,
                          integer_bound([wx, wy], [sx, sy]), noise, smem, no_int_hull)
  return keys


def reachable_keys(smem=SMEM_B200):
  """Every branch the launchers can take on a device with `smem` bytes of opt-in shared memory."""
  first = {"vec%d%s" % (k, e) for k in (1, 2, 4, 8) for e in ("", "+epi")} | {"general", "general+epi"}
  later = {("long",)}
  widths = {}
  for n in range(1, 4097):
    widths.setdefault(tile_width(n, smem), []).append(n)
  widths.pop(0, None)
  for tx, ns in widths.items():
    can_wide = any(tile_warps(n, tx) > 16 for n in ns)
    can_narrow = any(tile_warps(n, tx) <= 16 for n in ns)
    for tma in (True, False):
      for epi in (False, True):
        variants = (["wide"] if can_wide else []) + (["normal"] if can_narrow else [])
        if tx == 32 and tma and can_narrow:
          variants.append("noise")
        for v in variants:
          for ih in ((False, True) if tx == 32 and tma else (False,)):
            later.add(("tile", tx, tma, v, ih, epi))
  return first, later


# ---- case table -------------------------------------------------------------------------------

Case = namedtuple("Case", "name shape dtype order anisotropy mode border kind")
WIDTHS = [np.uint8, np.uint16, np.uint32, np.uint64]
SX_SIZES = [3, 124, 128, 132, 256, 260, 512, 516, 1020, 1024, 1025, 1028]
N_SIZES = [255, 256, 257, 258, 513, 1596, 1597, 3104, 3105, 4096, 4097]
KINDS = ["blocks", "balls", "sparse_zero", "few"]


def _table():
  out = []
  for i, sx in enumerate(SX_SIZES):            # first axis: every KK, plain and with an epilogue
    dt = WIDTHS[i % 4]
    out.append(Case("x%d-sq" % sx, (5, 7, sx), dt, "C", (2.0, 3.0, 1.0), "edtsq", i % 2 == 0, KINDS[i % 4]))
    out.append(Case("x%d-sdf" % sx, (3, 4, sx), WIDTHS[(i + 1) % 4], "C", (1.0, 1.0, 3.0), "sdf", i % 2 == 1,
                    KINDS[(i + 1) % 4]))
    if i % 3 == 0:
      out.append(Case("x%d-1d-edt" % sx, (sx,), WIDTHS[(i + 2) % 4], "C", (2.0,), "edt", True, "blocks"))
  for i, n in enumerate(N_SIZES):              # later axes: every tile width, TMA on / off, long lines
    dt = WIDTHS[i % 4]
    kind = KINDS[(i + 2) % 4]
    # Y lines: 36 adjacent lines (one full and one partial tile of 32; 2 / 4 / 5 tiles of 16 / 8)
    out.append(Case("y%d-tma" % n, (2, n, 36), dt, "C", (1.0, 2.0, 1.0), "edtsq", i % 2 == 0, kind))
    out.append(Case("y%d-2d-%s" % (n, "edt" if i % 2 else "sdf"), (n, 36), WIDTHS[(i + 1) % 4], "C", (3.0, 1.0),
                    "edt" if i % 2 else "sdf", i % 2 == 1, kind))
    out.append(Case("y%d-plain" % n, (2, n, 35), WIDTHS[(i + 2) % 4], "C", (1.0, 1.0, 1.0), "edtsq", True, kind))
    # Z lines: 12 x 3 = 36 adjacent lines, line stride 36 (TMA) / 7 x 5 = 35 (plain loads)
    out.append(Case("z%d-tma-%s" % (n, "edt" if i % 2 else "sq"), (n, 3, 12), WIDTHS[(i + 3) % 4], "C",
                    (2.0, 1.0, 1.0), "edt" if i % 2 else "edtsq", i % 2 == 0, kind))
    out.append(Case("z%d-plain-sdf" % n, (n, 5, 7), dt, "C", (1.0, 2.0, 1.0), "sdf", i % 2 == 1, kind))
  # fewer adjacent lines than a tile is wide: plain loads although the pointer is aligned
  out.append(Case("y1700-narrow", (3, 1700, 12), np.uint16, "C", (1.0, 1.0, 1.0), "edtsq", True, "balls"))
  out.append(Case("y3200-narrow", (2, 3200, 4), np.uint8, "C", (1.0, 1.0, 1.0), "edt", False, "blocks"))
  out.append(Case("z600-narrow", (600, 4, 4), np.uint32, "C", (1.0, 1.0, 1.0), "edtsq", True, "balls"))
  # Fortran order: x is the first array axis
  out.append(Case("f-order", (260, 40, 300), np.uint64, "F", (1.0, 3.0, 2.0), "sdf", False, "blocks"))
  # non-integer squared weights: double hull tests on the TX = 32 TMA path
  out.append(Case("y300-w1.3", (6, 300, 64), np.uint32, "C", (1.0, 1.3, 0.7), "edtsq", True, "balls"))
  out.append(Case("y300-2d-w1.3-sdf", (300, 64), np.uint16, "C", (1.3, 0.7), "sdf", False, "balls"))
  out.append(Case("z700-w2.9", (700, 8, 16), np.uint8, "C", (2.9, 1.0, 1.0), "edt", False, "blocks"))
  out.append(Case("z700-w2.9-sq", (700, 8, 16), np.uint64, "C", (2.9, 1.0, 1.0), "edtsq", True, "balls"))
  out.extend(HULL_CASES)
  return out


# Integer-hull magnitudes: the bound of the Z (Y) pass, fmax + w2 n^2, just below and just above
# 2147483000.  Sparse background and no border, so that the values run far beyond 2^24.
#   (sx, sy, sz) = (96, 64, 203), w = (178, 148, 207): 2147482969, 31 below the limit; wz = 208 above
#   2-D (sx, sy) = (1044, 512), w = (37, 50): 2147482384, 616 below; wy = 51 above
#   256^3 cubes: w = 104 (2126512128, int hull), w = 105 (2167603200, double hull)
HULL_CASES = [
  Case("ih-z-below", (203, 64, 96), np.uint32, "C", (207.0, 148.0, 178.0), "edtsq", False, "sparse_planes"),
  Case("ih-z-above", (203, 64, 96), np.uint16, "C", (208.0, 148.0, 178.0), "edtsq", False, "sparse_planes"),
  Case("ih-y2d-below", (512, 1044), np.uint8, "C", (50.0, 37.0), "edtsq", False, "sparse_planes"),
  Case("ih-y2d-above", (512, 1044), np.uint64, "C", (51.0, 37.0), "edtsq", False, "sparse_planes"),
  Case("ih-y2d-below-edt", (512, 1044), np.uint16, "C", (50.0, 37.0), "edt", False, "sparse_planes"),
  Case("ih-cube104", (256, 256, 256), np.uint8, "C", (104.0, 104.0, 104.0), "edtsq", False, "sparse_planes"),
  Case("ih-cube105", (256, 256, 256), np.uint8, "C", (105.0, 105.0, 105.0), "edtsq", False, "sparse_planes"),
  # integer data whose earlier passes alone exceed the bound (samples above 2^31, beyond int32):
  # double hull; the bound of integer_bound itself is what keeps the int hull off
  Case("dbl-y2d-fmax", (512, 1044), np.uint16, "C", (1.0, 52.0), "edtsq", False, "sparse_planes"),
  Case("dbl-z-fmax", (203, 64, 96), np.uint32, "C", (100.0, 300.0, 480.0), "edtsq", False, "sparse_planes"),
  # later axes with non-integer weights whose float32 squares are integers (3 and 5): int hull;
  # the same weights with the non-integer one on x: no int hull
  Case("ih-sqrt35", (128, 96, 64), np.uint32, "F", (1.0, 1.7320508, 2.236068), "edtsq", True, "balls"),
  Case("ih-sqrt35-wide-edt", (64, 40, 600), np.uint16, "F", (1.0, 1.7320508, 2.236068), "edt", False, "balls"),
  Case("ih-sqrt35-x", (128, 96, 64), np.uint32, "F", (1.7320508, 1.0, 2.236068), "edtsq", True, "balls"),
  Case("ih-wide-sdf", (700, 16, 32), np.uint32, "C", (3.0, 1.0, 1.0), "sdf", True, "blocks"),
]
CASES = _table()
CASE_BY_NAME = {c.name: c for c in CASES}
# cases re-run in child processes with the tile variant / integer hull forced by the A/B switches
FORCED_SUBSET = ["y256-tma", "y256-2d-edt", "y513-tma", "z258-tma-edt", "z513-tma-sq", "ih-z-below",
                 "ih-y2d-below", "ih-y2d-below-edt", "ih-sqrt35", "ih-sqrt35-wide-edt", "ih-wide-sdf", "y300-w1.3", "y300-2d-w1.3-sdf"]
FORCED_ENVS = {"ctas2": {"EDTB200_TILE_CTAS": "2"}, "ctas3": {"EDTB200_TILE_CTAS": "3"},
               "no-int-hull": {"EDTB200_NO_INT_HULL": "1"}}


def case_keys(case, smem=SMEM_B200, noise=False, no_int_hull=False):
  return dispatch(case.shape, case.order, np.dtype(case.dtype).itemsize, case.anisotropy, case.mode,
                  smem=smem, noise=noise, no_int_hull=no_int_hull)


def covered_keys(smem=SMEM_B200):
  """Branch keys the table is certain to reach.  Where the noise hint decides the variant (TX = 32
  with TMA staging, not wide) it depends on the previous transform in-process, so those branches
  count only for the forced subset: without the hint (EDTB200_TILE_CTAS=3) and with it (=2)."""
  first, later = set(), set()
  for c in CASES:
    for noise in ((False, True) if c.name in FORCED_SUBSET else (False,)):
      k = case_keys(c, smem, noise=noise)
      first.add(k["x"])
      later.update(v for a, v in k.items()
                   if a != "x" and (c.name in FORCED_SUBSET or v[3:4] != ("normal",) or not (v[1] == 32 and v[2])))
  return first, later


def sparse_planes(rng, shape):
  """All foreground but for one background voxel in about a third of the planes along the first
  array axis (the lines of the last pass), mostly on the planes' edges and corners, and one in
  the opposite corners of the first and the last plane.  The distances of nearby planes then
  differ by up to the whole range, the envelopes have vertices far apart, and the last plane
  holds samples close to the largest possible value (for the integer hull: g = f + w2 z^2 near
  the bound)."""
  a = np.ones(shape, dtype=np.int64)

  def edge_biased(s):
    u = rng.random()
    return 0 if u < 0.3 else s - 1 if u < 0.6 else int(rng.integers(0, s))

  for p in range(shape[0]):
    if rng.random() < 0.3:
      a[(p,) + tuple(edge_biased(s) for s in shape[1:])] = 0
  a[(0,) + tuple(s - 1 for s in shape[1:])] = 0
  a[(shape[0] - 1,) + (0,) * (len(shape) - 1)] = 0
  return a


def case_labels(case):
  rng = np.random.default_rng(zlib.crc32(case.name.encode()))
  if case.kind == "sparse_planes":
    a = sparse_planes(rng, case.shape).astype(case.dtype)
  else:
    a = cases.random_volume(rng, case.shape, case.kind, case.dtype)
  if np.dtype(case.dtype).itemsize == 8 and case.kind != "sparse_planes":
    a = np.where(a != 0, a | np.uint64(1 << 63), a).astype(np.uint64)     # labels that differ in bit 63 too
  return np.asfortranarray(a) if case.order == "F" else np.ascontiguousarray(a)


def run_case(edt_or_oracle, case, labels=None):
  labels = case_labels(case) if labels is None else labels
  fn = getattr(edt_or_oracle, case.mode)
  an = case.anisotropy[0] if len(case.shape) == 1 else case.anisotropy
  return fn(labels, anisotropy=an, black_border=case.border)


# ---- helpers ----------------------------------------------------------------------------------

def ulp_diff(a, b):
  a = np.asarray(a, np.float32).ravel()
  b = np.asarray(b, np.float32).ravel()
  special = ~np.isfinite(a) | ~np.isfinite(b)
  if not np.array_equal(a[special], b[special], equal_nan=True):
    return np.inf
  ai = a[~special].view(np.int32).astype(np.int64)
  bi = b[~special].view(np.int32).astype(np.int64)
  ai = np.where(ai < 0, np.int64(-2**31) - ai, ai)
  bi = np.where(bi < 0, np.int64(-2**31) - bi, bi)
  return 0 if ai.size == 0 else int(np.abs(ai - bi).max())


def assert_same(got, want, what):
  assert got.shape == want.shape, (what, got.shape, want.shape)
  if not np.array_equal(got, want, equal_nan=True):
    bad = np.argwhere(~((got == want) | (np.isnan(got) & np.isnan(want))))
    first = tuple(bad[0])
    raise AssertionError("%s: %d of %d voxels differ; first at %s: got %r want %r (max ulp %s)" % (
      what, len(bad), got.size, first, got[first], want[first], ulp_diff(got, want)))


def definition_edtsq(labels, anisotropy, black_border):
  """Squared distance from every voxel to the nearest voxel of another label (or, with a black
  border, the nearest voxel outside the volume), background 0: the feature voxel from scipy's
  exact feature transform, one call per label, its squared distance in float64 from integer
  offsets, rounded once to float32."""
  from scipy import ndimage
  w2 = np.array([f32_square(a) for a in anisotropy])
  assert np.all(w2 == np.floor(w2)), "integer squared weights only: the float64 sum is then exact"
  out = np.zeros(labels.shape, dtype=np.float64)
  for lab in np.unique(labels):
    if lab == 0:
      continue
    mask = labels == lab
    m = np.pad(mask, 1) if black_border else mask
    if m.all():
      out[mask] = np.inf
      continue
    idx = ndimage.distance_transform_edt(m, sampling=np.sqrt(w2), return_distances=False, return_indices=True)
    d2 = np.zeros(m.shape, dtype=np.float64)
    for ax in range(m.ndim):
      pos = np.arange(m.shape[ax]).reshape([-1 if a == ax else 1 for a in range(m.ndim)])
      d2 += w2[ax] * (idx[ax] - pos).astype(np.float64) ** 2
    del idx
    if black_border:
      d2 = d2[(slice(1, -1),) * m.ndim]
    out[mask] = d2[mask]
  return out.astype(np.float32)


def device_smem():
  import torch
  return int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)


# ---- CPU: the table reaches every branch ------------------------------------------------------

def test_case_table_covers_every_branch():
  first_all, later_all = reachable_keys()
  first, later = covered_keys()
  print("\nfirst-axis branches covered:", ", ".join(sorted(first)))
  print("later-axis branches covered:")
  for k in sorted(later, key=str):
    print("  ", k)
  assert first == first_all, sorted(first_all - first)
  assert later == later_all, sorted(later_all - later, key=str)
  # TX ranges of the issue's arithmetic: 32 up to 1596, 16 up to 3104, 8 up to 4096
  assert [later_key(n, 36, 36, 2, 36 * n, 1.0, 0, 0, -1, False, SMEM_B200)[1] for n in
          (1596, 1597, 3104, 3105, 4096)] == [32, 16, 16, 8, 8]
  assert later_key(4097, 36, 36, 2, 36 * 4097, 1.0, 0, 0, -1, False, SMEM_B200) == ("long",)
  # the integer-hull threshold cases sit on the intended sides of it
  for name, side in (("ih-z-below", True), ("ih-z-above", False), ("ih-y2d-below", True), ("ih-y2d-above", False),
                     ("ih-cube104", True), ("ih-cube105", False), ("ih-sqrt35", True), ("ih-sqrt35-x", False),
                     ("dbl-y2d-fmax", False), ("dbl-z-fmax", False)):
    c = CASE_BY_NAME[name]
    k = case_keys(c)
    last = k["z"] if len(c.shape) == 3 else k["y"]
    assert last[0] == "tile" and last[1] == 32 and last[2], (name, last)
    assert last[4] == side, (name, last)
  (sx, sy, sz), (wx, wy, wz) = x_fastest((203, 64, 96), (207.0, 148.0, 178.0), "C")
  margin = INT_LIMIT - (integer_bound([wx, wy], [sx, sy]) + wz * wz * sz * sz)
  assert 0 < margin <= 1000, margin
  margin2 = INT_LIMIT - (integer_bound([37.0], [1044]) + 50.0 ** 2 * 512 ** 2)
  assert 0 < margin2 <= 1000, margin2


def test_definition_reference_on_cpu(oracle):
  """The scipy-based definition agrees with the oracle's brute-force evaluation (no GPU)."""
  rng = np.random.default_rng(5)
  for shape, an in (((9, 11, 7), (1.0, 2.0, 3.0)), ((13, 10), (2.0, 1.0)), ((40,), (3.0,))):
    lab = cases.random_volume(rng, shape, "few", np.uint16)
    for bb in (False, True):
      a = an[0] if len(shape) == 1 else an
      assert_same(definition_edtsq(lab, an, bb), oracle.bruteforce_edtsq(lab, anisotropy=a, black_border=bb),
                  (shape, bb))


# ---- GPU --------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_case_table_covers_every_branch_on_device():
  """The same coverage with the device's own opt-in shared memory per block."""
  smem = device_smem()
  first_all, later_all = reachable_keys(smem)
  first, later = covered_keys(smem)
  print("\nshared_memory_per_block_optin = %d" % smem)
  assert first == first_all, sorted(first_all - first)
  assert later == later_all, sorted(later_all - later, key=str)


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c.name for c in CASES])
def test_case_vs_oracle(edt, oracle, name):
  case = CASE_BY_NAME[name]
  labels = case_labels(case)
  got = run_case(edt, case, labels)
  assert_same(got, run_case(oracle, case, labels), (name, case_keys(case, device_smem())))


DEFINITION_CASES = [
  ((96, 96, 96), np.uint8, "balls", (1.0, 1.0, 1.0), True),
  ((96, 80, 72), np.uint16, "balls", (40.0, 4.0, 4.0), False),
  ((64, 90, 70), np.uint32, "few_blocks", (3.0, 2.0, 1.0), True),
  ((70, 60, 96), np.uint64, "sparse_zero", (2.0, 1.0, 5.0), False),
  ((300, 280), np.uint32, "balls", (3.0, 5.0), True),
  ((520, 64), np.uint8, "few_blocks", (1.0, 7.0), False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(DEFINITION_CASES)))
def test_exact_definition(edt, i):
  """Below 2^24 with integer squared weights every intermediate value is exact: bit for bit."""
  shape, dtype, kind, an, bb = DEFINITION_CASES[i]
  rng = np.random.default_rng(100 + i)
  if kind == "few_blocks":
    small = rng.integers(0, 3, tuple((s + 15) // 16 for s in shape))
    lab = small
    for ax in range(len(shape)):
      lab = np.repeat(lab, 16, axis=ax)
    lab = lab[tuple(slice(0, s) for s in shape)].astype(dtype)
  else:
    lab = cases.random_volume(rng, shape, kind, dtype)
  want = definition_edtsq(lab, an, bb)
  assert np.nanmax(np.where(np.isinf(want), 0, want)) < 2**24
  assert_same(edt.edtsq(lab, anisotropy=an, black_border=bb), want, (shape, kind, an, bb))
  for order_lab in (np.asfortranarray(lab),):
    assert_same(edt.edtsq(order_lab, anisotropy=an, black_border=bb), want, "F order")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["ih-z-below", "ih-z-above", "ih-y2d-below", "ih-y2d-above", "ih-cube104",
                                  "ih-cube105", "dbl-y2d-fmax", "dbl-z-fmax"])
def test_large_magnitudes_vs_definition(edt, oracle, name):
  """Beyond 2^24 each pass rounds once: at most 2 ULP from the definition, bit for bit with the oracle."""
  case = CASE_BY_NAME[name]
  labels = case_labels(case)
  got = run_case(edt, case, labels)
  assert_same(got, run_case(oracle, case, labels), name)
  want = definition_edtsq(labels, case.anisotropy, case.border)
  finite = np.isfinite(want)
  if name.startswith("ih-"):
    assert want[finite].max() > 2**24               # fp32 rounding in the passes
  assert np.array_equal(np.isfinite(got), finite)
  ulps = ulp_diff(got[finite], want[finite])
  assert ulps <= 2, (name, ulps)


MISALIGNED_SHAPES = [(128, 128, 128), (64, 512, 64), (1000, 1028)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", MISALIGNED_SHAPES, ids=["x".join(map(str, s)) for s in MISALIGNED_SHAPES])
def test_misaligned_device_buffers(edt, oracle, shape):
  """Labels and out at storage offsets: general first-axis kernel, plain-load tiles."""
  import torch
  rng = np.random.default_rng(zlib.crc32(repr(shape).encode()))
  n = int(np.prod(shape))
  smem = device_smem()
  an = (1.0, 2.0, 3.0)[:len(shape)]
  for j, (np_t, torch_t) in enumerate(((np.uint8, torch.uint8), (np.int16, torch.int16), (np.int32, torch.int32),
                                       (np.int64, torch.int64))):
    kind = ("blocks", "balls", "blocks", "few")[j]
    lab = cases.random_volume(rng, shape, kind, np_t)
    mode = "edt" if j % 2 else "edtsq"
    want = getattr(oracle, mode)(lab, anisotropy=an, black_border=j < 2)
    aligned = torch.from_numpy(lab).cuda()
    ref = edt.edt_cuda(aligned, an, j < 2, sqrt=mode == "edt").cpu().numpy()
    assert_same(ref, want, (shape, np_t, "aligned"))
    fbuf = torch.empty(n + 4, dtype=torch.float32, device="cuda")
    out = fbuf[1:1 + n].view(shape)
    for k in (1, 2, 3):
      buf = torch.zeros(n + 4, dtype=torch_t, device="cuda")
      view = buf[k:k + n].view(shape)
      view.copy_(aligned)
      keys = dispatch(shape, "C", lab.itemsize, an, mode, lab_addr=view.data_ptr(), f_addr=out.data_ptr(), smem=smem)
      assert keys["x"].startswith("general") and all(not v[2] for a, v in keys.items() if a != "x"), keys
      got = edt.edt_cuda(view, an, j < 2, sqrt=mode == "edt", out=out)
      assert got.data_ptr() == out.data_ptr()
      assert_same(got.cpu().numpy(), want, (shape, np_t, k, keys))
    # out alone misaligned, labels aligned
    got = edt.edt_cuda(aligned, an, j < 2, sqrt=mode == "edt", out=out)
    assert_same(got.cpu().numpy(), want, (shape, np_t, "out misaligned"))


@pytest.mark.gpu
def test_noise_prediction_order(edt, oracle):
  """The tile variant depends on the previous transform's run statistics: structured data right
  after noise (the 2-CTA variant) and noise right after structured data must both be exact."""
  rng = np.random.default_rng(77)
  noise = rng.integers(0, 256, (96, 128, 128)).astype(np.uint32)
  balls = cases.random_volume(rng, (96, 128, 128), "balls", np.uint32)
  vor = np.ascontiguousarray(np.repeat(np.repeat(np.repeat(rng.integers(1, 9, (12, 16, 16)), 8, 0), 8, 1), 8, 2)
                             .astype(np.uint32))
  want = {k: oracle.edtsq(v, anisotropy=(1.0, 1.0, 2.0)) for k, v in (("noise", noise), ("balls", balls),
                                                                       ("voronoi", vor))}
  for seq in (("noise", "balls"), ("balls", "noise"), ("noise", "voronoi"), ("voronoi", "noise")):
    vols = {"noise": noise, "balls": balls, "voronoi": vor}
    for k in seq:
      got = edt.edtsq(vols[k], anisotropy=(1.0, 1.0, 2.0))
    assert_same(got, want[seq[-1]], seq)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", sorted(FORCED_ENVS))
def test_forced_variants(oracle, mode, tmp_path):
  """The forced subset in a child process with EDTB200_TILE_CTAS=2 / =3 or EDTB200_NO_INT_HULL=1
  (read once per process): each child writes digests, compared here with the oracle's."""
  env = dict(os.environ)
  env.update(FORCED_ENVS[mode])
  path = tmp_path / "cases.digest"
  res = subprocess.run([sys.executable, os.path.abspath(__file__), str(path)] + FORCED_SUBSET, env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
  assert res.returncode == 0, res.stdout + res.stderr
  got = json.loads(path.read_text())
  bad = [n for n in FORCED_SUBSET if got[n] != cases.digest(run_case(oracle, CASE_BY_NAME[n]))]
  assert not bad, (mode, bad)


def _pass_api(edt, lab_t, f, sx, sy, sz, steps):
  import torch
  lib = edt._lib()
  nb = lab_t.element_size()
  s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
  for step in steps:
    if step[0] == "first":
      _, w, bb, flags = step
      assert lib.edtb200_pass_first(lab_t.data_ptr(), nb, sx, sy, sz, w, bb, flags, f.data_ptr(), 0, s) == 0
    else:
      _, axis, w, lo, hi, flags = step
      assert lib.edtb200_pass_later(lab_t.data_ptr(), nb, axis, sx, sy, sz, w, lo, hi, flags, f.data_ptr(), 0, s) == 0
  torch.cuda.synchronize()
  return f.cpu().numpy()


ASYM_SHAPES = [(64, 300, 40), (36, 1700, 3), (35, 41, 520), (12, 3, 3200)]     # (sx, sy, sz)


@pytest.mark.gpu
@pytest.mark.parametrize("sxyz", ASYM_SHAPES, ids=["x".join(map(str, s)) for s in ASYM_SHAPES])
def test_asymmetric_borders(edt, oracle, sxyz):
  """edtb200_pass_later with border_lo != border_hi (the slab split's inner faces) on Y and on Z."""
  import torch
  sx, sy, sz = sxyz
  rng = np.random.default_rng(sx * sy + sz)
  for dtype in (np.uint16, np.uint64):
    lab = cases.random_volume(rng, (sz, sy, sx), "balls", dtype)                  # C order: z, y, x
    lab_t = torch.from_numpy(lab.view(np.dtype("i%d" % lab.itemsize))).cuda()
    for lo, hi in ((0, 1), (1, 0)):
      f = torch.empty(lab.shape, dtype=torch.float32, device="cuda")
      got = _pass_api(edt, lab_t, f, sx, sy, sz, [("first", 2.0, 1, 0), ("later", 1, 3.0, lo, hi, 0)])
      want = oracle.pass_later(lab, oracle.pass_first(lab, 2.0, True), 1, 3.0, lo, hi)
      assert_same(got, want, (sxyz, dtype, "Y", lo, hi))
      got = _pass_api(edt, lab_t, f, sx, sy, sz, [("first", 1.0, 0, 0), ("later", 1, 1.0, 1, 1, 0),
                                                  ("later", 2, 2.0, lo, hi, 0)])
      want = oracle.pass_later(lab, oracle.pass_later(lab, oracle.pass_first(lab, 1.0, False), 1, 1.0, 1, 1),
                               2, 2.0, lo, hi)
      assert_same(got, want, (sxyz, dtype, "Z", lo, hi))


def _numpy_label_stats(lab, dt):
  flat = lab.reshape(-1)
  d = dt.reshape(-1)
  keys, inv = np.unique(flat, return_inverse=True)
  inv = inv.reshape(-1)
  count = np.bincount(inv, minlength=len(keys))
  mx = np.full(len(keys), -np.inf, dtype=np.float32)
  np.maximum.at(mx, inv, d)
  idx = np.arange(flat.size)
  argmax = np.full(len(keys), flat.size, dtype=np.int64)
  hit = d == mx[inv]
  np.minimum.at(argmax, inv[hit], idx[hit])
  coords = np.unravel_index(idx, lab.shape)
  lo = np.stack([np.full(len(keys), 1 << 30) for _ in coords], 1)
  hi = np.stack([np.full(len(keys), -1) for _ in coords], 1)
  for a, c in enumerate(coords):
    np.minimum.at(lo[:, a], inv, c)
    np.maximum.at(hi[:, a], inv, c)
  keep = keys != 0
  return keys[keep], count[keep], mx[keep], argmax[keep], np.concatenate([lo, hi], 1)[keep]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["5000-uint32", "uint64-shared-low-bits", "uint64-bit63"])
def test_label_stats_regrow(edt, kind):
  """label_stats_cuda rebuilds its hash table (1024 slots) once it is more than half full."""
  import torch
  rng = np.random.default_rng(zlib.crc32(kind.encode()))
  shape = (40, 64, 48)
  cells = rng.integers(0, 5000, (10, 16, 12))
  base = np.repeat(np.repeat(np.repeat(cells, 4, 0), 4, 1), 4, 2)         # ~ 1900 distinct cells of 4^3
  base = (base * 7 + rng.integers(0, 7, shape) * (rng.random(shape) < 0.5)) % 5003   # ~ 5000 labels
  if kind == "5000-uint32":
    lab = base.astype(np.uint32)
  elif kind == "uint64-shared-low-bits":
    lab = ((base.astype(np.uint64) % np.uint64(50)) |
           ((base.astype(np.uint64) // np.uint64(50) + np.uint64(1)) << np.uint64(32)))
    lab[base == 0] = 0
  else:
    lab = np.where(base % 2 == 1, base.astype(np.uint64) | np.uint64(1 << 63), base.astype(np.uint64))
  nlab = len(np.unique(lab)) - int((lab == 0).any())
  assert nlab > 2000
  signed = np.dtype("i%d" % lab.itemsize)
  lab_t = torch.from_numpy(lab.view(signed)).cuda()
  dt_t = edt.edt_cuda(lab_t, (1.0, 2.0, 3.0), True)
  dt = dt_t.cpu().numpy()
  stats = edt.label_stats_cuda(lab_t, dt_t)
  keys, count, mx, argmax, box = _numpy_label_stats(lab, dt)
  assert np.array_equal(stats["labels"].cpu().numpy().astype(np.uint64), keys.astype(np.uint64))
  assert np.array_equal(stats["count"].cpu().numpy(), count)
  assert np.array_equal(stats["max"].cpu().numpy(), mx)
  assert np.array_equal(stats["argmax"].cpu().numpy(), argmax)
  assert np.array_equal(stats["box"].cpu().numpy(), box)
  # each_cuda: every label's image is dt on that label and 0 elsewhere; summed over all labels
  # (in place, one image) they give dt on the foreground exactly once
  acc = torch.zeros_like(dt_t)
  labels_seen = []
  for i, (value, img) in enumerate(edt.each_cuda(lab_t, dt_t, in_place=True)):
    acc += img
    labels_seen.append(value)
    if i % 997 == 0:
      want = np.where(lab.view(signed) == value, dt, 0).astype(np.float32)
      assert_same(img.cpu().numpy(), want, (kind, value))
  assert len(labels_seen) == nlab
  assert np.array_equal(np.array(labels_seen, dtype=signed).view(lab.dtype), keys)
  assert_same(acc.cpu().numpy(), np.where(lab != 0, dt, 0).astype(np.float32), (kind, "sum of images"))


# ---- child process of test_forced_variants ----------------------------------------------------

if __name__ == "__main__":
  sys.path.insert(0, ROOT)
  import edt_b200
  out_path, names = sys.argv[1], sys.argv[2:]
  result = {n: cases.digest(run_case(edt_b200, CASE_BY_NAME[n])) for n in names}
  with open(out_path, "w") as fh:
    json.dump(result, fh)
