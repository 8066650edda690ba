"""GPU parity tests (-m gpu) on BASELINE-sized structured volumes and on the per-label views.

* Long runs with varying heights (Voronoi cells, balls) at 512 rows per line -- the inputs that
  exercise the lower-envelope stages of the later-axis kernel (hull build per chunk, stitching
  across chunk boundaries, read-out) -- compared LIVE with the compiled, unmodified reference
  (oracle/_ref) where it is present, else with the C restatement.
* The whole 512^3 headline volume (BASELINE configs[1]) against the compiled reference's stored result.
* edt.each / each_cuda / label_stats_cuda against the reference's own edt.each
  (src/edt.pyx:951-994) and against plain numpy masking.
"""
import numpy as np
import pytest

from test_parity_gpu import assert_same

pytestmark = pytest.mark.gpu


def voronoi_labels(shape, nseeds, seed, dtype=np.uint32):
  """Nearest-seed labelling (cfg2c of SURVEY.md section 8d), F-ordered."""
  from scipy.spatial import cKDTree
  rng = np.random.default_rng(seed)
  pts = rng.uniform(0, 1, (nseeds, 3)) * np.array(shape)
  grid = np.stack(np.meshgrid(*[np.arange(s, dtype=np.float32) for s in shape], indexing="ij"), -1).reshape(-1, 3)
  _, idx = cKDTree(pts).query(grid, workers=-1)
  return np.asfortranarray((idx + 1).astype(dtype).reshape(shape))


def ball_labels(shape, nballs, rmin, rmax, seed, dtype=np.uint8):
  """Binary union of random balls (cfg3b of SURVEY.md section 8d), F-ordered."""
  rng = np.random.default_rng(seed)
  ax = [np.arange(s, dtype=np.float32) for s in shape]
  gx, gy, gz = np.meshgrid(*ax, indexing="ij", sparse=True)
  lab = np.zeros(shape, dtype=bool)
  for _ in range(nballs):
    c = rng.uniform(0, 1, 3) * np.array(shape)
    r = rng.uniform(rmin, rmax)
    lab |= ((gx - c[0]) ** 2 + (gy - c[1]) ** 2 + (gz - c[2]) ** 2) <= r * r
  return np.asfortranarray(lab.astype(dtype))


def checker(reference, oracle):
  """The compiled reference with all host threads where it exists, else the C restatement."""
  import os
  if reference is not None:
    return lambda fn, lab, **kw: getattr(reference, fn)(lab, parallel=os.cpu_count() or 1, **kw)
  return lambda fn, lab, **kw: getattr(oracle, fn)(lab, **kw)


@pytest.mark.parametrize("kind", ["voronoi", "balls"])
def test_long_varying_runs_512_rows(edt, oracle, reference, kind):
  # lines of 512 voxels along x and y (16 chunks of 32 rows, 3 CTAs per SM), 96 along z
  shape = (512, 512, 96)
  lab = voronoi_labels(shape, 40, 5) if kind == "voronoi" else ball_labels(shape, 12, 30, 110, 6)
  ref = checker(reference, oracle)
  for bb in (False, True):
    assert_same(edt.edtsq(lab, anisotropy=(1, 1, 1), black_border=bb),
                ref("edtsq", lab, anisotropy=(1, 1, 1), black_border=bb), (kind, shape, bb))
  # the long axis last as well (z lines of 512 voxels), anisotropic, through sqrt and sign
  lab2 = np.asfortranarray(np.transpose(lab, (2, 1, 0)))
  assert_same(edt.sdf(lab2, anisotropy=(3, 2, 1)), ref("sdf", lab2, anisotropy=(3, 2, 1)), (kind, "sdf"))


@pytest.mark.parametrize("kind", ["voronoi", "balls"])
def test_structured_256_cubed_live(edt, oracle, reference, kind):
  shape = (256, 256, 256)
  lab = voronoi_labels(shape, 120, 7) if kind == "voronoi" else ball_labels(shape, 30, 15, 60, 8)
  ref = checker(reference, oracle)
  assert_same(edt.edtsq(lab, anisotropy=(1, 1, 1)), ref("edtsq", lab, anisotropy=(1, 1, 1)), (kind, 256))
  assert_same(edt.edt(lab, anisotropy=(0.7, 1.3, 2.9), black_border=True),
              ref("edt", lab, anisotropy=(0.7, 1.3, 2.9), black_border=True), (kind, 256, "non-integer"))


def test_cfg2_full_volume_live(edt):
  # BASELINE.json configs[1], the whole 512^3 volume against the compiled reference's result, stored
  # as a digest (bit-exact, see cases.digest) by tests/golden/make_golden.py
  import json
  import os
  import cases
  with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")) as fh:
    want = json.load(fh)["cfg2_512"]["edtsq"]
  got = edt.edtsq(cases.cfg2_volume(), anisotropy=(1, 1, 1))
  assert got.dtype == np.float32 and got.shape == (512, 512, 512)
  assert cases.digest(got) == want, "cfg2 512^3 differs from the compiled reference's edtsq"


def test_wide_lines_and_rows_that_are_not_stored(edt, oracle, reference):
  """Lines of 513..1024 rows (one wide CTA per SM, decoupled warps, chunk mask) and the rows the later
  passes do not store because they keep their value (the passes work in place): solid volumes with
  and without a border through every epilogue, label noise (every row of Y / Z unchanged), blocks."""
  ref = checker(reference, oracle)
  rng = np.random.default_rng(31)
  wide = np.ones((24, 1024, 16), dtype=np.uint8, order="F")
  for fn in ("edtsq", "edt", "sdf"):
    for bb in (False, True):
      assert_same(getattr(edt, fn)(wide, anisotropy=(6, 6, 30), black_border=bb),
                  ref(fn, wide, anisotropy=(6, 6, 30), black_border=bb), ("wide ones", fn, bb))
  wide[11, 700, 5] = 0
  wide[3, 64:96, :] = 7                                     # a chunk-aligned slab of another label
  assert_same(edt.edt(wide, anisotropy=(1, 2, 1)), ref("edt", wide, anisotropy=(1, 2, 1)), "wide hole")
  for n in (1000, 1024, 513):
    noise = np.asfortranarray(rng.integers(0, 200, (20, n, 12), dtype=np.uint32))
    for _ in range(2):                                      # the second call takes the label-noise variant
      got = edt.edtsq(noise, black_border=True)
    assert_same(got, ref("edtsq", noise, black_border=True), ("wide noise", n))
    blocks = np.asfortranarray(np.repeat(np.repeat(rng.integers(1, 5, (3, (n + 31) // 32, 2), dtype=np.uint16), 8, 0),
                                         32, 1)[:, :n].repeat(8, 2))
    assert_same(edt.sdf(blocks, anisotropy=(2, 1, 3)), ref("sdf", blocks, anisotropy=(2, 1, 3)), ("wide blocks", n))
  # 512-row lines (three CTAs per SM): solid two-label volume, every function
  solid = np.ones((40, 512, 36), dtype=np.uint16, order="F")
  solid[:, :, 18:] = 2
  solid[:, 300:, :9] = 0
  for fn in ("edtsq", "edt", "sdfsq", "sdf"):
    assert_same(getattr(edt, fn)(solid, anisotropy=(2, 1, 3), black_border=True),
                ref(fn, solid, anisotropy=(2, 1, 3), black_border=True), ("solid", fn))


# ---- per-label views ------------------------------------------------------------------

def many_labels(shape, nlabels, seed, dtype=np.uint32):
  lab = voronoi_labels(shape, nlabels, seed, dtype)
  rng = np.random.default_rng(seed + 1)
  lab[rng.uniform(size=shape) < 0.1] = 0                      # some background
  # spread the label values out (the table hashes them)
  lut = np.concatenate([[0], rng.choice(np.arange(1, 10 ** 6), nlabels, replace=False)]).astype(dtype)
  return np.asfortranarray(lut[lab])


@pytest.mark.parametrize("order", ["F", "C"])
def test_each_against_reference_each(edt, reference, order):
  lab = many_labels((64, 60, 56), 320, 11)
  if order == "C":
    lab = np.ascontiguousarray(lab)
  dt = edt.edt(lab, anisotropy=(1, 2, 1.5), black_border=True)
  want = {}
  if reference is not None:
    for key, img in reference.each(lab, dt, in_place=False):
      want[int(key)] = img
  else:
    for key in np.unique(lab):
      if key != 0:
        want[int(key)] = np.where(lab == key, dt, np.float32(0))
  assert len(want) >= 300
  it = edt.each(lab, dt, in_place=False)
  assert len(it) == len(want)
  seen = []
  for key, img in it:
    assert img.dtype == np.float32 and img.shape == lab.shape
    assert img.flags.f_contiguous if order == "F" else img.flags.c_contiguous
    assert np.array_equal(img, want[int(key)]), key
    seen.append(int(key))
  assert seen == sorted(want)
  # in_place: one image reused, read-only while it is out
  count = 0
  for key, img in edt.each(lab, dt, in_place=True):
    assert not img.flags.writeable
    assert np.array_equal(img, want[int(key)]), key
    count += 1
  assert count == len(want)


def test_label_stats_and_each_cuda(edt):
  import torch
  lab_np = np.ascontiguousarray(many_labels((40, 72, 65), 310, 13, np.int64))
  lab_np[lab_np == lab_np.max()] = -5                           # a negative label: compared as raw bits
  lab = torch.from_numpy(lab_np).cuda()
  dt = edt.edt_cuda(lab, (2.0, 1.0, 1.0), False, sqrt=True)
  dt_np = dt.cpu().numpy()
  stats = edt.label_stats_cuda(lab, dt)
  keys = stats["labels"].cpu().numpy()
  uniq = np.unique(lab_np)
  uniq = uniq[uniq != 0]
  assert sorted(keys.tolist()) == sorted(uniq.tolist())
  flat_lab, flat_dt = lab_np.ravel(), dt_np.ravel()
  for k, cnt, mx, am, box in zip(keys.tolist(), stats["count"].tolist(), stats["max"].tolist(),
                                 stats["argmax"].tolist(), stats["box"].tolist()):
    where = np.flatnonzero(flat_lab == k)
    assert cnt == where.size
    assert np.float32(mx) == flat_dt[where].max()
    assert am == where[np.argmax(flat_dt[where])]               # first index of the maximum
    idx = np.argwhere(lab_np == k)
    assert box[:3] == idx.min(0).tolist() and box[3:] == idx.max(0).tolist()
  n = 0
  for key, img in edt.each_cuda(lab, dt):
    assert torch.equal(img, torch.where(lab == key, dt, torch.zeros((), device=dt.device)))
    n += 1
  assert n == len(uniq)
  prev = None
  for key, img in edt.each_cuda(lab, dt, in_place=True):
    assert prev is None or img is prev
    assert torch.equal(img, torch.where(lab == key, dt, torch.zeros((), device=dt.device)))
    prev = img


def test_device_graph_path_treats_negative_floats_as_background(edt):
  """With a voxel graph, float labels mean foreground iff value > 0 (src/edt_voxel_graph.hpp:76,
  151) -- on the device path as on the host path (negative values and NaN are background)."""
  import torch
  rng = np.random.default_rng(21)
  lab = rng.choice(np.array([-2.5, -0.0, 0.0, 1.0, 3.5, np.nan], dtype=np.float32), size=(12, 17, 9))
  graph = rng.integers(0, 64, lab.shape).astype(np.uint8)
  host = edt.edtsq(lab, anisotropy=(1, 2, 1), black_border=True, voxel_graph=graph)
  dev = edt.edtsq(torch.from_numpy(lab).cuda(), anisotropy=(1, 2, 1), black_border=True,
                  voxel_graph=torch.from_numpy(graph).cuda())
  assert np.array_equal(dev.cpu().numpy(), host)
  assert np.all(host[~(lab > 0)] == 0)
