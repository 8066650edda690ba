"""CPU tests (no GPU): pin the oracle.

The oracle (oracle/edt_oracle.c) is only trusted because it reproduces
  (a) the reference's own golden vectors (tests/cases.py, restated from automated_test.py),
  (b) the committed fixtures produced by the compiled reference (tests/golden/),
  (c) digests of the compiled reference's outputs on a few hundred more seeded cases (tests/golden/),
  (d) a brute-force evaluation of the definition on tiny volumes.
All comparisons are exact (bit-for-bit), as in the reference's tests.
"""
import json
import os

import numpy as np
import pytest

import cases

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_vectors.npz")
DIGESTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")


def same(a, b):
  return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


@pytest.mark.parametrize("case", cases.KNOWN_ANSWERS, ids=[c[0] for c in cases.KNOWN_ANSWERS])
def test_known_answers(oracle, case):
  for dtype in case[4]:
    labels, kwargs, expected = cases.known_answer_arrays(case, dtype)
    got = oracle.edtsq(labels, **kwargs)
    assert same(got, expected), (case[0], dtype, got)


def test_empty_and_bad_dims(oracle):
  assert oracle.edtsq(np.zeros((0,), np.uint8)).shape == (0,)
  assert oracle.edtsq(np.zeros((1, 0), np.uint8)).shape == (1, 0)
  with pytest.raises(TypeError):
    oracle.edtsq(np.zeros((2, 2, 2, 2), np.uint8))


def test_golden_fixtures(oracle):
  z = np.load(GOLDEN)
  for seed in z["seeds"]:
    key = "s%d" % seed
    labels = z[key + "_labels"]
    an = z[key + "_aniso"]
    an = float(an[0]) if labels.ndim == 1 else tuple(an)
    bb = bool(z[key + "_border"])
    assert same(oracle.edtsq(labels, anisotropy=an, black_border=bb), z[key + "_edtsq"]), seed
    assert same(oracle.edt(labels, anisotropy=an, black_border=bb), z[key + "_edt"]), seed
    assert same(oracle.sdf(labels, anisotropy=an, black_border=bb), z[key + "_sdf"]), seed
  cfg1 = np.ones((64, 64, 64), dtype=np.uint32, order="F")
  got = oracle.edtsq(cfg1, black_border=True)
  assert same(got, z["cfg1_edtsq"])
  assert got.max() == 1024.0


def test_golden_voxel_graph_fixtures(oracle):
  """The voxel_graph restatement (oracle.voxel_graph_edtsq) against the compiled reference's
  outputs for edtsq / edt / sdf under a connectivity graph (edt.pyx:514-620, 736-844)."""
  z = np.load(GOLDEN)
  for seed in z["graph_seeds"]:
    key = "g%d" % seed
    labels, graph = z[key + "_labels"], z[key + "_graph"]
    kw = dict(anisotropy=tuple(z[key + "_aniso"]), black_border=bool(z[key + "_border"]), voxel_graph=graph)
    with np.errstate(invalid="ignore"):
      assert same(oracle.edtsq(labels, **kw), z[key + "_edtsq"]), seed
      assert same(oracle.edt(labels, **kw), z[key + "_edt"]), seed
      assert same(oracle.sdf(labels, **kw), z[key + "_sdf"]), seed
    l2, g2, k2 = cases.random_graph_case(int(seed))
    assert np.array_equal(l2, labels) and np.array_equal(g2, graph)


def test_voxel_graph_known_answer(oracle):
  """The reference's own voxel-graph test, automated_test.py:736-789 (its first two asserts; the
  third one there is vacuous, so the blocked-edge geometry is pinned by the fixtures instead)."""
  labels = np.ones((5, 6), dtype=np.int64)
  graph = np.full((5, 6), 0b111111, dtype=np.uint8)
  assert np.all(oracle.edt(labels, voxel_graph=graph) == np.inf)
  ring = np.array([[0.5] * 6, [0.5, 1.5, 1.5, 1.5, 1.5, 0.5], [0.5, 1.5, 2.5, 2.5, 1.5, 0.5],
                   [0.5, 1.5, 1.5, 1.5, 1.5, 0.5], [0.5] * 6], dtype=np.float32)
  assert same(oracle.edt(labels, voxel_graph=graph, black_border=True), ring)
  # forbid the step between the two centre voxels of row 2: both end up half a voxel from background
  graph[2, 2] = 0b111110
  got = oracle.edt(labels, voxel_graph=graph, black_border=True)
  assert got[2, 2] == 0.5 and got[2, 1] == 1.5 and got[1, 2] == np.float32(np.sqrt(1.25))
  with pytest.raises(TypeError):
    oracle.edtsq(np.ones(5, np.uint8), voxel_graph=np.ones(5, np.uint8))


def test_fixture_cases_are_reproducible():
  """The generator is deterministic: the committed inputs equal cases.random_case(seed)."""
  z = np.load(GOLDEN)
  for seed in z["seeds"][:8]:
    labels, kwargs = cases.random_case(int(seed))
    assert np.array_equal(labels, z["s%d_labels" % seed])
    assert labels.flags.f_contiguous == z["s%d_labels" % seed].flags.f_contiguous


def test_live_against_compiled_reference(oracle):
  """The oracle against the compiled reference's outputs on 300 random and 60 voxel-graph cases,
  stored as digests (bit-exact, see cases.digest) by make_golden.py."""
  with open(DIGESTS) as fh:
    want = json.load(fh)
  for seed in cases.DIGEST_SEEDS:
    labels, kwargs = cases.random_case(seed)
    ref = want["random_case"][str(seed)]
    assert cases.digest(oracle.edtsq(labels, **kwargs)) == ref["edtsq"], seed
    if seed % 3 == 0:
      assert cases.digest(oracle.sdf(labels, **kwargs)) == ref["sdf"], seed
      assert cases.digest(oracle.edt(labels, **kwargs)) == ref["edt"], seed
  for seed in cases.DIGEST_GRAPH_SEEDS:
    labels, graph, kwargs = cases.random_graph_case(seed)
    ref = want["random_graph_case"][str(seed)]
    with np.errstate(invalid="ignore"):
      assert cases.digest(oracle.edtsq(labels, voxel_graph=graph, **kwargs)) == ref["edtsq"], seed
      assert cases.digest(oracle.sdf(labels, voxel_graph=graph, **kwargs)) == ref["sdf"], seed


def test_definition_bruteforce(oracle):
  rng = np.random.default_rng(7)
  for trial in range(40):
    nd = 1 + trial % 3
    shape = tuple(int(rng.integers(1, 9)) for _ in range(nd))
    kind = ["few", "blocks", "sparse_zero", "iid"][trial % 4]
    labels = cases.random_volume(rng, shape, kind, np.uint16)
    an = cases.INTEGER_ANISOTROPIES[trial % 4][:nd]
    an = an[0] if nd == 1 else an
    for bb in (False, True):
      got = oracle.edtsq(labels, anisotropy=an, black_border=bb)
      want = oracle.bruteforce_edtsq(labels, anisotropy=an, black_border=bb)
      assert same(got, want), (trial, shape, kind, an, bb)


def test_multilabel_equals_masked_binary(oracle):
  """README.md:195-199 of the reference: one multi-label transform equals the per-label
  binary transforms masked together."""
  rng = np.random.default_rng(3)
  labels = cases.random_volume(rng, (20, 17, 13), "blocks", np.uint32)
  multi = oracle.edtsq(labels, anisotropy=(1, 2, 3), black_border=True)
  acc = np.zeros_like(multi)
  for lab in np.unique(labels):
    if lab == 0:
      continue
    mask = labels == lab
    acc += oracle.edtsq(mask, anisotropy=(1, 2, 3), black_border=True) * mask
  assert same(multi, acc)


def test_order_and_scaling_invariance(oracle):
  rng = np.random.default_rng(5)
  labels = cases.random_volume(rng, (15, 22, 9), "blocks", np.uint8)
  c = oracle.edtsq(np.ascontiguousarray(labels), anisotropy=(2, 3, 5))
  f = oracle.edtsq(np.asfortranarray(labels), anisotropy=(2, 3, 5))
  assert same(c, f)
  base = oracle.edtsq(labels != 0)
  for w in (2.0, 7.0, 149.0):   # squared form of automated_test.py:641-649 (exact for integers)
    assert same(np.float32(w * w) * base, oracle.edtsq(labels != 0, anisotropy=(w, w, w)))
  box = np.zeros((15, 15, 15), dtype=bool, order="F")   # automated_test.py:641-649 verbatim geometry
  box[2:12, 2:12, 5:10] = True
  img = oracle.edt(box, anisotropy=(1, 1, 1))
  for w in (3.0, 50.0, 149.0):
    assert same(np.float32(w) * img, oracle.edt(box, anisotropy=(w, w, w)))
