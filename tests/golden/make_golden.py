"""Generate the fixtures under tests/golden/ by running the UNMODIFIED compiled reference
(oracle/_ref, built by oracle/Makefile from the reference's sources) on seeded inputs.

Run where the reference's sources are available:  python tests/golden/make_golden.py
The fixtures are committed, so the tests only read them and never need the reference.

reference_vectors.npz: each case stores the input labels, the call arguments and the reference's
edtsq / edt / sdf; the g* cases do the same for the voxel_graph= path.

reference_digests.json: digests (cases.digest) of the reference's outputs on inputs the tests
regenerate from their seeds: cases.DIGEST_SEEDS, cases.DIGEST_GRAPH_SEEDS and the whole 512^3
headline volume of BASELINE.json configs[1] (cases.cfg2_volume).
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import cases  # noqa: E402
from oracle import oracle  # noqa: E402

SEEDS = list(range(1000, 1048))
GRAPH_SEEDS = list(range(0, 36))


def main():
  ref = oracle.load_reference()
  if ref is None:
    raise SystemExit("oracle/_ref is not built: run `make -C oracle ref REF=<the reference's checkout>`")
  blob = {}
  meta = []
  for seed in SEEDS:
    labels, kwargs = cases.random_case(seed)
    an = kwargs["anisotropy"]
    key = "s%d" % seed
    blob[key + "_labels"] = labels
    blob[key + "_aniso"] = np.atleast_1d(np.asarray(an, dtype=np.float64))
    blob[key + "_border"] = np.array(kwargs["black_border"])
    blob[key + "_edtsq"] = ref.edtsq(labels, **kwargs)
    blob[key + "_edt"] = ref.edt(labels, **kwargs)
    blob[key + "_sdf"] = ref.sdf(labels, **kwargs)
    meta.append(seed)
  # the reference's own headline small config: 64^3 uint32 ones, F order, black border
  cfg1 = np.ones((64, 64, 64), dtype=np.uint32, order="F")
  blob["cfg1_edtsq"] = ref.edtsq(cfg1, black_border=True, parallel=1)
  blob["seeds"] = np.array(meta)
  # voxel_graph path (edt.pyx:514-620, 736-844): edtsq / edt / sdf under a connectivity graph
  for seed in GRAPH_SEEDS:
    labels, graph, kwargs = cases.random_graph_case(seed)
    key = "g%d" % seed
    blob[key + "_labels"] = labels
    blob[key + "_graph"] = graph
    blob[key + "_aniso"] = np.asarray(kwargs["anisotropy"], dtype=np.float64)
    blob[key + "_border"] = np.array(kwargs["black_border"])
    with np.errstate(invalid="ignore"):
      blob[key + "_edtsq"] = ref.edtsq(labels, voxel_graph=graph, **kwargs)
      blob[key + "_edt"] = ref.edt(labels, voxel_graph=graph, **kwargs)
      blob[key + "_sdf"] = ref.sdf(labels, voxel_graph=graph, **kwargs)
  blob["graph_seeds"] = np.array(GRAPH_SEEDS)
  out = os.path.join(HERE, "reference_vectors.npz")
  np.savez_compressed(out, **blob)
  print("wrote", out, os.path.getsize(out), "bytes,", len(meta), "cases")
  write_digests(ref)


def write_digests(ref):
  random_case = {}
  for seed in cases.DIGEST_SEEDS:
    labels, kwargs = cases.random_case(seed)
    entry = {"edtsq": cases.digest(ref.edtsq(labels, **kwargs))}
    if seed % 3 == 0:
      entry["sdf"] = cases.digest(ref.sdf(labels, **kwargs))
      entry["edt"] = cases.digest(ref.edt(labels, **kwargs))
    random_case[str(seed)] = entry
  graph_case = {}
  for seed in cases.DIGEST_GRAPH_SEEDS:
    labels, graph, kwargs = cases.random_graph_case(seed)
    with np.errstate(invalid="ignore"):
      graph_case[str(seed)] = {"edtsq": cases.digest(ref.edtsq(labels, voxel_graph=graph, **kwargs)),
                               "sdf": cases.digest(ref.sdf(labels, voxel_graph=graph, **kwargs))}
  want = ref.edtsq(cases.cfg2_volume(), anisotropy=(1, 1, 1), black_border=False, parallel=os.cpu_count() or 1)
  blob = {"random_case": random_case, "random_graph_case": graph_case, "cfg2_512": {"edtsq": cases.digest(want)}}
  out = os.path.join(HERE, "reference_digests.json")
  with open(out, "w") as fh:
    json.dump(blob, fh, indent=0, sort_keys=True)
    fh.write("\n")
  print("wrote", out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
  main()
