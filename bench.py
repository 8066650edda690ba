#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native multi-label EDT.

Metric (BASELINE.json): Mvoxels/s of edtsq on a 512^3 uint32 multi-label volume
(configs[1]: iid random labels 0..255, anisotropy (1,1,1)), plus the HBM roofline fraction of
the dominant kernel, plus the same metric end to end from host memory, plus the reference's
own CPU implementation timed on this box's host cores.

  python bench.py --gpus 1 --steps 20 --warmup 3          # our arm
  python bench.py --impl reference --steps 2 --warmup 1   # the unmodified reference (CPU)
  python bench.py --dump-outputs DIR ...                  # also save a sample of the result (float32 .npy)
  torchrun ... bench.py --gpus N ...                      # one rank per GPU, weak scaling:
                                                          # each rank owns one 512^3 Z slab

One JSON line on stdout (rank 0).  A "step" is one full transform (X, Y, Z passes) of the
volume.  Inputs (512 MiB labels + 512 MiB distances) are larger than the 126 MB L2, so no L2
flush is needed between steps.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
  os.environ["NCCL_DEBUG"] = "WARN"              # keep NCCL's version banner off stdout (one JSON line only)

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

SHAPE = (512, 512, 512)          # x, y, z (x fastest)
ANISOTROPY = (1.0, 1.0, 1.0)
LABEL_BYTES = 4
WORKLOAD = "edtsq 512x512x512 uint32 iid-random labels 0..255, anisotropy (1,1,1), black_border=False (BASELINE.json configs[1])"


def make_labels(seed=0, shape=SHAPE):
  """cfg2 of BASELINE.md section 3: np.asfortranarray(rng(0).integers(0,256,(512,)*3, uint32))."""
  rng = np.random.default_rng(seed)
  return np.asfortranarray(rng.integers(0, 256, shape, dtype=np.uint32))


def measured_peak_gbs():
  path = os.path.join(ROOT, "MEASURED_PEAKS.json")
  try:
    with open(path) as fh:
      return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
  except Exception:
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
  """DRAM bytes per launch of the dominant kernel from the committed ncu summary, if any."""
  path = os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")
  try:
    with open(path) as fh:
      return json.load(fh)
  except Exception:
    return None


class ClockSampler:
  """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
  QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
           "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
           "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

  def __init__(self, gpu_index):
    self.gpu_index = gpu_index
    self.lines = []
    self.proc = None
    self.thread = None

  def start(self):
    try:
      self.proc = subprocess.Popen(
        ["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.QUERY,
         "--format=csv,noheader,nounits", "-lms", "200"],
        stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except Exception:
      self.proc = None
      return
    def pump():
      for line in self.proc.stdout:
        self.lines.append(line.strip())
    self.thread = threading.Thread(target=pump, daemon=True)
    self.thread.start()

  def stop(self):
    if self.proc is None:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    time.sleep(0.25)
    self.proc.terminate()
    try:
      self.proc.wait(timeout=5)
    except Exception:
      self.proc.kill()
    sm, smax, reasons = [], [], set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for line in self.lines:
      parts = [p.strip() for p in line.split(",")]
      if len(parts) < 9:
        continue
      try:
        sm.append(float(parts[1])); smax.append(float(parts[2]))
      except ValueError:
        continue
      for name, val in zip(names, parts[5:9]):
        if val.lower().startswith("active"):
          reasons.add(name)
    return {"sm_mhz": statistics.median(sm) if sm else None,
            "sm_max_mhz": max(smax) if smax else None,
            "samples": len(sm), "reasons": sorted(reasons)}


def host_description():
  """CPU model / sockets / cores of this box, the affinity of this process and the load average:
  what the CPU arm's number depends on (SURVEY.md section 8d asks for them beside it)."""
  info = {"cpu_count": os.cpu_count()}
  try:
    info["affinity"] = len(os.sched_getaffinity(0))
  except Exception:
    pass
  try:
    out = subprocess.run(["lscpu"], capture_output=True, text=True, timeout=10).stdout
    for line in out.splitlines():
      key, _, val = line.partition(":")
      key = key.strip()
      if key in ("Model name", "Socket(s)", "Core(s) per socket", "Thread(s) per core", "NUMA node(s)"):
        info[key.lower().replace("(s)", "s").replace(" ", "_")] = val.strip()
  except Exception:
    pass
  try:
    info["loadavg_1m"] = os.getloadavg()[0]
  except Exception:
    pass
  return info


def bind_to_gpu_numa(local):
  """Run this rank on the CPUs of the NUMA node its GPU hangs off, so that the pinned host buffers of
  the end-to-end leg are allocated next to the GPU's PCIe root (SURVEY.md section 8d: 'pin with taskset
  if NUMA').  Returns a description for the JSON line; does nothing when sysfs does not tell."""
  try:
    import torch
    prop = torch.cuda.get_device_properties(local)
    bdf = "%04x:%02x:%02x.0" % (prop.pci_domain_id, prop.pci_bus_id, prop.pci_device_id)
    with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as fh:
      node = int(fh.read().strip())
    if node < 0:
      return {"gpu_pci": bdf, "numa_node": node, "bound": False}
    with open("/sys/devices/system/node/node%d/cpulist" % node) as fh:
      cpus = set()
      for part in fh.read().strip().split(","):
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    os.sched_setaffinity(0, cpus)
    return {"gpu_pci": bdf, "numa_node": node, "bound": True, "cpus": len(cpus)}
  except Exception as exc:
    return {"bound": False, "why": repr(exc)}


def dist_env():
  rank = int(os.environ.get("RANK", "0"))
  world = int(os.environ.get("WORLD_SIZE", "1"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  return rank, world, local


# ---------------------------------------------------------------------------------------
# reference arm: the unmodified reference (oracle/_ref) on the host cores
# ---------------------------------------------------------------------------------------

def reference_arm(args):
  rank, world, _ = dist_env()
  if rank != 0:
    return
  from oracle import oracle
  ref = oracle.load_reference()
  kind = "reference"
  if ref is None:                      # cannot happen where oracle/_ref was built; keep the arm alive
    ref, kind = oracle, "port"
  cores = os.cpu_count() or 1
  labels = make_labels()
  # bounded sample: a full-x/y Z slab of the workload, deep enough for ~<=8 s per step
  probe = np.asfortranarray(labels[:, :, :32])
  t0 = time.perf_counter()
  ref.edtsq(probe, anisotropy=ANISOTROPY, black_border=False, parallel=cores)
  rate = probe.size / (time.perf_counter() - t0)            # voxels/s
  budget_s = max(1.0, min(8.0, 150.0 / max(1, args.steps + args.warmup)))
  depth = int(min(SHAPE[2], max(32, (rate * budget_s) // (SHAPE[0] * SHAPE[1]) // 32 * 32)))
  sample = np.asfortranarray(labels[:, :, :depth])
  for _ in range(args.warmup):
    ref.edtsq(sample, anisotropy=ANISOTROPY, black_border=False, parallel=cores)
  step_s = []
  t0 = time.perf_counter()
  for _ in range(args.steps):
    t1 = time.perf_counter()
    ref.edtsq(sample, anisotropy=ANISOTROPY, black_border=False, parallel=cores)
    step_s.append(time.perf_counter() - t1)
  dt = time.perf_counter() - t0
  mvox = sample.size * args.steps / dt / 1e6
  sample_desc = "512x512x%d Z slab of the workload per step, parallel=%d threads" % (depth, cores)
  line = {
    "impl": "reference", "metric": "Mvoxels/s edtsq 512^3 uint32", "value": mvox, "unit": "Mvoxels/s",
    "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
    "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
    "vs_baseline": None, "dtype": "f32 (f64 envelope internals)", "data": "synthetic",
    "config": {"workload": WORKLOAD, "sample": sample_desc},
    "cpu_baseline": {"value": mvox, "unit": "Mvoxels/s", "cores": cores, "kind": kind, "sample": sample_desc,
                     "best_step_value": sample.size / min(step_s) / 1e6,
                     "threads": "the reference's own thread pool, parallel=%d, not pinned (the reference has no "
                                "affinity control); the box's load and NUMA placement move this number between "
                                "boxes, see `host`" % cores,
                     "host": host_description()},
    "e2e": {"value": mvox, "unit": "Mvoxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    "gpu_launches": 0,
  }
  print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------

def cpu_baseline_leg():
  """The reference's CPU path on this box's host cores, on a bounded sample (rank 0, N=1)."""
  from oracle import oracle
  ref = oracle.load_reference()
  kind = "reference"
  if ref is None:
    ref, kind = oracle, "port"
  cores = (os.cpu_count() or 1) if kind == "reference" else 1
  labels = make_labels()
  probe = np.asfortranarray(labels[:, :, :32])
  t0 = time.perf_counter()
  ref.edtsq(probe, anisotropy=ANISOTROPY, black_border=False, parallel=cores)
  rate = probe.size / (time.perf_counter() - t0)
  depth = int(min(SHAPE[2], max(32, (rate * 15.0) // (SHAPE[0] * SHAPE[1]) // 32 * 32)))
  depth = max(32, depth // 3 // 32 * 32)              # three repetitions share the ~15 s budget
  sample = np.asfortranarray(labels[:, :, :depth])
  times = []
  for _ in range(3):
    t0 = time.perf_counter()
    ref.edtsq(sample, anisotropy=ANISOTROPY, black_border=False, parallel=cores)
    times.append(time.perf_counter() - t0)
  dt = min(times)
  out = {"value": sample.size / dt / 1e6, "unit": "Mvoxels/s", "cores": cores, "kind": kind,
         "sample": "best of 3 edtsq calls on a 512x512x%d Z slab of the workload (%.1f s each), parallel=%d, "
                   "threads not pinned" % (depth, dt, cores),
         "all_runs_s": times, "host": host_description()}
  if cores > 1:
    # the same code on ONE thread (SURVEY.md section 8d asks for both), on a thinner slab
    thin = np.asfortranarray(labels[:, :, :max(32, depth // 8)])
    t0 = time.perf_counter()
    ref.edtsq(thin, anisotropy=ANISOTROPY, black_border=False, parallel=1)
    dt1 = time.perf_counter() - t0
    out["single_thread"] = {"value": thin.size / dt1 / 1e6, "unit": "Mvoxels/s",
                            "sample": "512x512x%d slab (%.1f s), parallel=1" % (thin.shape[2], dt1)}
  return out


def rows_changed(lab, an, bb, sqrt=False):
  """Voxels whose value the Y and the Z pass change (anisotropy as edt_cuda takes it: (w_z, w_y, w_x)).
  The later passes work in place and do not store rows that keep their value, so the bytes a pass
  HAS to move are: labels read + distances read + 4 bytes per voxel that changes."""
  import torch
  from edt_b200.distributed import CudaPasses
  passes = CudaPasses(lab.device)
  f = torch.empty(lab.shape, dtype=torch.float32, device=lab.device)
  passes.pass_first(lab, f, an[2], bb, False)
  before = f.clone()
  passes.pass_later(lab, f, 1, an[1], bb, bb)
  cy = int((f != before).sum().item())
  before.copy_(f)
  passes.pass_later(lab, f, 2, an[0], bb, bb, sqrt=sqrt, negate=False)
  cz = int((f != before).sum().item())
  del before, f
  return cy, cz


def workload_matrix(dev, peak, steps=5):
  """Device-resident transform times of the structured workloads of SURVEY.md section 8d (the
  headline workload has run length ~1 and never runs the envelope scan; these do)."""
  import torch
  import edt_b200
  from edt_b200 import workloads
  rows = []
  n = SHAPE[0]
  for name, sqrt in (("cfg2", False), ("cfg2b", False), ("cfg3", False), ("cfg3", True), ("balls", False),
                     ("voronoi", False)):
    lab, an, bb = workloads.generate(name, n, dev)
    out = torch.empty(lab.shape, dtype=torch.float32, device=dev)
    for _ in range(3):
      edt_b200.edt_cuda(lab, an, bb, sqrt=sqrt, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
      edt_b200.edt_cuda(lab, an, bb, sqrt=sqrt, out=out)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    L = lab.element_size()
    cy, cz = rows_changed(lab, an, bb, sqrt)
    alg = (3 * L + 12) * lab.numel() + 4 * (cy + cz)       # see rows_changed; (3 L + 20) N if every row changed
    rows.append({"workload": name, "function": "edt" if sqrt else "edtsq", "shape": [n, n, n], "label_bytes": L,
                 "anisotropy": list(an), "black_border": bb, "ms": ms, "Mvoxels_s": lab.numel() / ms / 1e3,
                 "rows_changed": {"y": cy / lab.numel(), "z": cz / lab.numel()},
                 "algorithmic_GBps": alg / ms / 1e6, "frac": alg / ms / 1e6 / peak})
    del lab, out
    torch.cuda.empty_cache()
  return rows


def pageable_e2e(labels_np, steps=3):
  """edt_b200.edtsq(ndarray): the drop-in call with a plain (pageable) numpy array in and out."""
  import edt_b200
  edt_b200.edtsq(labels_np, anisotropy=ANISOTROPY, black_border=False)
  times = []
  for _ in range(steps):
    t0 = time.perf_counter()
    res = edt_b200.edtsq(labels_np, anisotropy=ANISOTROPY, black_border=False)
    times.append(time.perf_counter() - t0)
  best = min(times)
  return {"value": labels_np.size / best / 1e6, "unit": "Mvoxels/s", "ms_per_call": best * 1e3,
          "all_calls_ms": [t * 1e3 for t in times],
          "note": "edt_b200.edtsq(numpy array), pageable memory both ways (staged through pinned buffers by "
                  "the library's copy threads), best of %d" % steps}, res


def slab_parity_check(dev, rank, world, passes, peer_halo_factory):
  """Before anything is timed at N > 1: a structured 512 x 512 x (64*world) volume (32^3 blocks of
  labels with background) is transformed by the slab-split path (edtsq and sdf) and every rank
  compares ITS slab with the same rows of the single-GPU transform of the whole volume."""
  import torch
  import torch.distributed as dist
  import edt_b200
  import edt_b200.distributed as ed
  from edt_b200 import workloads
  depth = 64
  lab, _, _ = workloads.generate("cfg2b", SHAPE[0], dev, nz=depth * world)      # same seed on every rank
  lab = (lab % 7).to(torch.int32)                                               # label 0 = background
  mine = lab[rank * depth:(rank + 1) * depth].contiguous()
  an_zyx = (2.0, 1.0, 1.0)
  ok = True
  for signed, sqrt in ((False, False), (True, True)):
    whole = edt_b200.edt_cuda(lab, an_zyx, False, sqrt=sqrt, signed=signed)
    got = ed.slab_transform(mine, an_zyx, False, sqrt=sqrt, signed=signed, passes=passes,
                            depths=[depth] * world, peer_halo=peer_halo_factory(depth))
    ok = ok and bool(torch.equal(got, whole[rank * depth:(rank + 1) * depth]))
  flag = torch.tensor([1 if ok else 0], device=dev)
  dist.all_reduce(flag, op=dist.ReduceOp.MIN)
  return bool(flag.item())


DUMP_VOXELS = 1 << 23            # 32 MiB of float32 over all ranks


def dump_outputs(path, out, rank, world):
  """Write a fixed, seeded sample of this rank's edtsq result (the distances a caller of the timed
  path receives) as float32 to path/edtsq.npy (path/edtsq_rank<r>.npy with several ranks), so that
  two builds run with the same arguments can be compared output for output."""
  import torch
  idx = np.random.default_rng(12345 + rank).integers(0, out.numel(), DUMP_VOXELS // world)
  idx.sort()
  sample = out.reshape(-1)[torch.from_numpy(idx).to(out.device)].cpu().numpy().astype(np.float32)
  os.makedirs(path, exist_ok=True)
  np.save(os.path.join(path, "edtsq.npy" if world == 1 else "edtsq_rank%d.npy" % rank), sample)


def ours(args):
  import torch
  import torch.distributed as dist
  import edt_b200

  rank, world, local = dist_env()
  numa = bind_to_gpu_numa(local) if world > 1 else None      # ranks share the host: each next to its GPU
  if world > 1:
    # high-priority NCCL stream: lets the halo exchange run beside the SM-filling Z-pass kernel
    opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local), pg_options=opts)
  torch.cuda.set_device(local)
  dev = torch.device("cuda", local)
  lib = edt_b200._lib()
  sx, sy, sz = SHAPE
  nvox = sx * sy * sz

  # every rank owns one 512^3 slab (weak scaling); distinct seeds so ranks do different work
  labels_np = make_labels(seed=rank)
  labels_host = torch.from_numpy(np.ascontiguousarray(labels_np.T)).pin_memory()   # memory: x fastest
  out_host = torch.empty(labels_host.shape, dtype=torch.float32).pin_memory()
  labels_dev = labels_host.to(dev, non_blocking=True)
  f_dev = torch.empty(labels_host.shape, dtype=torch.float32, device=dev)
  torch.cuda.synchronize()

  stream = torch.cuda.current_stream(dev)
  sptr = ctypes.c_void_p(stream.cuda_stream)
  lp, fp = labels_dev.data_ptr(), f_dev.data_ptr()

  def check(rc):
    if rc != 0:
      raise RuntimeError(lib.edtb200_last_error().decode())

  DEV_FLAGS = 4 | 8            # EDTB200_LABELS_ON_DEVICE | EDTB200_OUT_ON_DEVICE

  def step(events=None):
    # one full transform through the public C-ABI entry point, device-resident, asynchronous
    check(lib.edtb200_transform(lp, LABEL_BYTES, 3, sx, sy, sz, *ANISOTROPY, 0, DEV_FLAGS, fp, local, sptr))

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  if world > 1:
    # weak scaling: the ranks' 512^3 slabs form ONE 512 x 512 x (512*world) volume (axis 0 = z),
    # transformed by the slab-split path (X/Y local, Z through the NVLink exchange)
    import edt_b200.distributed as ed
    passes = ed.CudaPasses(dev)
    result = {}
    peer_halo, peer_why = ed.make_peer_halo(dev, sy, sx, torch.int32, ed.DEFAULT_HALO)
    ok = torch.tensor([1 if peer_halo is not None else 0], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)            # all ranks or none
    if int(ok.item()) == 0:
      peer_halo = None
    def halo_for(depth):
      # the parity volume has thinner slabs than the timed one: its own staging buffer
      ph, _ = ed.make_peer_halo(dev, sy, sx, torch.int32, ed.DEFAULT_HALO)
      okp = torch.tensor([1 if ph is not None else 0], device=dev)
      dist.all_reduce(okp, op=dist.ReduceOp.MIN)
      return ph if int(okp.item()) == 1 else None
    parity_checked = slab_parity_check(dev, rank, world, passes, halo_for)
    verdicts = []
    def step(events=None):
      # the halo path's exactness verdict is a device flag; it is read for all steps at once,
      # inside the timed region, after the last step has been queued (no per-step host sync)
      result["out"] = ed.slab_transform(labels_dev, (ANISOTROPY[2], ANISOTROPY[1], ANISOTROPY[0]), False,
                                        passes=passes, info=result, depths=[sz] * world, peer_halo=peer_halo,
                                        defer_check="local" if peer_halo is not None else True)
      if "verdict" in result:
        verdicts.append(result.pop("verdict"))

  for _ in range(max(3, args.warmup)):
    step()
  if world > 1:
    ed.check_verdicts(verdicts)          # also warms the one collective the timed region contains
    del verdicts[:]
  barrier()

  sampler = ClockSampler(local)
  if rank == 0:
    sampler.start()
  evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.steps)]
  start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  barrier()
  start.record(stream)
  for k in range(args.steps):
    step(evs[k])
  if world > 1:
    clean = ed.check_verdicts(verdicts[-args.steps:])
    if not clean:
      raise RuntimeError("halo method was not exact for this workload; rerun with method=transpose")
  stop.record(stream)
  barrier()
  elapsed_ms = start.elapsed_time(stop)
  if args.dump_outputs:
    dump_outputs(args.dump_outputs, result["out"] if world > 1 else f_dev, rank, world)
  if True:
    # per-pass device times: the same K steps once more with the library recording CUDA events
    # around every pass (on the launch stream, no syncs).  Kept out of the timed region above
    # because an event between two passes keeps the next pass from starting under the previous
    # one's tail (programmatic dependent launch), i.e. it would time a slightly slower product.
    lib.edtb200_profile_passes(1)
    for k in range(args.steps):
      step()
    torch.cuda.synchronize()
    lib.edtb200_profile_passes(0)        # keeps the recorded events, stops recording
  # The timed region lasts a few milliseconds, shorter than one nvidia-smi sampling period, so
  # the same steps keep running (untimed) for ~0.7 s while the sampler is still on: the clock
  # record then describes the GPU under exactly this load.
  soak_until = time.perf_counter() + 0.7
  while time.perf_counter() < soak_until:
    for _ in range(20):
      step()
    torch.cuda.synchronize()
  verdicts_soak_ok = True
  if world > 1:
    verdicts_soak_ok = ed.check_verdicts(verdicts[-4:])
  clocks = sampler.stop() if rank == 0 else None
  if clocks is not None:
    clocks["note"] = "sampled every 200 ms over the timed region plus an identical 0.7 s untimed soak"

  t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  elapsed_ms = float(t.item())
  ms_per_step = elapsed_ms / args.steps
  value = nvox * world / (ms_per_step * 1e-3) / 1e6

  peak, peak_src = measured_peak_gbs()
  if world > 1:
    # whole step against HBM for orientation (bytes that have to move, see rows_changed; set below)
    # dominant kernel: the Z pass of this rank's slab, timed by the library's per-pass events over the
    # K steps that followed the timed region (rank 0's slab; every rank runs the same kernels)
    zms = None
    try:
      buf3 = (ctypes.c_float * 3)()
      zs = []
      for back in range(min(args.steps, 250)):
        check(lib.edtb200_pass_ms(back, ctypes.cast(buf3, ctypes.c_void_p)))
        zs.append(float(buf3[2]))
      zms = statistics.mean(zs) if zs else None
    except Exception:
      zms = None
    # labels + distances read + 4 B per voxel the pass changes (rows that keep their value are not stored)
    cy, cz = rows_changed(labels_dev, (ANISOTROPY[2], ANISOTROPY[1], ANISOTROPY[0]), False)
    zalg = (LABEL_BYTES + 4) * nvox + 4 * cz
    alg = 3 * (LABEL_BYTES + 4) * nvox + 4 * (cy + cz)
    traffic = ncu_traffic()
    roofline = {"bound": "hbm", "kernel": "later_axis_tile_kernel<4,32,false,true,false,2,true> (Z pass of one slab)",
                "achieved": (zalg / (zms * 1e-3) / 1e9) if zms else None, "peak": peak, "unit": "GB/s",
                "frac": (zalg / (zms * 1e-3) / 1e9 / peak) if zms else None, "peak_source": peak_src,
                "traffic": traffic.get("dram_bytes_per_launch") if traffic else None,
                "algorithmic_bytes_per_launch": zalg, "ms": zms,
                "whole_step": {"what": "X, Y, Z passes + %s, per rank" % (
                                   "face staging and fix-up reading the neighbours' faces over NVLink"
                                   if result.get("method") == "halo" else "Z-slab<->Y-slab transposes"),
                               "algorithmic_bytes": alg, "GBps": alg / (ms_per_step * 1e-3) / 1e9,
                               "frac": alg / (ms_per_step * 1e-3) / 1e9 / peak},
                "nvlink_bytes_per_gpu_per_step": (2 * 512 * 512 * (2 * 4 + LABEL_BYTES + 1)
                                                  if result.get("method") == "halo"
                                                  else int(nvox * (LABEL_BYTES + 8) * (world - 1) / world))}
    e2e_steps = max(2, min(args.steps, 5))
    hl_t, ho_t = labels_host, out_host
    def e2e_once():
      lab = hl_t.to(dev, non_blocking=True)
      res = ed.slab_transform(lab, (ANISOTROPY[2], ANISOTROPY[1], ANISOTROPY[0]), False, passes=passes,
                              depths=[sz] * world, peer_halo=peer_halo)
      ho_t.copy_(res, non_blocking=True)
      torch.cuda.synchronize()
    e2e_once()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
      e2e_once()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())
    e2e = {"value": nvox * world / e2e_s / 1e6, "unit": "Mvoxels/s", "ms_per_step": e2e_s * 1e3,
           "steps": e2e_steps, "h2d_bytes_per_step": nvox * LABEL_BYTES * world,
           "d2h_bytes_per_step": nvox * 4 * world, "host_memory": "pinned", "numa_binding_rank0": numa}
    # BASELINE configs[4] as written asks for sdf: the same slab step with the sign and sqrt fused, on the
    # iid slabs and on 32^3 blocks of labels (device-resident, CUDA events, max over ranks)
    cfg5 = []
    try:
      from edt_b200 import workloads
      blocks, _, _ = workloads.generate("cfg2b", sx, dev, nz=sz * world)
      blocks = blocks[rank * sz:(rank + 1) * sz].contiguous()
      # blocks of 32 need a halo that reaches 16 voxels: 32 rows (what method="auto" escalates to)
      halo32 = None
      if peer_halo is not None:
        halo32, _ = ed.make_peer_halo(dev, sy, sx, torch.int32, 32)
        ok32 = torch.tensor([1 if halo32 is not None else 0], device=dev)
        dist.all_reduce(ok32, op=dist.ReduceOp.MIN)
        if int(ok32.item()) == 0:
          halo32 = None
      for name, lab, ph in (("iid", labels_dev, peer_halo), ("blocks32", blocks, halo32)):
        info = {}
        vs = []
        def sdf_step():
          ed.slab_transform(lab, (ANISOTROPY[2], ANISOTROPY[1], ANISOTROPY[0]), False, sqrt=True, signed=True,
                            passes=passes, info=info, depths=[sz] * world, peer_halo=ph,
                            defer_check="local" if ph is not None else True)
          vs.append(info.pop("verdict"))
        for _ in range(3):
          sdf_step()
        ed.check_verdicts(vs)
        del vs[:]
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(10):
          sdf_step()
        e1.record(stream)
        exact = ed.check_verdicts(vs)
        barrier()
        tt = torch.tensor([e0.elapsed_time(e1) / 10], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        cfg5.append({"labels": name, "function": "sdf", "ms_per_step": float(tt.item()),
                     "Mvoxels_s": nvox * world / float(tt.item()) / 1e3, "halo_exact": bool(exact),
                     "method": info.get("method"), "halo_rows": ph.halo if ph is not None else None})
      del blocks
    except Exception as exc:
      cfg5 = {"error": repr(exc)}
    if rank == 0:
      line = {
        "metric": "Mvoxels/s edtsq 512^3 uint32", "value": value, "unit": "Mvoxels/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (u32 labels)", "data": "synthetic",
        "config": {"workload": "edtsq 512x512x%d uint32 iid-random labels 0..255, anisotropy (1,1,1), "
                               "Z-slab split, one 512^3 slab per GPU (BASELINE.json configs[4] geometry)" % (512 * world),
                   "parallelism": "z-slab x%d; X,Y passes local; Z pass local + face fix-up reading the neighbours' "
                                  "faces %s; method used: %s" % (
                                      world, "in place over NVLink (symmetric memory)" if peer_halo is not None
                                      else "received through NCCL send/recv (%s)" % peer_why, result.get("method")),
                   "l2": "inputs (1 GiB per rank per step) larger than L2; no flush needed",
                   "timing": "CUDA events on the launch stream, max over ranks"},
        "roofline": roofline, "e2e": e2e, "gpu_launches": (5 if result.get("method") == "halo" else 3) * args.steps,
        "clocks": clocks,
        "cfg5_sdf": cfg5,
        "parity_checked": parity_checked,
        "parity_check": "before timing: edtsq and sdf of a 512x512x%d volume of 32^3 label blocks (with background, "
                        "anisotropy 2 along z) through the slab split, every rank's slab bit-equal to the same rows "
                        "of the single-GPU transform" % (64 * world),
      }
      print(json.dumps(line), flush=True)
    dist.destroy_process_group()
    return

  # per-pass device times -> roofline of the dominant kernel (the library kept CUDA events around
  # every pass of the K steps that followed the timed region; they are only read now)
  samples = []
  buf3 = (ctypes.c_float * 3)()
  for back in range(min(args.steps, 250)):
    check(lib.edtb200_pass_ms(back, ctypes.cast(buf3, ctypes.c_void_p)))
    samples.append([float(buf3[0]), float(buf3[1]), float(buf3[2])])
  pass_ms = [statistics.mean(smp[i] for smp in samples) for i in range(3)]
  # bytes a pass has to move: labels + distances read (X: written), + 4 per voxel a later pass changes
  # (rows that keep their value are not stored: the later passes work in place)
  cy, cz = rows_changed(labels_dev, (ANISOTROPY[2], ANISOTROPY[1], ANISOTROPY[0]), False)
  alg_bytes = [(LABEL_BYTES + 4) * nvox, (LABEL_BYTES + 4) * nvox + 4 * cy, (LABEL_BYTES + 4) * nvox + 4 * cz]
  names = ["first_axis_vec_kernel<4,4,true,false> (X)", "later_axis_tile_kernel<4,32,false,true,false,2,true> (Y)",
           "later_axis_tile_kernel<4,32,false,true,false,2,true> (Z)"]
  dom = max(range(3), key=lambda i: pass_ms[i])
  achieved = alg_bytes[dom] / (pass_ms[dom] * 1e-3) / 1e9
  traffic = ncu_traffic()
  roofline = {
    "bound": "hbm", "kernel": names[dom], "achieved": achieved, "peak": peak, "unit": "GB/s",
    "frac": achieved / peak, "peak_source": peak_src,
    "traffic": traffic.get("dram_bytes_per_launch") if traffic else None,
    "algorithmic_bytes_per_launch": alg_bytes[dom],
    "algorithmic_bytes_note": "labels + distances read + 4 B per voxel whose value the pass changes (fractions: "
                              "Y %.4f, Z %.4f of the voxels on this workload); rows that keep their value are not "
                              "stored, the later passes work in place" % (cy / nvox, cz / nvox),
    "per_pass_source": "CUDA events around each pass of %d further identical steps run right after the "
                       "timed region (events between passes would serialise them inside it)" % min(args.steps, 250),
    "per_pass": [{"kernel": names[i], "ms": pass_ms[i], "algorithmic_bytes": alg_bytes[i],
                  "GBps": alg_bytes[i] / (pass_ms[i] * 1e-3) / 1e9,
                  "frac": alg_bytes[i] / (pass_ms[i] * 1e-3) / 1e9 / peak} for i in range(3)],
    "whole_transform": {"algorithmic_bytes": sum(alg_bytes), "GBps": sum(alg_bytes) / (ms_per_step * 1e-3) / 1e9,
                        "frac": sum(alg_bytes) / (ms_per_step * 1e-3) / 1e9 / peak},
  }

  # end to end through the public C-ABI call with HOST buffers (pinned): H2D + passes + D2H
  e2e_steps = max(2, min(args.steps, 10))
  hl, ho = labels_host.data_ptr(), out_host.data_ptr()
  for _ in range(2):
    check(lib.edtb200_transform(hl, LABEL_BYTES, 3, sx, sy, sz, *ANISOTROPY, 0, 0, ho, local, None))
  barrier()
  t0 = time.perf_counter()
  for _ in range(e2e_steps):
    check(lib.edtb200_transform(hl, LABEL_BYTES, 3, sx, sy, sz, *ANISOTROPY, 0, 0, ho, local, None))
  torch.cuda.synchronize()
  e2e_s = (time.perf_counter() - t0) / e2e_steps
  te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(te, op=dist.ReduceOp.MAX)
  e2e_s = float(te.item())
  e2e = {"value": nvox * world / e2e_s / 1e6, "unit": "Mvoxels/s", "ms_per_step": e2e_s * 1e3,
         "steps": e2e_steps, "h2d_bytes_per_step": nvox * LABEL_BYTES, "d2h_bytes_per_step": nvox * 4,
         "host_memory": "pinned"}

  # sanity: the device-resident result equals the host-path result
  same = bool(torch.equal(f_dev.cpu(), out_host))

  # the same call for a batch of volumes (edtb200_transform_batch): upload of volume k+1 and
  # download of volume k-1 overlap the passes of volume k.  Reported beside the single-call number,
  # never instead of it: the headline e2e.value is the one-volume synchronous call above.
  try:
    nb = 6
    out2 = torch.empty(labels_host.shape, dtype=torch.float32).pin_memory()
    lab_ptrs = (ctypes.c_void_p * nb)(*([hl] * nb))
    out_ptrs = (ctypes.c_void_p * nb)(*[(ho if k % 2 == 0 else out2.data_ptr()) for k in range(nb)])
    check(lib.edtb200_transform_batch(lab_ptrs, out_ptrs, 2, LABEL_BYTES, 3, sx, sy, sz, *ANISOTROPY, 0, 0, local))
    t0 = time.perf_counter()
    check(lib.edtb200_transform_batch(lab_ptrs, out_ptrs, nb, LABEL_BYTES, 3, sx, sy, sz, *ANISOTROPY, 0, 0, local))
    batch_s = (time.perf_counter() - t0) / nb
    e2e["batch_pipelined"] = {"value": nvox / batch_s / 1e6, "unit": "Mvoxels/s", "ms_per_volume": batch_s * 1e3,
                              "volumes": nb, "equals_single_call": bool(torch.equal(out2, out_host)),
                              "note": "edtb200_transform_batch, pinned host buffers, both PCIe directions busy"}
    del out2
  except Exception as exc:
    e2e["batch_pipelined"] = {"error": repr(exc)}

  if rank == 0:
    line = {
      "metric": "Mvoxels/s edtsq 512^3 uint32", "value": value, "unit": "Mvoxels/s",
      "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_per_step,
      "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
      "dtype": "f32 (u32 labels)", "data": "synthetic",
      "config": {"workload": WORKLOAD, "per_gpu": "one 512^3 volume per rank" if world > 1 else "one 512^3 volume",
                 "l2": "inputs (1 GiB per step) larger than L2; no flush needed",
                 "timing": "CUDA events on the launch stream, max over ranks"},
      "roofline": roofline,
      "e2e": e2e,
      "gpu_launches": 3 * args.steps,
      "clocks": clocks,
      "device_equals_host_path": same,
    }
    if world == 1:
      try:
        line["workloads"] = workload_matrix(dev, peak)
      except Exception as exc:
        line["workloads"] = {"error": repr(exc)}
      try:
        line["e2e"]["pageable"], res_np = pageable_e2e(labels_np)
        line["e2e"]["pageable"]["equals_device_path"] = bool(np.array_equal(res_np, f_dev.cpu().numpy().T))
        del res_np
      except Exception as exc:
        line["e2e"]["pageable"] = {"error": repr(exc)}
    if world == 1 and not args.no_cpu_baseline:
      try:
        line["cpu_baseline"] = cpu_baseline_leg()
      except Exception as exc:   # the baseline is a report, never the product
        line["cpu_baseline"] = {"error": repr(exc)}
    print(json.dumps(line), flush=True)
  if world > 1:
    dist.destroy_process_group()


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=20)
  ap.add_argument("--warmup", type=int, default=3)
  ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
  ap.add_argument("--no-cpu-baseline", action="store_true")
  ap.add_argument("--dump-outputs", metavar="DIR",
                  help="after the timed steps, write a seeded sample of the last step's edtsq result to DIR/*.npy")
  args = ap.parse_args()
  if args.steps < 1:
    ap.error("--steps must be at least 1")
  if args.dump_outputs and args.impl == "reference":
    ap.error("--dump-outputs is only available for --impl ours")
  if args.impl == "reference":
    reference_arm(args)
  else:
    ours(args)


if __name__ == "__main__":
  main()
