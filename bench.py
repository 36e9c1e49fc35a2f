#!/usr/bin/env python
"""Benchmark of the GraphCast 6 h step on B200 (contract: see DESIGN.md section 6).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # CPU baseline arm

A "step" is one 6 h forecast step of GraphCast 0.25 deg (721x1440, 37 levels,
mesh 6, latent 512, 16 message steps) on synthetic N(0,1) inputs with
Haiku-default random weights.  Prints ONE JSON line on rank 0.

  value    : steps/s with inputs resident in HBM (pack -> step -> unpack), timed with CUDA
             events around K un-instrumented steps (the path a user runs: CUDA-graph replay of
             the step), max over ranks; N>1 = one independent forecast (ensemble member) per
             GPU, no data-path collective ("weak" scaling).
  e2e      : steps/s through the public API (GraphCast.__call__) with pinned HOST
             inputs: per step H2D of inputs+forcings and D2H of the predictions.
  roofline : the dominant kernel family (the tcgen05 fused layer / chain kernels) --
             algorithmic FLOPs of all its launches in a step / their summed CUDA-event time,
             measured in a SEPARATE profiling pass of the same loop (events around every launch,
             direct launches); `hbm` gives every kernel's achieved GB/s and fraction of the
             measured copy bandwidth; `traffic` is read from the committed ncu launch list.
  cpu_baseline / --impl reference : the fp32 CPU oracle (torch-CPU) on a bounded sample of the
             SAME workload: a contiguous block of 1/16 of the rows of every stage of the real
             0.25 degree graph (oracle/sampled_step.py), scaled by the row fraction.

--dump-outputs DIR writes what the last headline step returned, so that two builds run with the
same arguments (hence the same seeded inputs and weights) can be compared output for output:
  DIR/predictions.npy  float32 [n_out, k]: the step's output planes at k grid nodes (all of
                       them when they fit in 32 MiB, else a fixed seeded sample)
  DIR/grid_index.npy   float64 [k]: the grid node index of each column

The source tree may be read-only: nothing is written there (no bytecode; the static-graph cache
goes to a per-user temporary directory unless GRAPHCAST_B200_CACHE says otherwise).
"""

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

if "reference" in sys.argv:
  # The CPU arm uses every host thread; torchrun exports OMP_NUM_THREADS=1 to its workers,
  # which would silently make it single-threaded.  Must happen before numpy / torch load.
  for _v in ("OMP_NUM_THREADS", "MKL_NUM_THREADS"):
    os.environ[_v] = str(os.cpu_count() or 1)

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

WORKLOADS = {
    # name: (resolution, mesh_size, task name)
    "graphcast_0.25deg_37lvl": (0.25, 6, "TASK"),
    "graphcast_operational_0.25deg_13lvl": (0.25, 6, "TASK_13_PRECIP_OUT"),
    "graphcast_small_1deg_13lvl": (1.0, 5, "TASK_13"),
    "sample_2deg_13lvl": (2.0, 4, "TASK_13"),
    "tiny_4deg_13lvl": (4.0, 3, "TASK_13"),
}
DEFAULT_WORKLOAD = "graphcast_0.25deg_37lvl"
REFERENCE_BUDGET_S = 150.0   # wall-clock target of a whole `--impl reference` run
DUMP_BYTES = 32 << 20        # --dump-outputs: size of the sampled output (the full 0.25 deg one is 943 MB)


def algorithmic_flops(ng, nm, e1, e2, e3, c_in, n_out, steps, d=512):
  """2*MAC of every MLP in one step, reference dataflow (SURVEY.md section 8d)."""
  mlp = lambda rows, d_in, d_out: rows * (d_in * d + d * d_out)
  mac = (mlp(ng, c_in + 3, d) + mlp(nm, c_in + 3, d) + mlp(e1, 4, d) + mlp(e1, 3 * d, d)
         + mlp(nm, 2 * d, d) + mlp(ng, d, d)
         + mlp(e2, 4, d) + steps * (mlp(e2, 3 * d, d) + mlp(nm, 2 * d, d))
         + mlp(e3, 4, d) + mlp(e3, 3 * d, d) + mlp(ng, 2 * d, d) + mlp(ng, d, n_out))
  return 2.0 * mac


class ClockSampler:
  """nvidia-smi clocks / throttle reasons sampled during the timed region."""

  def __init__(self, gpu_index=0):
    self.rows = []
    self.proc = None
    self.gpu_index = gpu_index

  def start(self):
    q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    try:
      self.proc = subprocess.Popen(
          ["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
           "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      self.thread = threading.Thread(target=self._read, daemon=True)
      self.thread.start()
    except OSError:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.rows.append([x.strip() for x in line.split(",")])

  def stop(self):
    if self.proc is None:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    self.proc.terminate()
    try:
      self.proc.wait(timeout=5)
    except Exception:
      self.proc.kill()
    sm, smax, reasons = [], [], set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for r in self.rows:
      try:
        sm.append(float(r[0])); smax.append(float(r[1]))
      except (ValueError, IndexError):
        continue
      for name, v in zip(names, r[3:7]):
        if v.lower().startswith("active"):
          reasons.add(name)
    # "under load": samples with clocks above idle
    load = [x for x in sm if x > 500] or sm
    return {"sm_mhz": float(np.median(load)) if load else None,
            "sm_max_mhz": max(smax) if smax else None,
            "reasons": sorted(reasons), "samples": len(sm)}


def dist_env():
  rank = int(os.environ.get("RANK", "0"))
  world = int(os.environ.get("WORLD_SIZE", "1"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  return rank, world, local


def _cpu_sample(args, torch, steps, warmup, threads=None):
  """The bounded CPU sample shared by `cpu_baseline` and `--impl reference`: the fp32 oracle on a
  contiguous block of `--cpu-fraction` of the rows of every stage of the real workload graph
  (oracle/sampled_step.py); returns (seconds per sample (median), threads, description)."""
  from graphcast_b200 import graph as graph_lib, graphcast, synthetic
  from oracle import gnn as oracle_gnn, sampled_step
  cores = os.cpu_count() or 1
  res, mesh, task_name = WORKLOADS[args.workload]
  task = getattr(graphcast, task_name)
  lat, lon = synthetic.grid_coords(res)
  g = graph_lib.cached_static_graph(grid_lat=lat, grid_lon=lon, mesh_size=mesh,
                                    radius_query_fraction_edge_length=0.6)
  c_in = synthetic.num_input_channels(task)
  n_out = graphcast.num_outputs(task)
  params = oracle_gnn.init_params(c_in=c_in, n_out=n_out, msg_steps=16, seed=1)
  samp = sampled_step.SampledStep(g.as_dict(), params, c_in, args.cpu_fraction)
  # Thread count: torch's CPU ops regress badly with 128 threads on the GPU boxes' hosts, so
  # calibrate on one sample each (the first doubles as the page-fault warm-up), keep the fastest.
  best = None
  for n in ([threads] if threads else thread_candidates(cores)):
    torch.set_num_threads(n)
    t = samp.time_one()
    if best is None or t < best[0]:
      best = (t, n)
  torch.set_num_threads(best[1])
  for _ in range(warmup):
    samp.run()
  ts = [samp.time_one() for _ in range(max(steps, 1))]
  dt = float(np.median(ts))
  desc = (f"fp32 oracle on the first {args.cpu_fraction:.4f} of the rows of every stage of "
          f"{args.workload} (real graph indices, full-size gather tables): {dt:.2f} s per sample "
          f"measured (median of {len(ts)}), x{1.0 / args.cpu_fraction:.0f} per step")
  return dt, best[1], desc


def run_reference(args):
  """CPU arm: the fp32 oracle (restatement of the reference; its JAX stack cannot be installed
  here) on the host cores; each "step" is one bounded sample of the same workload."""
  rank, world, _ = dist_env()
  if rank != 0:
    return
  import torch
  t_wall = time.perf_counter()
  dt, cores, desc = _cpu_sample(args, torch, args.steps, args.warmup)
  s_per_step = dt / args.cpu_fraction
  value = 1.0 / s_per_step
  line = {
      "impl": "reference", "metric": "6h-step forecasts/sec", "value": value, "unit": "steps/s",
      "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": s_per_step * 1e3,
      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
      "data": "synthetic",
      "config": {"workload": args.workload, "sample_fraction": args.cpu_fraction,
                 "measured_ms_per_sample": dt * 1e3,
                 "note": "ms_per_step = measured_ms_per_sample / sample_fraction (each timed step is "
                         "a bounded sample of the workload, as the contract allows)",
                 "wall_s": time.perf_counter() - t_wall},
      "cpu_baseline": {"value": value, "unit": "steps/s", "cores": cores, "kind": "port",
                       "sample": desc},
      "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
      "gpu_launches": 0,
  }
  print(json.dumps(line), flush=True)


def full_workload_sizes(name):
  """(Ng, Nm, E_g2m, E_mesh, E_m2g, c_in, n_out, steps) of a named workload
  (edge counts: SURVEY.md section 8 table, measured with this repo's builder)."""
  from graphcast_b200 import graphcast, synthetic
  res, mesh, task_name = WORKLOADS[name]
  task = getattr(graphcast, task_name)
  n_lat, n_lon = int(round(180 / res)) + 1, int(round(360 / res))
  ng = n_lat * n_lon
  nm = 10 * 4 ** mesh + 2
  e2 = sum(60 * 4 ** l for l in range(mesh + 1))
  e1 = {(0.25, 6): 1618818, (1.0, 5): 101892}.get((res, mesh))
  if e1 is None:
    e1 = int(1.56 * ng)
  return (ng, nm, e1, e2, 3 * ng, synthetic.num_input_channels(task),
          graphcast.num_outputs(task), 16)


def thread_candidates(cores):
  """Thread counts worth trying for the torch-CPU oracle, most promising first."""
  c = [min(cores, 32), min(cores, 16)]
  if cores <= 64:
    c.append(cores)
  return sorted(set(c), reverse=True)


def cpu_baseline_sample(args, torch):
  """Bounded CPU sample on rank 0 (reported beside the GPU number): same sampler as the
  reference arm, 3 samples."""
  dt, cores, desc = _cpu_sample(args, torch, steps=3, warmup=0)
  return {"value": args.cpu_fraction / dt, "unit": "steps/s", "cores": cores, "kind": "port",
          "sample": desc}


def ncu_traffic(workload, precision):
  """DRAM bytes per step of the tensor-core kernels from the committed ncu launch list of this
  build (profiles/r02_launches_ncu.csv: dram__bytes_read.sum + dram__bytes_write.sum per
  launch).  None when no list for this configuration is committed."""
  path = os.path.join(REPO, "profiles", "r02_launches_ncu.csv")
  if workload != DEFAULT_WORKLOAD or precision != "bf16x3" or not os.path.exists(path):
    return None, None
  tc, total = 0.0, 0.0
  try:
    for line in open(path):
      if line.startswith("#") or line.startswith("id,"):
        continue
      parts = line.rstrip("\n").rsplit(",", 3)
      name, rd, wr = parts[0], float(parts[2]), float(parts[3])
      total += rd + wr
      if "mlp_chain_tc_kernel" in name or "mlp_layer_tc_kernel" in name:
        tc += rd + wr
  except Exception:
    return None, None
  return tc, f"ncu, profiles/r02_launches_ncu.csv (whole step {total / 1e9:.1f} GB)"


def dump_outputs(out_dir, planes_out):
  """Writes the step output planes_out [n_out, Ng] (device, fp32) to out_dir: every grid node if
  it fits in DUMP_BYTES, else the same seeded sample of grid nodes on every run."""
  import torch
  n_out, ng = planes_out.shape
  k = min(ng, DUMP_BYTES // (4 * n_out + 8))
  idx = np.arange(ng) if k == ng else np.sort(np.random.default_rng(0).choice(ng, k, replace=False))
  sample = planes_out.index_select(1, torch.as_tensor(idx, device=planes_out.device))
  os.makedirs(out_dir, exist_ok=True)
  np.save(os.path.join(out_dir, "predictions.npy"), sample.cpu().numpy())
  np.save(os.path.join(out_dir, "grid_index.npy"), idx.astype(np.float64))


def run_b200(args):
  import torch
  import torch.distributed as dist
  from graphcast_b200 import _native, graphcast, synthetic

  rank, world, local = dist_env()
  if world > 1:
    dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
  torch.cuda.set_device(local)
  dev = torch.device(f"cuda:{local}")
  lib = _native.lib()
  if args.cluster:
    _native.check(lib.gcb_set_cluster_size(args.cluster), "gcb_set_cluster_size")
  if os.environ.get("GCB_DEBUG_FLAGS"):   # kernel experiment switches (gcb_debug_flags); not for results
    _native.check(lib.gcb_debug_flags(int(os.environ["GCB_DEBUG_FLAGS"])), "gcb_debug_flags")

  res, mesh, task_name = WORKLOADS[args.workload]
  task = getattr(graphcast, task_name)
  cfg = graphcast.ModelConfig(resolution=res, mesh_size=mesh, latent_size=512, gnn_msg_steps=16,
                              hidden_layers=1, radius_query_fraction_edge_length=0.6)
  c_in = synthetic.num_input_channels(task)
  t_setup = time.perf_counter()
  inputs, template, forcings = synthetic.make_example(task, res, batch=1, seed=rank,
                                                      pinned=True)
  params = graphcast.init_params(cfg, task, c_in, seed=1)
  model = graphcast.GraphCast(cfg, task, params=params, precision=args.precision, device=dev,
                              pregather=args.pregather, fuse=args.fuse, chain_lag=args.chain_lag,
                              image_residual=args.image_residual, deep_chains=args.deep_chains)
  # First call builds the static graph, uploads weights, allocates the workspace.
  pred = model(inputs, template, forcings)
  torch.cuda.synchronize()
  eng = model.engine
  setup_s = time.perf_counter() - t_setup
  n_out = eng.n_out
  h2d = sum(int(np.prod(v.shape)) * 4 for ds in (inputs, forcings) for v in ds.data_vars.values())
  d2h = n_out * eng.num_grid * 4

  # ---------------- device-resident timed region --------------------------------
  planes_in = model._planes_in[0]
  planes_out = torch.empty([n_out, eng.num_grid], dtype=torch.float32, device=dev)

  def one_step():
    eng.pack_inputs(planes_in)
    eng.step()
    eng.unpack_outputs(planes_out)

  for _ in range(max(args.warmup, 3)):
    one_step()
  torch.cuda.synchronize()
  sampler = ClockSampler(local)
  if rank == 0:
    sampler.start()
  if world > 1:
    dist.barrier()
  torch.cuda.synchronize()
  # Headline: K un-instrumented steps (gcb_forward replays its CUDA graph, as for any caller).
  ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  ev0.record()
  for _ in range(args.steps):
    one_step()
  ev1.record()
  torch.cuda.synchronize()
  if world > 1:
    dist.barrier()
  elapsed_ms = ev0.elapsed_time(ev1)
  clocks = sampler.stop() if rank == 0 else None
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, planes_out)

  # Profiling pass (separate from the headline): the same loop with a CUDA-event pair around
  # every launch (direct launches instead of graph replay) -> per-kernel durations.
  prof_steps = max(1, min(args.steps, args.profile_steps))
  cap = 256 * prof_steps
  lib.gcb_profile_begin()
  pv0, pv1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  pv0.record()
  for _ in range(prof_steps):
    one_step()
  pv1.record()
  torch.cuda.synchronize()
  prof_ms_per_step = pv0.elapsed_time(pv1) / prof_steps
  kinds = (C.c_int32 * cap)(); ms = (C.c_float * cap)()
  flops = (C.c_double * cap)(); nbytes = (C.c_double * cap)(); cnt = C.c_int32(0)
  _native.check(lib.gcb_profile_end(cap, kinds, ms, flops, nbytes, C.byref(cnt)), "profile_end")
  n_launch = min(cnt.value, cap)
  per_step_launches = cnt.value // prof_steps

  t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  ms_per_step = float(t.item()) / args.steps
  value = world * 1e3 / ms_per_step

  if args.dump_launches and rank == 0:
    with open(args.dump_launches, "w") as f:
      f.write("idx,kind,ms,gflop,gbyte\n")
      lo = (prof_steps - 1) * per_step_launches
      for i in range(lo, min(lo + per_step_launches, n_launch)):
        f.write(f"{i - lo},{kinds[i]},{ms[i]:.4f},{flops[i] / 1e9:.2f},{nbytes[i] / 1e9:.4f}\n")
  # per-kind aggregation (this rank)
  kind_names = {0: "mlp_layer_tc", 1: "segment_sum", 2: "pack", 3: "unpack", 4: "mlp_layer_simt",
                5: "rows_to_image", 6: "mlp_chain_tc", 7: "gather_rows"}
  agg = {}
  for i in range(n_launch):
    a = agg.setdefault(kind_names[kinds[i]], [0.0, 0.0, 0.0, 0])
    a[0] += ms[i]; a[1] += flops[i]; a[2] += nbytes[i]; a[3] += 1
  m = eng._model
  alg_flops = algorithmic_flops(m.num_grid, m.num_mesh, m.e_g2m, m.e_mesh, m.e_m2g, c_in, n_out, 16)
  # the tensor-core kernel family: single fused layers + fused chains (same MMA / epilogue code)
  tc = [0.0, 0.0, 0.0, 0]
  for k in ("mlp_layer_tc", "mlp_chain_tc", "mlp_layer_simt"):
    if k in agg:
      tc = [x + y for x, y in zip(tc, agg[k])]
  tc_ms_per_step = max(tc[0] / prof_steps, 1e-9)
  achieved_tflops = alg_flops / (tc_ms_per_step * 1e-3) / 1e12
  peaks = {}
  try:
    peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
  except Exception:
    pass
  peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
  peak_hbm = peaks.get("hbm_gbs", 6500.0)
  peak_src = ("measured (MEASURED_PEAKS.json: bf16_tflops_sustained, hbm_gbs)" if peaks
              else "fallback 1.4 PFLOP/s, 6.5 TB/s (B200_PROFILING.md)")
  products = {"bf16x3": 3, "bf16": 1, "fp32_simt": 1}[args.precision]
  # MACs the kernels really issue (the split edge layers execute fewer than the reference
  # dataflow the algorithmic figure is defined on), times the products per MAC.
  executed_tflops = (tc[1] / prof_steps) * products / (tc_ms_per_step * 1e-3) / 1e12
  traffic, traffic_src = ncu_traffic(args.workload, args.precision)
  roofline = {
      "kernel": "gcb::mlp_chain_tc_kernel + gcb::mlp_layer_tc_kernel (fused tcgen05 layers)",
      "bound": "tensor",
      "achieved": achieved_tflops, "peak": peak_tf, "unit": "TFLOP/s",
      "frac": achieved_tflops / peak_tf, "traffic": traffic,
      "traffic_unit": "DRAM bytes per step, all launches of this kernel family",
      "traffic_source": traffic_src, "peak_source": peak_src,
      "launches_per_step": tc[3] // prof_steps, "kernel_ms_per_step": tc_ms_per_step,
      "kernel_share_of_step": tc_ms_per_step / prof_ms_per_step,
      "profile_pass": {"steps": prof_steps, "ms_per_step": prof_ms_per_step,
                       "note": "event pair around every launch, direct launches; the headline "
                               "ms_per_step is timed separately without instrumentation"},
      "algorithmic_tflop_per_step": alg_flops / 1e12,
      "tensor_products_per_mac": products,
      "executed_tflop_per_step": tc[1] / prof_steps * products / 1e12,
      "executed_tensor_tflops": executed_tflops,
      "tensor_pipe_frac": executed_tflops / peak_tf,
      "algorithmic_hbm_GB_per_step": sum(v[2] for v in agg.values()) / prof_steps / 1e9,
      "other_kernels_ms_per_step": {k: v[0] / prof_steps for k, v in agg.items()
                                    if not k.startswith("mlp_")},
      # every kernel against the HBM roofline: algorithmic bytes / CUDA-event time / measured copy bandwidth
      "hbm": {k: {"GB_per_step": v[2] / prof_steps / 1e9, "ms_per_step": v[0] / prof_steps,
                  "GBps": (v[2] / 1e9) / (v[0] * 1e-3) if v[0] > 0 else None,
                  "hbm_frac": ((v[2] / 1e9) / (v[0] * 1e-3) / peak_hbm) if v[0] > 0 else None}
              for k, v in agg.items()},
      "hbm_peak_GBps": peak_hbm,
  }

  # ---------------- end-to-end through the public API ---------------------------
  # Serving loop: every step uploads its inputs from pinned host memory (GraphCast.__call__
  # stages them on its own copy stream, double buffered) and downloads its predictions to
  # pinned host memory on a second copy stream; the host only synchronises at the end, so
  # the transfers of neighbouring steps overlap the kernels.  All K uploads, K steps and K
  # downloads are inside the timed region.
  host_out = [{name: torch.empty(v.shape, dtype=torch.float32, pin_memory=True)
               for name, v in pred.data_vars.items()} for _ in range(2)]
  d2h_stream = torch.cuda.Stream(device=dev)
  compute = torch.cuda.current_stream(dev)

  def e2e_step(i):
    p = model(inputs, template, forcings)           # H2D of every input inside
    done = torch.cuda.Event()
    done.record(compute)
    with torch.cuda.stream(d2h_stream):
      d2h_stream.wait_event(done)
      for name, v in p.data_vars.items():
        v.data.record_stream(d2h_stream)
        host_out[i % 2][name].copy_(v.data, non_blocking=True)   # D2H of the predictions

  e2e_steps = max(2, min(args.steps, args.e2e_steps))
  e2e_step(0)
  torch.cuda.synchronize()
  if world > 1:
    dist.barrier()
  t0 = time.perf_counter()
  for i in range(e2e_steps):
    e2e_step(i)
  torch.cuda.synchronize()
  e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
  t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dist.barrier()
  e2e_value = world * 1e3 / float(t.item())

  if rank == 0:
    cpu = None
    if world == 1 and not args.skip_cpu_baseline:
      cpu = cpu_baseline_sample(args, torch)
    line = {
        "metric": "6h-step forecasts/sec", "value": value, "unit": "steps/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": {"bf16x3": "bf16x3 (3 bf16 tensor-core products, fp32 accumulate; parity mode)",
                  "bf16": "bf16", "fp32_simt": "f32"}[args.precision],
        "data": "synthetic",
        "config": {"workload": args.workload, "resolution_deg": res, "mesh_size": mesh,
                   "levels": len(task.pressure_levels), "latent": 512, "msg_steps": 16,
                   "batch": 1, "precision": args.precision, "cluster": args.cluster or "default(2)",
                   "pregather": bool(args.pregather), "fuse": bool(args.fuse), "chain_lag": args.chain_lag,
                   "image_residual": bool(args.image_residual), "deep_chains": bool(args.deep_chains),
                   "parallelism": "1 forecast per GPU (ensemble members), no collective",
                   "l2_policy": "working set per step (>20 GB) far exceeds the 126 MB L2; no flush needed",
                   "setup_s": setup_s},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "ms_per_step": float(t.item()), "steps": e2e_steps},
        "gpu_launches": per_step_launches * args.steps,
        "gpu_launches_per_step": per_step_launches,
        "roofline": roofline,
        "cpu_baseline": cpu,
    }
    print(json.dumps(line), flush=True)
  if world > 1:
    dist.destroy_process_group()


def run_partitioned(args):
  """BASELINE config 4: ONE forecast per step, mesh-node partitioned over all ranks (strong
  scaling): receiver-owned edges, one grouped NCCL all-to-all-v of halo rows per message-passing
  step (graphcast_b200/partitioned.py)."""
  import torch
  import torch.distributed as dist
  from graphcast_b200 import _native, engine, graph as graph_lib, graphcast, partitioned, synthetic

  rank, world, local = dist_env()
  torch.cuda.set_device(local)
  dev = torch.device(f"cuda:{local}")
  if world > 1:
    dist.init_process_group("nccl", device_id=dev)
  res, mesh, task_name = WORKLOADS[args.workload]
  task = getattr(graphcast, task_name)
  cfg = graphcast.ModelConfig(resolution=res, mesh_size=mesh, latent_size=512, gnn_msg_steps=16,
                              hidden_layers=1, radius_query_fraction_edge_length=0.6)
  c_in = synthetic.num_input_channels(task)
  n_out = graphcast.num_outputs(task)
  lat, lon = synthetic.grid_coords(res)
  g = graph_lib.cached_static_graph(grid_lat=lat, grid_lon=lon, mesh_size=mesh,
                                    radius_query_fraction_edge_length=0.6)
  params = graphcast.init_params(cfg, task, c_in, seed=1)
  pe = partitioned.PartitionedEngine(g, params, c_in=c_in, n_out=n_out, msg_steps=16, rank=rank,
                                     world=world, device=dev, precision=args.precision,
                                     image_residual=args.image_residual)
  lg = pe.local
  gen = torch.Generator(device=dev).manual_seed(0)          # same full field on every rank
  planes_full = torch.randn(c_in, g.num_grid_nodes, device=dev, generator=gen)
  planes_local = planes_full[:, torch.as_tensor(lg.local_grid_ids, device=dev)].contiguous()
  if not args.check:
    del planes_full
  n_owned = int(lg.grid_owned.size)
  planes_out = torch.empty([n_out, n_owned], dtype=torch.float32, device=dev)

  def one_step(timed_halo=False):
    pe.step(planes_local, timed_halo)
    with pe.engine._on_device():
      _native.check(pe._lib.gcb_unpack_grid_outputs(
          pe.engine.grid_out.data_ptr(), 256, n_out, n_owned, None, None, None, None,
          planes_out.data_ptr(), pe.engine._stream()), "gcb_unpack_grid_outputs")

  for _ in range(max(args.warmup, 3)):
    one_step()
  torch.cuda.synchronize()
  sampler = ClockSampler(local)
  if rank == 0:
    sampler.start()
  if world > 1:
    dist.barrier()
  torch.cuda.synchronize()
  ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  ev0.record()
  for _ in range(args.steps):
    one_step()
  ev1.record()
  torch.cuda.synchronize()
  if world > 1:
    dist.barrier()
  t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  ms_per_step = float(t.item()) / args.steps
  clocks = sampler.stop() if rank == 0 else None
  # Cost of the halo exchanges: the same K steps with the exchanges skipped (results are then
  # wrong, the kernels and their sizes are the same), max over ranks; the difference is what the
  # 17 exchanges of a step cost in latency, including the waiting they introduce.
  pe.skip_exchange = True
  one_step()
  torch.cuda.synchronize()
  if world > 1:
    dist.barrier()
  ev0.record()
  for _ in range(args.steps):
    one_step()
  ev1.record()
  torch.cuda.synchronize()
  h = torch.tensor([ev0.elapsed_time(ev1) / args.steps], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(h, op=dist.ReduceOp.MAX)
  pe.skip_exchange = False
  one_step()                                               # restore a valid state for --check
  torch.cuda.synchronize()

  # Per-kernel profile of rank 0 (separate pass: an event pair around every launch of the C ABI).
  lib = _native.lib()
  prof_steps = max(1, min(args.steps, args.profile_steps))
  cap = 512 * prof_steps
  lib.gcb_profile_begin()
  for _ in range(prof_steps):
    one_step()
  torch.cuda.synchronize()
  kinds = (C.c_int32 * cap)(); kms = (C.c_float * cap)()
  kfl = (C.c_double * cap)(); kby = (C.c_double * cap)(); cnt = C.c_int32(0)
  _native.check(lib.gcb_profile_end(cap, kinds, kms, kfl, kby, C.byref(cnt)), "profile_end")
  launches_per_step = cnt.value // prof_steps
  tc_ms = sum(kms[i] for i in range(min(cnt.value, cap)) if kinds[i] in (0, 6)) / prof_steps

  # End to end: every step uploads this rank's input planes from pinned host memory and downloads
  # its share of the predictions to pinned host memory (both inside the timed region).
  host_in = torch.empty(planes_local.shape, dtype=torch.float32, pin_memory=True)
  host_in.copy_(planes_local)
  host_out = torch.empty(planes_out.shape, dtype=torch.float32, pin_memory=True)

  def e2e_step():
    # PartitionedEngine.step_from_host: upload on a copy stream, download on a second side stream,
    # double-buffered, so the copies of neighbouring steps overlap the kernels
    return pe.step_from_host(host_in, host_out)

  e2e_steps = max(2, min(args.steps, args.e2e_steps))
  e2e_step()
  e2e_step()
  torch.cuda.synchronize()
  if world > 1:
    dist.barrier()
  t0 = time.perf_counter()
  for _ in range(e2e_steps):
    e2e_step()
  torch.cuda.synchronize()
  e2e = torch.tensor([(time.perf_counter() - t0) * 1e3 / e2e_steps], dtype=torch.float64, device=dev)
  io = torch.tensor([host_in.numel() * 4, host_out.numel() * 4], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(e2e, op=dist.ReduceOp.MAX)
    dist.all_reduce(io, op=dist.ReduceOp.SUM)
  one_step()                                               # valid state again for --check
  torch.cuda.synchronize()
  # same inputs -> the pipelined host path must have delivered the device path's result bit for bit
  e2e_same = torch.tensor([int(torch.equal(host_out.to(dev), planes_out))], device=dev)
  if world > 1:
    dist.all_reduce(e2e_same, op=dist.ReduceOp.MIN)
  if not bool(e2e_same.item()):
    raise RuntimeError("step_from_host delivered a result that differs from the device-resident step")

  check = None
  if args.check:
    # partitioned output (gathered) against the single-GPU step with the same kernels
    n_max = torch.tensor([n_owned], device=dev)
    if world > 1:
      dist.all_reduce(n_max, op=dist.ReduceOp.MAX)
    pad = torch.zeros([int(n_max.item()), 256], dtype=torch.float32, device=dev)
    pad[:n_owned] = pe.engine.grid_out[:n_owned]
    parts = [torch.empty_like(pad) for _ in range(world)]
    if world > 1:
      dist.all_gather(parts, pad)
    else:
      parts = [pad]
    owners = [partitioned.build_local_graph(g, world, r).grid_owned for r in range(world)] if rank == 0 else None
    if rank == 0:
      del pe
      torch.cuda.empty_cache()
      eng = engine.Engine(g, params, c_in=c_in, n_out=n_out, msg_steps=16, precision=args.precision,
                          device=dev, image_residual=args.image_residual, deep_chains=False)
      eng.pack_inputs(planes_full)
      eng.step()
      torch.cuda.synchronize()
      full = eng.grid_out[:, :n_out]
      scale = float(full.abs().max())
      err = 0.0
      for r in range(world):
        ids = torch.as_tensor(owners[r], device=dev)
        err = max(err, float((parts[r][:ids.numel(), :n_out] - full[ids]).abs().max()) / scale)
      check = {"max_abs_rel_err_vs_single_gpu": err, "bitwise_equal": err == 0.0}

  alg_flops = algorithmic_flops(g.num_grid_nodes, g.num_mesh_nodes, len(g.g2m_senders),
                                len(g.mesh_senders), len(g.m2g_senders), c_in, n_out, 16)
  try:
    peak_tf = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json"))).get("bf16_tflops_sustained", 1400.0)
  except Exception:
    peak_tf = 1400.0
  if rank == 0:
    st = partitioned.plan_statistics(g, world) if world > 1 else None
    line = {
        "metric": "6h-step forecasts/sec", "value": 1e3 / ms_per_step, "unit": "steps/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": args.precision, "data": "synthetic",
        "config": {"workload": args.workload, "mode": "partitioned",
                   "parallelism": f"one forecast over {world} GPUs: mesh nodes by recursive coordinate "
                                  "bisection, edges owned by their receiver, grid nodes by containing "
                                  "triangle; 17 halo exchanges (NCCL all_to_all_v of fp32 rows) per step",
                   "image_residual": bool(args.image_residual),
                   "ms_per_step_without_halo_exchange": float(h.item()),
                   "halo_exchange_ms_per_step": ms_per_step - float(h.item()),
                   "halo_exchanges_per_step": 17 if world > 1 else 0,
                   "partition": st},
        "clocks": clocks, "check": check,
        "e2e": {"value": 1e3 / float(e2e.item()), "unit": "steps/s", "ms_per_step": float(e2e.item()),
                "h2d_bytes_per_step": int(io[0].item()), "d2h_bytes_per_step": int(io[1].item()),
                "steps": e2e_steps,
                "note": "PartitionedEngine.step_from_host: every rank uploads its local input planes from pinned host "
                        "memory and downloads its owned prediction rows every step; copies double-buffered on "
                        "side streams (overlapping neighbouring steps); result checked bit-identical to the "
                        "device-resident step"},
        "gpu_launches": launches_per_step * args.steps * world,
        "gpu_launches_per_step": launches_per_step * world,
        "gpu_launches_note": "kernels launched through the C ABI per forecast step, summed over ranks "
                             "(rank 0 counted, x world); the NCCL all_to_all kernels come on top",
        "roofline": {
            "kernel": "gcb::mlp_chain_tc_kernel + gcb::mlp_layer_tc_kernel (fused tcgen05 layers), rank 0",
            "bound": "tensor", "unit": "TFLOP/s",
            "achieved": alg_flops / world / (max(tc_ms, 1e-9) * 1e-3) / 1e12, "peak": peak_tf,
            "frac": alg_flops / world / (max(tc_ms, 1e-9) * 1e-3) / 1e12 / peak_tf,
            "kernel_ms_per_step": tc_ms, "kernel_share_of_step": tc_ms / ms_per_step,
            "traffic": None,
            "note": "algorithmic FLOPs of the whole step / ranks, over rank 0's tensor-core kernel time"},
        "cpu_baseline": None,
    }
    print(json.dumps(line), flush=True)
  if world > 1:
    dist.destroy_process_group()


def run_rollout(args):
  """BASELINE config 3: an N-step autoregressive rollout through the public API
  (`rollout.chunked_prediction_generator`): device-resident state (the next inputs are assembled on
  the GPU), forcings generated per step on the device (TISR kernel + progress features), every
  prediction copied to pinned host memory.  value = forecast steps per second over the rollout."""
  import torch
  from graphcast_b200 import graphcast, rollout, synthetic
  rank, world, local = dist_env()
  if rank != 0:
    return
  torch.cuda.set_device(local)
  dev = torch.device(f"cuda:{local}")
  res, mesh, task_name = WORKLOADS[args.workload]
  task = getattr(graphcast, task_name)
  cfg = graphcast.ModelConfig(resolution=res, mesh_size=mesh, latent_size=512, gnn_msg_steps=16,
                              hidden_layers=1, radius_query_fraction_edge_length=0.6)
  c_in = synthetic.num_input_channels(task)
  n = args.rollout
  inputs, template, _ = synthetic.make_example(task, res, num_target_steps=n, seed=0, pinned=True)
  dt = (np.datetime64("2021-03-17T06:00:00") + np.asarray(template.coords["time"][1])).astype("datetime64[ns]")[None, :]
  template = template.assign_coords(datetime=(("batch", "time"), dt))
  params = graphcast.init_params(cfg, task, c_in, seed=1)
  model = graphcast.GraphCast(cfg, task, params=params, precision=args.precision, device=dev)
  fn = lambda rng, inputs, targets_template, forcings: model(inputs, targets_template, forcings)
  gen = list(task.forcing_variables)
  sink = rollout.PinnedPredictionSink(depth=2)
  host = None

  def run(template_n):
    nonlocal host
    count = 0
    for chunk in rollout.chunked_prediction_generator(fn, None, inputs, template_n, 1, None,
                                                      generate_forcings=gen):
      host = sink(chunk)                     # D2H on a side stream, under the next step's kernels
      count += 1
    sink.wait()
    torch.cuda.synchronize()
    return count

  run(rollout.extend_targets_template(template, 2))          # warm-up: graph build, first replays
  t0 = time.perf_counter()
  steps = run(template)
  secs = time.perf_counter() - t0
  d2h = sum(int(np.prod(v.shape)) * 4 for v in host.values())
  line = {
      "metric": "6h-step forecasts/sec", "value": steps / secs, "unit": "steps/s", "n_gpus": 1,
      "steps": steps, "warmup": 2, "ms_per_step": secs / steps * 1e3, "higher_is_better": True,
      "scaling": "weak", "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
      "config": {"workload": args.workload + f"_rollout{steps}", "mode": "rollout",
                 "seconds_per_rollout": secs,
                 "note": "rollout.chunked_prediction_generator: device-resident state, forcings "
                         "generated on the device, every prediction copied to pinned host memory by "
                         "rollout.PinnedPredictionSink (side stream, overlapping the next step); wall clock"},
      "e2e": {"value": steps / secs, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": d2h},
  }
  print(json.dumps(line), flush=True)


def main():
  # Exactly one JSON line may reach stdout: libraries (NCCL's version banner, warnings) are
  # diverted to stderr by pointing fd 1 at fd 2 for the duration of the run.
  real_stdout = os.dup(1)
  os.dup2(2, 1)
  sys.stdout = os.fdopen(real_stdout, "w", buffering=1)
  os.environ["NCCL_DEBUG"] = os.environ.get("GCB_NCCL_DEBUG", "INFO")   # communicator lines on stderr
  # The project modules are imported after this point; the tree may be read-only.
  sys.dont_write_bytecode = True
  os.environ.setdefault("GRAPHCAST_B200_CACHE",
                        os.path.join(tempfile.gettempdir(), f"graphcast_b200_cache_{os.getuid()}"))
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=10)
  ap.add_argument("--warmup", type=int, default=3)
  ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
  ap.add_argument("--mode", choices=["auto", "replicas", "partitioned"], default="auto",
                  help="partitioned (default for N > 1): ONE forecast over all GPUs, mesh-node partition "
                       "+ NCCL halo exchange per message-passing step (strong scaling); replicas: one "
                       "independent forecast per GPU, no collective (weak scaling)")
  ap.add_argument("--rollout", type=int, default=0,
                  help="BASELINE config 3: time an N-step autoregressive rollout through the public API")
  ap.add_argument("--check", action="store_true",
                  help="partitioned mode: compare the gathered output with the single-GPU step")
  ap.add_argument("--workload", choices=sorted(WORKLOADS), default=DEFAULT_WORKLOAD)
  ap.add_argument("--precision", choices=["bf16x3", "bf16", "fp32_simt"], default="bf16x3")
  ap.add_argument("--cpu-fraction", dest="cpu_fraction", type=float, default=1.0 / 16,
                  help="row fraction of every stage of the workload the CPU sample runs")
  ap.add_argument("--profile-steps", dest="profile_steps", type=int, default=5)
  ap.add_argument("--e2e-steps", dest="e2e_steps", type=int, default=10)
  ap.add_argument("--skip-cpu-baseline", action="store_true")
  ap.add_argument("--cluster", type=int, default=0, help="CTAs per cluster (0 = library default)")
  ap.add_argument("--dump-launches", default="", help="write per-launch (kind, ms, GFLOP, GB) of the last timed step to this file")
  ap.add_argument("--dump-outputs", default="", metavar="DIR",
                  help="write the output of the last timed step to DIR/*.npy (single-forecast GPU path)")
  ap.add_argument("--no-fuse", dest="fuse", action="store_false",
                  help="one launch per linear layer (hidden activations through HBM)")
  ap.add_argument("--chain-lag", dest="chain_lag", type=int, default=0)
  ap.add_argument("--masters", dest="image_residual", action="store_false",
                  help="keep fp32 masters of the latent streams next to the operand images")
  ap.add_argument("--no-deep", dest="deep_chains", action="store_false",
                  help="two-layer chains only (no [embedder -> edge MLP] / [node MLP -> projections] launches)")
  ap.add_argument("--no-pregather", dest="pregather", action="store_false",
                  help="evaluate the first edge-MLP layer over the concatenated K=1536 input")
  args = ap.parse_args()
  if args.steps < 1:
    ap.error("--steps must be at least 1")
  partitioned = args.mode == "partitioned" or (args.mode == "auto" and dist_env()[1] > 1)
  if args.dump_outputs and (args.impl == "reference" or args.rollout > 0 or partitioned):
    ap.error("--dump-outputs applies to the single-forecast GPU path (--impl b200, no --rollout, "
             "--mode replicas for N > 1)")
  if args.impl == "reference":
    run_reference(args)
  elif args.rollout > 0:
    run_rollout(args)
  elif partitioned:
    run_partitioned(args)
  else:
    run_b200(args)


if __name__ == "__main__":
  main()
