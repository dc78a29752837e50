#!/usr/bin/env python3
"""Benchmark of the PARESIS image-formation hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Metric (BASELINE.json): speckle image-sets/s.  One image-set = everything PARESIS's main.py
produces for one membrane position (main.py:63-110): a fresh membrane thickness map, the
sample and reference images (plus propagation and white images at position 0), detector
blur, binning and Poisson noise included.  Workload = BASELINE.json configs[1]: 2048^2
oversampled grid, monochromatic 52 keV, 20 membrane positions, ray-tracing refraction model,
detector PSF 1.2 px + Poisson noise (experiment "B200_2048_mono" of the shipped XML).

One step = JOBS_PER_STEP (40) jobs of 20 membrane positions each = 800 image-sets, so that the timed region of the
default run lasts seconds, not milliseconds (a sustained measurement: clocks and power settle).  `value` is measured
with all inputs resident in HBM (sphere field, sample map); `e2e` runs 20-position jobs through the drop-in Python API
(Experiment.getMyGeometry + computeSampleAndReferenceImages_RT, numpy results on the host, membrane map copied back as
main.py:99 does) and is quoted next to the platform's device->host ceiling measured in the same run (`e2e.d2h_ceiling`).
N > 1: one process per GPU (torchrun), each rank its own positions, no data-path collective for this workload
(positions are independent) -> weak scaling.

The same line carries, measured live in the same run:
  `energy_sharded` -- BASELINE.json configs[2] (4096^2, 64 energies, 20 positions): the spectrum of every position is
      dealt round-robin over the N ranks, each rank accumulates its energies, applies the linear part of the detector and
      ONE NCCL reduce per detector bin sums the detector-resolution partials on the owner, which draws the Poisson noise
      (paresis_b200/shard.py; Experiment.py:482-483, :501-521).  Strong scaling: the job is fixed, N splits it.
  `grid_8192` (N = 1) -- BASELINE.json configs[4] sub-sample (8192^2, 8 of the 128 energies x 4 positions): throughput
      and per-kernel roofline fractions at a grid whose working set does NOT fit the 126 MB L2.

At N = 1 the line also carries `splat`: BASELINE.json's second figure, the stand-alone refraction splat
(`paresis_splat`, 16 algorithmic bytes per study pixel) timed live on a membrane's displacement field at 2048^2 and
8192^2, direct REDs (variant 2) next to the shared-memory tile kernel (variant 3), as GB/s and fraction of the HBM peak.

`--impl reference` times the CPU oracle port of the same path (oracle/, fp64 numpy + C) on the
host cores, one process per core, on a bounded sample of the same workload.

`--dump-outputs DIR` writes, after the timed steps, what the last job of the last timed step returned on rank 0
(ImageFormation.compute_rt_positions: thickness, sample, reference, propag, white, sums) as DIR/<name>.npy, so that two
builds run with the same arguments can be compared output for output (the inputs depend only on the arguments).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

EXPERIMENT = "B200_2048_mono"
POSITIONS = 20
JOBS_PER_STEP = 40      # a timed step = 40 jobs x 20 positions (a job is one paresis_rt_run_positions call)
E2E_JOBS_PER_STEP = 5   # an end-to-end step = 5 jobs x 20 positions through the Python API
METRIC = "speckle_image_sets_per_s"
UNIT = "image-sets/s"
WORKLOAD = "2048^2 grid (detector 1024^2 x os 2), mono 52 keV, 20 membrane positions, RayT, PSF 1.2 px + Poisson"

# algorithmic bytes per LAUNCH (fp32), SURVEY.md section 8(d) / DESIGN.md "Kernels": n study pixels, det detector pixels
ALG_BYTES = {
    "raster_spheres": lambda n, det: 4.0 * n,                 # write the thickness map once
    "refract_membrane_hop": lambda n, det: 8.0 * n,           # read t_m, write I_bs
    "refract_sample_ref_hop": lambda n, det: 20.0 * n,        # read I_bs, t_m, t_s; write sample + reference
    "detect": lambda n, det: 2 * (4.0 * n + 4.0 * det),       # sample + reference images in one launch: read, write counts
}
SLOTS = 5               # membrane positions in flight (same-box A/B: 3 -> 5 is +1.2 %, 6 no better)
PER_LAUNCH = 0   # > 1: that many positions share each kernel launch (blockIdx.z) instead; measured no faster (DESIGN.md)


DUMP_OUTPUTS = ("thickness", "sample", "reference", "propag", "white", "sums")
DUMP_MAX_ELEMENTS = 1 << 22     # per output: 16 MiB of float32; the six outputs of a job stay under 64 MB in all


def dump_outputs(directory, res, torch):
    """Write each output of one compute_rt_positions call as <directory>/<name>.npy, float32 or float64 as computed.
    An output of at most DUMP_MAX_ELEMENTS values is written whole, in its shape.  A larger one (the thickness maps and
    the sample / reference images of 20 positions) is written as a 1-D sample of its flattened values: DUMP_MAX_ELEMENTS
    indices drawn without replacement by numpy's default_rng(0), in increasing order -- the same indices on every run."""
    os.makedirs(directory, exist_ok=True)
    for name in DUMP_OUTPUTS:
        t = res[name]
        assert t.dtype in (torch.float32, torch.float64), (name, t.dtype)
        if t.numel() > DUMP_MAX_ELEMENTS:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_MAX_ELEMENTS, replace=False))
            t = t.reshape(-1).index_select(0, torch.as_tensor(idx, device=t.device))
        np.save(os.path.join(directory, name + ".npy"), t.cpu().numpy())


def config_dict(**extra):
    c = {"workload": WORKLOAD, "experiment": EXPERIMENT, "positions_per_step": POSITIONS * JOBS_PER_STEP, "positions_per_job": POSITIONS,
         "grid": 2048, "energies": 1, "propagation": "ray tracing (RayT)"}
    c.update(extra)
    return c


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line)

    def mark(self):
        """Samples taken from here on count (the sampler itself starts earlier: nvidia-smi needs ~0.3 s to spin up)."""
        self.first = len(self.lines)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        self.lines = self.lines[getattr(self, "first", 0):] or self.lines[-3:]
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------
# CPU side (oracle port): cpu_baseline and --impl reference
# ---------------------------------------------------------------------------------------------
def _oracle_setup():
    """The same experiment, as scalars for the oracle (values = what the shim derives from the XML)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import paresis_oracle as po
    from paresis_b200 import workspace
    from paresis_b200.hostio import tables
    os.chdir(workspace.make_workspace(tempfile.mkdtemp(prefix="paresis_cpu_")))
    energy = 52.0
    cusn, pmma, nylon = (tables.interpolate(m, [energy])[0] for m in ("CuSn", "PMMA", "Nylon"))
    setup = po.Setup(140.0, 1.6, 3.6, (1024, 1024), 6.0, 2, 30000.0, [(energy, 1.0)], 50.0, 1.2)
    mdb = {energy: ([cusn[0], pmma[0]], [cusn[1], pmma[1]])}
    sdb = {energy: ([nylon[0]], [nylon[1]])}
    sample_t = po.sample_cylinder(700.0, 30.0, setup.study_dims[0], setup.study_dims[1], setup.study_pixel_um)
    rows = workspace.synthetic_sphere_rows(0, 60000)
    return po, setup, mdb, sdb, sample_t, rows


def _oracle_position(ctx, point, seed):
    po, setup, mdb, sdb, sample_t, rows = ctx
    np.random.seed(seed)
    rng = np.random.RandomState(seed)
    mem = po.membrane_segmented(rows, 50.0, 3, setup.study_dims[0], setup.study_dims[1], setup.membrane_pixel_um, 6000.0)
    out = po.compute_rt(setup, mem, mdb, sample_t, sdb, point, poisson=rng.poisson)
    return float(out[0].sum())


_worker_ctx = None


def _worker_init():
    global _worker_ctx
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    _worker_ctx = _oracle_setup()
    _oracle_position(_worker_ctx, 1, 12345)  # warm caches (FFT plans, page faults)


def _worker_run(args):
    point, seed = args
    return _oracle_position(_worker_ctx, point, seed)


def cpu_baseline_single(positions=tuple(range(8))):
    """Scalar port on one core: image-sets/s over a bounded sample of the workload (8 positions: 10-15 s of CPU work)."""
    ctx = _oracle_setup()
    _oracle_position(ctx, 1, 999)
    t0 = time.perf_counter()
    for p in positions:
        _oracle_position(ctx, p, 100 + p)
    dt = time.perf_counter() - t0
    return {"value": len(positions) / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "%d of the 20 positions (0..%d) at the full 2048^2 grid, fp64 numpy + C oracle, %.1f s"
                      % (len(positions), len(positions) - 1, dt)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    workers = max(1, min(cores, 32))
    per_step = workers                      # bounded sample: one position per worker per step (a step takes ~10-15 s)
    with mp.get_context("fork").Pool(workers, initializer=_worker_init) as pool:
        for w in range(args.warmup):
            pool.map(_worker_run, [(1, 5000 + w * per_step + i) for i in range(per_step)])
        t0 = time.perf_counter()
        for s in range(args.steps):
            pool.map(_worker_run, [(0 if i == 0 else 1, 100 + s * per_step + i) for i in range(per_step)])
        dt = time.perf_counter() - t0
    value = per_step * args.steps / dt
    sample = "%d positions per step (one per worker process, position 0 once per step) at the full 2048^2 grid" % per_step
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(positions_per_step=per_step, note="CPU oracle port of the reference path; the reference "
                                  "itself is Python/Numba and cannot travel to the GPU box"),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# GPU side
# ---------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with torch.distributed.run --nproc-per-node N (see module docstring)")
    torch.cuda.set_device(local)
    from paresis_b200.hostio import affinity
    bound = affinity.bind_to_gpu(local)        # host threads + first-touch pinned buffers next to this rank's GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from paresis_b200 import _cabi as abi
    from paresis_b200 import geometry, transfer, workspace
    ws = workspace.make_workspace(tempfile.mkdtemp(prefix="paresis_bench_r%d_" % rank))
    workspace.enter(ws)
    import Experiment as shim

    exp_dict = dict(experimentName=EXPERIMENT, filepath=os.path.join(ws, "out", ""), overSampling=2, nbExpPoints=POSITIONS,
                    simulation_type="RayT", expID="bench", seed=1234 + rank)
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        exp = shim.Experiment(exp_dict)
    n = int(exp.exp_dict["studyDimensions"][0])
    det = int(exp.myDetector.det_param["myDimensions"][0])
    eng = exp._get_engine()
    mem = exp.myMembrane
    flush = torch.empty(256 * 1024 * 1024 // 4, device="cuda", dtype=torch.float32)
    plan = geometry.MembranePlan(mem, n, n, mem.membranePixelSize)
    thresholds = list(exp._open_bins(0))
    exp.myDetector.det_param["myBinsThersholds"] = []
    scene = exp._scene(thresholds, per_position_membrane=True)
    points = list(range(POSITIONS))
    state = {"buffers": None}

    def device_job(step, probe_label=None, events=None, slots=None):
        """20 positions in one library call, everything resident in HBM; results stay on the device."""
        np.random.seed((10_000 * rank + step) % (2 ** 32))
        offsets = [plan.draw_offsets() for _ in points]         # the reference's randint draws, in its order
        pe = None
        if probe_label is not None:
            # all positions when profiling one at a time; ONE position per step in the timed region (it runs alone
            # on the GPU for that moment, see paresis_rt_position.probe_start)
            probed = points if (slots or args.slots) == 1 else [POSITIONS // 2]
            pe = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) if p in probed else None
                  for p in points]
            events.extend(e for e in pe if e is not None)
        with abi.on_stream():
            res = eng.compute_rt_positions(scene, plan, offsets, points, sequence_base=step * POSITIONS,
                                           n_slots=slots or args.slots, probe_label=probe_label, probe_events=pe,
                                           buffers=state["buffers"], per_launch=args.per_launch if slots is None else 0)
        state["buffers"] = res["buffers"]
        return res

    def api_job(step):
        """The same job through the reference-facing API: host results, membrane map copied back."""
        np.random.seed((20_000 * rank + step + 7) % (2 ** 32))
        geometry.drop_device_tables()                       # the sphere list crosses PCIe once per job
        h0, d0 = transfer.bytes_h2d, transfer.bytes_d2h
        exp.myDetector.det_param["myBinsThersholds"] = []    # position 0 closes the last bin in place (Experiment.py:429)
        with contextlib.redirect_stdout(io.StringIO()):
            for point in range(POSITIONS):
                mem.myGeometry = []
                mem.getMyGeometry(exp.exp_dict['studyDimensions'], mem.membranePixelSize, 2, point, POSITIONS)
                res = exp.computeSampleAndReferenceImages_RT(point)
                thick = mem.myGeometry[0]                   # main.py:99 saves it
                assert thick.shape == (n, n) and res[0].shape == (1, det, det)
        return transfer.bytes_h2d - h0, transfer.bytes_d2h - d0

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- per-kernel shares (untimed, after a warm-up): which kernel dominates the step?
    device_job(-1)
    torch.cuda.synchronize()
    eng.check_flag()
    shares = profile_kernels(abi, device_job, torch)
    dominant = max(shares, key=lambda k: shares[k]["ms_per_step"])
    k_events = []

    # ---- timed region: device-resident job
    sampler = ClockSampler(local)
    sampler.start()
    jobs = args.jobs_per_step
    for w in range(args.warmup):
        for jb in range(jobs):
            device_job(100_000 + w * jobs + jb)
    barrier()
    sampler.mark()
    launches0 = abi.launches
    step_events = []
    wall0 = time.perf_counter()
    for s in range(args.steps):
        flush.zero_()                                       # L2 flush between timed steps (not timed)
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for jb in range(jobs):                              # one probed position per step, in its first job
            if jb == 0:
                last = device_job(s * jobs, dominant, k_events)
            else:
                last = device_job(s * jobs + jb)
        e1.record()
        step_events.append((e0, e1))
        if s % 8 == 7:
            torch.cuda.synchronize()                        # bound the host's lead over the GPU (event / launch queues)
    barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()
    launches = abi.launches - launches0
    dev_s = sum(a.elapsed_time(b) for a, b in step_events) * 1e-3
    eng.check_flag()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last, torch)
    k_ms = [a.elapsed_time(b) for a, b in k_events]
    t = torch.tensor([dev_s], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_s = float(t.item())
    value = world * POSITIONS * jobs * args.steps / dev_s

    # ---- e2e through the public API (host results)
    for w in range(max(1, min(args.warmup, 2))):
        api_job(3000 + w)
    barrier()
    t0 = time.perf_counter()
    h2d = d2h = 0
    for s in range(args.steps):
        h2d = d2h = 0
        for jb in range(E2E_JOBS_PER_STEP):
            a, b = api_job(s * E2E_JOBS_PER_STEP + jb)
            h2d += a; d2h += b
    barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * POSITIONS * E2E_JOBS_PER_STEP * args.steps / float(t.item())
    h2d += E2E_JOBS_PER_STEP * POSITIONS * 3 * 2 * 8          # the per-layer membrane offsets travel as kernel arguments
    ceiling = d2h_ceiling(torch, dist, world)
    e2e_gbs = e2e_value * (d2h / (E2E_JOBS_PER_STEP * POSITIONS)) / 1e9          # whole-job device->host rate of the e2e run
    sharded = energy_sharded(args, torch, dist, shim, geometry, abi, rank, world, ws)

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        alg = ALG_BYTES[dominant](n * n, det * det)
        traffic = None
        for name in ("r02_traffic.json", "r01_traffic.json"):               # dram__bytes_{read,write}.sum of one ncu --set full capture
            traffic_path = os.path.join(ROOT, "profiles", name)
            if os.path.exists(traffic_path):
                traffic = json.load(open(traffic_path)).get(dominant, {}).get("dram_bytes")
                break
        avg_ms = float(np.mean(k_ms)) if k_ms else shares[dominant]["ms_per_launch"]
        achieved = alg / (avg_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_s / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": config_dict(l2="flushed between timed steps (256 MiB write, outside the per-step events)",
                                  timing="CUDA events per step on the launching stream, max over ranks",
                                  wall_ms_per_step=wall / args.steps * 1e3, positions_in_flight=args.slots,
                                  host_cpus_bound=len(bound) if bound else None),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(d2h),
                    "positions_per_step": E2E_JOBS_PER_STEP * POSITIONS, "pinned_buffers_allocated": transfer.pinned_allocs,
                    "d2h_gbs": e2e_gbs, "d2h_ceiling": ceiling, "frac_of_d2h_ceiling": e2e_gbs / ceiling["aggregate_gbs"],
                    "note": "results are float64 images + the float32 membrane map (main.py:99) in pinned host memory: "
                            "the run is bound by the device->host link, whose ceiling is measured here with plain "
                            "cudaMemcpyAsync copies of 64 MiB buffers on all ranks at once"},
            "energy_sharded": sharded,
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": dominant, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "alg_bytes_per_launch": alg, "avg_launch_ms": avg_ms, "launches_timed": len(k_ms),
                         "note": "CUDA events around the kernel of one position per timed step; that position runs alone on "
                                 "the GPU (the other %d in flight drain first), so the interval is this kernel only" % (args.slots - 1)},
            "kernel_shares": shares,
        }
        if world == 1:
            line["splat"] = splat_roofline(abi, geometry, exp, torch, flush, peak)
            line["grid_8192"] = grid_8192(args, torch, shim, geometry, abi, ws, peak, flush)
            line["fresnel"] = fresnel_section(args, torch, shim, geometry, ws, peak)
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_single()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def splat_roofline(abi, geometry, exp, torch, flush, peak):
    """BASELINE.json's second figure: the stand-alone refraction splat (paresis_splat = fastloopNumba: read I, Dx, Dy,
    out += ; 16 algorithmic bytes per study pixel, SURVEY.md 8d) on the displacement field of one membrane position,
    at the workload grid and at a DRAM-resident one.  CUDA events per launch, L2 flushed before each, median of 10."""
    from paresis_b200 import hostmath as hm
    mem = exp.myMembrane
    pix = float(exp.exp_dict["studyPixelSize"])
    k = hm.wavenumber(52e3)
    delta = 5.97e-7        # CuSn at 52 keV (TablesDeltaBeta.xls)
    out = {"kernel": "paresis_splat", "alg_bytes_per_pixel": 16, "field": "membrane displacement of one position (object hop)",
           "unit": "GB/s", "peak": peak, "grids": {}}
    for n in (2048, 8192):
        np.random.seed(n)
        geom, _ = geometry.membrane_segmented(mem, n, n, mem.membranePixelSize, 1, mem.myPMMAThickness)
        phi = (-(k * delta) * geom.entries[0].double()).contiguous()
        dxp = torch.zeros((n + 30, n + 30), device="cuda"); dyp = torch.zeros_like(dxp)
        inten = torch.full((n, n), 7500.0, device="cuda")
        tmp = torch.zeros((n, n), device="cuda")
        abi.refract_phi(inten, phi, tmp, 3.6, 52.0, float(exp.exp_dict["magnification"]), pix, 15, dxp, dyp)
        dx = dxp[15:-15, 15:-15].contiguous(); dy = dyp[15:-15, 15:-15].contiguous()
        del dxp, dyp, phi, geom
        inten = (inten * (0.7 + 0.6 * torch.rand((n, n), device="cuda"))).contiguous()
        res = {"mean_abs_displacement_px": float((dx.abs().mean() + dy.abs().mean()).item() / 2)}
        for variant, label in ((2, "direct_red"), (3, "smem_tiles"), (4, "owner_strips"), (5, "owner_strips_accumulate")):
            for _ in range(3):
                abi.splat(inten, dx, dy, tmp, margin=15, variant=variant)
            times = []
            for _ in range(10):
                flush.zero_()
                e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
                e0.record(); abi.splat(inten, dx, dy, tmp, margin=15, variant=variant); e1.record()
                torch.cuda.synchronize()
                times.append(e0.elapsed_time(e1))
            ms = float(np.median(times))
            gbs = 16.0 * n * n / (ms * 1e-3) / 1e9
            res[label] = {"variant": variant, "avg_launch_ms": ms, "achieved": gbs, "frac": gbs / peak}
        out["grids"][str(n)] = res
        del dx, dy, inten, tmp
        torch.cuda.empty_cache()
    return out


def d2h_ceiling(torch, dist, world, mib=64, reps=24):
    """What the platform gives a plain device->host copy: one cudaMemcpyAsync per 64 MiB buffer into pinned memory, all
    ranks at the same time (the ranks of a node share the host's PCIe root / memory bandwidth)."""
    n = mib * 1024 * 1024
    dev = torch.empty(n, device="cuda", dtype=torch.uint8)
    host = [torch.empty(n, dtype=torch.uint8, pin_memory=True) for _ in range(2)]
    for h in host:
        h.copy_(dev, non_blocking=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(reps):
        host[k & 1].copy_(dev, non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    gbs = reps * n / (e0.elapsed_time(e1) * 1e-3) / 1e9
    t = torch.tensor([gbs, gbs], device="cuda", dtype=torch.float64)
    if world > 1:
        lo = t[1:].clone()
        dist.all_reduce(t[:1], op=dist.ReduceOp.SUM)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        t[1] = lo[0]
    return {"aggregate_gbs": float(t[0].item()), "min_rank_gbs": float(t[1].item()), "ranks": world, "buffer_mib": mib}


def energy_sharded(args, torch, dist, shim, geometry, abi, rank, world, ws):
    """BASELINE.json configs[2]: 4096^2, 64 energies, 20 membrane positions, the spectrum of each position sharded over
    the ranks and summed with ONE NCCL reduce per detector bin (paresis_b200/shard.py).  Strong scaling."""
    if args.skip_extras:
        return None
    import contextlib
    import io
    from paresis_b200 import shard
    positions, reps = 20, 2
    with contextlib.redirect_stdout(io.StringIO()):
        exp = shim.Experiment(dict(experimentName="B200_4096_poly64", filepath=os.path.join(ws, "out", ""), overSampling=2,
                                   nbExpPoints=positions, simulation_type="RayT", expID="shard", seed=99))
    n = int(exp.exp_dict["studyDimensions"][0])
    det = int(exp.myDetector.det_param["myDimensions"][0])
    eng, mem = exp._get_engine(), exp.myMembrane
    exp.myDetector.det_param["myBinsThersholds"] = []
    thresholds = list(exp._open_bins(0))
    reduce_events = []
    pending = [None]

    def job(rep):
        np.random.seed(777 + rep)                                # the same membrane positions on every rank
        with contextlib.redirect_stdout(io.StringIO()):
            for point in range(positions):
                # the membrane of this position, cut on every rank (no host copy of the map: nobody saves it here)
                mem.myGeometry, _ = geometry.membrane_segmented(mem, n, n, mem.membranePixelSize, point, mem.myPMMAThickness)
                scene = exp._scene(thresholds)
                # the host-side tail of a position (means + NaN guard: an all_reduce and a device->host read) is taken
                # after the NEXT position has been queued
                nxt = shard.compute_rt_energy_sharded(eng, scene, point, owner=0, sequence_base=rep * positions,
                                                      reduce_events=reduce_events if rep >= 0 else None, defer=True)
                if pending[0] is not None:
                    pending[0].finish()
                pending[0] = nxt
            pending[0].finish()
            pending[0] = None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    job(-1)
    barrier()
    launches0 = abi.launches
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for rep in range(reps):
        job(rep)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    red_ms = sum(a.elapsed_time(b) for a, b in reduce_events)
    t = torch.tensor([ms, red_ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, red_ms = float(t[0].item()), float(t[1].item())
    n_red = len(reduce_events)
    images_first, images_rest = 4, 2
    bytes_per_reduce = det * det * 4 * images_rest
    return {"workload": "4096^2 grid, 64 energies (20..83 keV), 20 membrane positions, RayT, one detector bin; energies round-robin over ranks",
            "experiment": "B200_4096_poly64", "scaling": "strong", "n_gpus": world, "metric": METRIC, "unit": UNIT,
            "value": reps * positions / (ms * 1e-3), "ms_per_position": ms / (reps * positions),
            "energies_per_rank": [len(shard.energies_of(list(range(len(exp.mySource.mySpectrum))), r, world)) for r in range(world)],
            "collective": {"op": "ncclReduce(sum, fp32) of detector-resolution partial images, one per detector bin and position" if world > 1 else "none (one rank)",
                           "reduces": n_red, "bytes_per_reduce": bytes_per_reduce, "bytes_per_reduce_first_position": det * det * 4 * images_first,
                           "reduce_ms_total": red_ms, "reduce_ms_per_position": red_ms / (reps * positions),
                           "reduce_share_of_time": red_ms / ms if ms > 0 else None,
                           "effective_gbs": (n_red * bytes_per_reduce / (red_ms * 1e-3) / 1e9) if red_ms > 0 and world > 1 else None,
                           "note": "CUDA events around dist.reduce on the compute stream: includes waiting for the slowest rank"},
            "gpu_launches": int(abi.launches - launches0), "timing": "CUDA events around %d x %d positions, max over ranks" % (reps, positions)}


def grid_8192(args, torch, shim, geometry, abi, ws, peak, flush):
    """BASELINE.json configs[4] sub-sample on one GPU: 8192^2, 8 of the 128 energies x 4 membrane positions, through the same
    many-positions call as the headline; per-kernel CUDA-event times and roofline fractions at a DRAM-resident grid."""
    if args.skip_extras:
        return None
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        exp = shim.Experiment(dict(experimentName="B200_8192_poly128", filepath=os.path.join(ws, "out", ""), overSampling=2,
                                   nbExpPoints=4, simulation_type="RayT", expID="g8k", seed=5))
    keep = list(range(0, 128, 16))
    exp.mySource.mySpectrum = [exp.mySource.mySpectrum[i] for i in keep]
    n = int(exp.exp_dict["studyDimensions"][0])
    det = int(exp.myDetector.det_param["myDimensions"][0])
    eng, mem = exp._get_engine(), exp.myMembrane
    exp.myDetector.det_param["myBinsThersholds"] = []
    thresholds = list(exp._open_bins(0))
    scene = exp._scene(thresholds, per_position_membrane=True)
    plan = geometry.MembranePlan(mem, n, n, mem.membranePixelSize)
    points = [1, 2, 3, 4]
    state = {"buffers": None}

    def job(step, probe_label=None, events=None, slots=2):
        np.random.seed(4000 + step)
        offsets = [plan.draw_offsets() for _ in points]
        pe = None
        if probe_label is not None:
            pe = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in points]
            events.extend(pe)
        with abi.on_stream():
            res = eng.compute_rt_positions(scene, plan, offsets, points, sequence_base=step * 8, n_slots=slots,
                                           probe_label=probe_label, probe_events=pe, buffers=state["buffers"])
        state["buffers"] = res["buffers"]

    job(-1)
    torch.cuda.synchronize()
    eng.check_flag()
    times = []
    for step in range(3):
        flush.zero_()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); job(step); e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    ms = float(np.median(times))
    kernels = {}
    px, dpx, n_e = float(n) * n, float(det) * det, len(keep)
    # algorithmic bytes per launch; the object hop of a polychromatic bin runs 4 energies per launch (12 + 8/G B/px per energy)
    alg = {"raster_spheres": 4.0 * px, "refract_membrane_hop": 8.0 * px, "refract_sample_ref_hop": (12.0 * 4 + 8.0) * px,
           "detect": 2 * (4.0 * px + 4.0 * dpx)}
    for k, label in enumerate(("raster_spheres", "refract_membrane_hop", "refract_sample_ref_hop", "detect")):
        ev = []
        job(-3 - k, label, ev, slots=1)
        torch.cuda.synchronize()
        v = float(np.mean([a.elapsed_time(b) for a, b in ev]))
        gbs = alg[label] / (v * 1e-3) / 1e9
        kernels[label] = {"ms_per_launch": v, "alg_bytes_per_launch": alg[label], "achieved_gbs": gbs, "frac": gbs / peak}
    del state, eng, exp
    geometry.drop_device_tables()
    torch.cuda.empty_cache()
    return {"workload": "8192^2 grid, 8 of the 128 energies (20, 28, ... 76 keV) x 4 membrane positions, RayT, one detector bin",
            "experiment": "B200_8192_poly128", "positions_per_s": len(points) / (ms * 1e-3), "ms_per_position": ms / len(points),
            "ms_per_energy_and_position": ms / len(points) / n_e, "kernels": kernels, "peak_gbs": peak,
            "note": "per-kernel rows: CUDA events around the first launch of that kind in each position, positions one at a time; "
                    "the object hop is the 4-energy group kernel of a polychromatic bin"}


def fresnel_section(args, torch, shim, geometry, ws, peak):
    """BASELINE.json configs[3]: the Fresnel-propagator model (Experiment.py:279-405, wavePropagation :219-252) at 4096^2 and
    8192^2, device time per membrane position (three propagations: reference beam, membrane->object, object->detector).
    A propagation is two per-axis circular convolutions of period N + 30 (csrc/fresnel.cu): per axis one kernel that takes
    a line through two power-of-two transforms in shared memory (fresnel_lines.cuh) and one that adds the reflect-margin
    terms and transposes.  Roofline entry: the algorithmic traffic of that formulation, one read + one write of the complex
    wave per kernel = 4 x 16 B per pixel and propagation, against the time of the whole position (which also holds the two
    transmissions, the |.|^2 accumulation and the detector)."""
    if args.skip_extras:
        return None
    import contextlib
    import io
    out = {"alg_bytes_per_pixel_per_propagation": 64, "propagations_per_position": 3, "line_transform": "in shared memory, M = 2N",
           "peak_gbs": peak, "grids": {}}
    for n in (4096, 8192):
        with contextlib.redirect_stdout(io.StringIO()):
            exp = shim.Experiment(dict(experimentName="B200_%d_mono" % n, filepath=os.path.join(ws, "out", ""), overSampling=2,
                                       nbExpPoints=4, simulation_type="Fresnel", expID="fr", seed=3))
        eng, mem = exp._get_engine(), exp.myMembrane
        exp.myDetector.det_param["myBinsThersholds"] = []
        thresholds = list(exp._open_bins(0))
        np.random.seed(n)
        times = []
        for point in (1, 2, 3, 4):
            mem.myGeometry, _ = geometry.membrane_segmented(mem, n, n, mem.membranePixelSize, point, mem.myPMMAThickness)
            scene = exp._scene(thresholds)
            torch.cuda.synchronize()
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(); eng.compute_fresnel(scene, point); e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        ms = float(np.median(times[1:]))
        gbs = 3 * 64.0 * float(n) ** 2 / (ms * 1e-3) / 1e9
        out["grids"][str(n)] = {"ms_per_position": ms, "positions_per_s": 1e3 / ms, "period": n + 30, "line_transform_length": 2 * n,
                                "achieved_gbs": gbs, "frac": gbs / peak}
        del eng, exp, scene
        geometry.drop_device_tables()
        torch.cuda.empty_cache()
    return out


def profile_kernels(abi, job, torch):
    """Untimed jobs, one position in flight, with CUDA events around one kernel class at a time (the probe of
    paresis_rt_run_positions): ms per launch and per 20-position step."""
    out = {}
    launches_per_step = {"raster_spheres": POSITIONS, "refract_membrane_hop": POSITIONS + 1,
                         "refract_sample_ref_hop": POSITIONS, "detect": POSITIONS}
    for k, label in enumerate(("raster_spheres", "refract_membrane_hop", "refract_sample_ref_hop", "detect")):
        ev = []
        job(-3 - k, label, ev, slots=1)
        torch.cuda.synchronize()
        v = [a.elapsed_time(b) for a, b in ev][1:]      # position 0 carries the extra images: steady state only
        out[label] = {"ms_per_step": float(np.mean(v)) * launches_per_step[label], "ms_per_launch": float(np.mean(v)),
                      "launches": launches_per_step[label]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=("b200", "reference"))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--slots", type=int, default=SLOTS, help="membrane positions in flight on the GPU")
    ap.add_argument("--jobs-per-step", type=int, default=JOBS_PER_STEP, help="20-position jobs per timed step")
    ap.add_argument("--skip-extras", action="store_true", help="headline only: no splat / 8192^2 / energy-sharded sections")
    ap.add_argument("--per-launch", type=int, default=PER_LAUNCH, help="membrane positions per kernel launch (0: one launch per position, on --slots streams)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed job as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.steps < 1):
        ap.error("--dump-outputs needs the GPU path (--impl b200) and at least one timed step")
    if args.dump_outputs:
        args.dump_outputs = os.path.abspath(args.dump_outputs)     # the run changes into a temporary workspace
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
