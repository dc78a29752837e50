"""Cost of a Fresnel scan as one library call for many membrane positions (compute_fresnel_positions,
paresis_fresnel_run_positions) against the position-by-position loop (geometry.membrane_segmented + compute_fresnel per
position, as bench.py's fresnel_section runs it).

    python tools/fresnel_positions_bench.py OUT.json
    torchrun --nproc_per_node N tools/fresnel_positions_bench.py OUT.json      (each rank: its shard.positions_of share)

Per grid (B200_2048_mono, B200_4096_mono, B200_8192_mono run as Fresnel: one energy, Poisson noise on), 20 positions per
call, never position 0:
  - before any timing, the images of three positions from the two paths are compared (same seed, same offsets): they
    must be bit for bit equal;
  - the loop and the new call at 1, 2 and 3 slots, each warmed up once, then alternated in one process 5 times; CUDA
    events around each call (the loop's host round-trips included, the new call's outputs written into buffers kept
    from the warm-up); median ms per position and the spread (min, max) of the 5.
With torchrun every rank times its share of a 20-position call per rank (positions rank, rank + N, ...) with the default
slots and reports positions/s; OUT.json then gets "ranks_<N>".  The card's name and power limit are read in the same run.
"""
import contextlib
import io
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")]
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from paresis_b200 import geometry, shard, workspace  # noqa: E402

POSITIONS = 20
REPEATS = 5
SLOTS = (1, 2, 3)
DEFAULT_SLOTS = 2          # compute_fresnel_positions' default


def card(index):
    q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or "nvidia-smi unavailable"


def experiment(shim, n):
    with contextlib.redirect_stdout(io.StringIO()):
        e = shim.Experiment(dict(experimentName="B200_%d_mono" % n, filepath="x/", overSampling=2, nbExpPoints=POSITIONS + 1,
                                 simulation_type="Fresnel", expID="f", poissonNoise=True, seed=3))
    e.myDetector.det_param["myBinsThersholds"] = []
    return e, list(e._open_bins(0))


class Grid:
    def __init__(self, shim, n):
        self.n = n
        self.e, self.thresholds = experiment(shim, n)
        self.eng = self.e._get_engine()
        mem = self.e.myMembrane
        self.mem = mem
        self.plan = geometry._plan(mem, n, n, mem.membranePixelSize)
        self.scene = self.e._scene(self.thresholds, per_position_membrane=True)
        self.buffers = {}            # outputs of a call, by number of positions: reused as a scan would

    def loop(self, points):
        """The per-position flow: cut the membrane, then one compute_fresnel (which reads its sums on the host)."""
        mem, n, out = self.mem, self.n, []
        for point in points:
            mem.myGeometry, _ = geometry.membrane_segmented(mem, n, n, mem.membranePixelSize, point, mem.myPMMAThickness)
            out.append(self.eng.compute_fresnel(self.e._scene(self.thresholds), point))
        return out

    def positions(self, points, slots):
        offsets = [self.plan.draw_offsets() for _ in points]
        res = self.eng.compute_fresnel_positions(self.scene, self.plan, offsets, points, n_slots=slots,
                                                 buffers=self.buffers.get(len(points)))
        self.buffers[len(points)] = res["buffers"]
        return res

    def agree(self):
        points = [1, 2, 3]
        np.random.seed(self.n)
        loop = self.loop(points)
        np.random.seed(self.n)
        res = self.positions(points, DEFAULT_SLOTS)
        worst, equal = 0.0, True
        for p in range(len(points)):
            for k in ("sample", "reference"):
                a, b = res[k][p].cpu().numpy(), loop[p][k].cpu().numpy()
                equal &= bool(np.array_equal(a, b))
                d = np.linalg.norm(a.astype(np.float64) - b) / np.linalg.norm(b.astype(np.float64))
                worst = max(worst, float(d))
        if not equal:
            raise SystemExit("B200_%d_mono: the two paths' images differ (rel L2 %.3e)" % (self.n, worst))
        return worst


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def single(shim):
    out = {}
    points = list(range(1, POSITIONS + 1))
    for n in (2048, 4096, 8192):
        g = Grid(shim, n)
        rel = g.agree()
        runs = {"loop": lambda: g.loop(points)}
        for k in SLOTS:
            runs["slots_%d" % k] = (lambda k=k: g.positions(points, k))
        for fn in runs.values():                                  # warm-up: transfer kernels, slot plans, buffers
            fn()
        ms = {name: [] for name in runs}
        for _ in range(REPEATS):
            for name, fn in runs.items():
                ms[name].append(timed(fn) / POSITIONS)
        med = {name: round(float(np.median(v)), 4) for name, v in ms.items()}
        out[str(n)] = dict(ms_per_position=med, spread_ms=({name: [round(min(v), 4), round(max(v), 4)] for name, v in ms.items()}),
                           speedup_vs_loop={name: round(med["loop"] / med[name], 3) for name in med if name != "loop"},
                           images_rel_l2_positions_vs_loop=rel, images_bitwise_equal=True)
        del g
        geometry.drop_device_tables()
        torch.cuda.empty_cache()
    return dict(card=card(0), workload="B200_<N>_mono as Fresnel, one energy, Poisson noise on, %d positions per call "
                                       "(never position 0), median of %d alternated runs after one warm-up" % (POSITIONS, REPEATS),
                grids=out)


def ranks(shim, rank, world):
    out = {}
    for n in (2048, 4096, 8192):
        g = Grid(shim, n)
        mine = [p + 1 for p in shard.positions_of(POSITIONS * world, rank, world)]
        np.random.seed(n + rank)
        g.positions(mine, DEFAULT_SLOTS)                         # warm-up
        ms = []
        for _ in range(REPEATS):
            if world > 1:
                dist.barrier()
            ms.append(timed(lambda: g.positions(mine, DEFAULT_SLOTS)))
        t = torch.tensor([float(np.median(ms))], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out[str(n)] = dict(positions_per_rank=len(mine), slowest_rank_ms=round(float(t[0]), 3),
                           positions_per_s_per_rank=round(len(mine) / (float(t[0]) * 1e-3), 2))
        del g
        geometry.drop_device_tables()
        torch.cuda.empty_cache()
    return dict(card=card(torch.cuda.current_device()), n_gpus=world, slots=DEFAULT_SLOTS, grids=out,
                timing="CUDA events around one call per rank, median of %d, max over ranks" % REPEATS)


def main():
    out = os.path.abspath(sys.argv[1])
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    workspace.enter(workspace.make_workspace(tempfile.mkdtemp()))
    import Experiment as shim
    if "RANK" in os.environ:
        key, res = "ranks_%d" % world, ranks(shim, rank, world)
    else:
        key, res = "single", single(shim)
    if world > 1:
        dist.destroy_process_group()
    if rank != 0:
        return
    data = {}
    if os.path.exists(out):
        with open(out) as fh:
            data = json.load(fh)
    data[key] = res
    with open(out, "w") as fh:
        json.dump(data, fh, indent=1, sort_keys=True)
    print(json.dumps({key: res}))


if __name__ == "__main__":
    main()
