"""Cost of a scattering (dark-field) sample as one library call per position (paresis_df_run), and of the energy-sharded
call on such a sample.

    python tools/df_bench.py single OUT.json
    torchrun --nproc_per_node N tools/df_bench.py scaling OUT.json     (N = 1, 2, 4, 8; plain python = 1 GPU)

single : ms per membrane position (noise off) of B200_2048_mono and B200_4096_poly64 (64 energies, one detector bin) with
         the sample made of Lung: compute_rt against the per-energy Python loop it replaced (restated in
         tests/test_gpu_dark_field_run.py), alternated in one process: one warm-up position, then 5 positions, each timed
         before and after in turn; medians.  CUDA events around the call, the sample and reference images read to the
         host on both sides (the loop hands back host images).  The images of the two are compared too.
scaling: ms per position of B200_4096_poly64 with Lung through shard.compute_rt_energy_sharded, energies round-robin over
         the ranks, one NCCL reduce per bin (+ one for the dark-field map at position 0); 1 warm-up + 4 timed positions
         (membrane cut included), deferred finish as bench.py runs; max over ranks.
OUT.json is a JSON object; each run adds its own entry ("single", or "scaling_<N>") and keeps the others.  The card's
name and power limit are read in the same run.
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


def card(index):
    q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or "nvidia-smi unavailable"


def experiment(shim, name, positions):
    """The experiment with its sample made of Lung, one detector bin."""
    with contextlib.redirect_stdout(io.StringIO()):
        e = shim.Experiment(dict(experimentName=name, filepath="x/", overSampling=2, nbExpPoints=positions,
                                 simulation_type="RayT", expID="d", poissonNoise=False, seed=3))
        smp = e.mySampleofInterest
        smp.myMaterials = ["Lung"] * len(smp.myMaterials)
        smp.delta, smp.beta = [], []
        smp.getDeltaBeta(e.mySource.mySpectrum)
    e.myDetector.det_param["myBinsThersholds"] = []
    return e, list(e._open_bins(0))


def new_membrane(e, point):
    mem = e.myMembrane
    n = int(e.exp_dict["studyDimensions"][0])
    mem.myGeometry, _ = geometry.membrane_segmented(mem, n, n, mem.membranePixelSize, point, mem.myPMMAThickness)


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def single(shim):
    from test_gpu_dark_field_run import _old_loop
    out = {}
    for name in ("B200_2048_mono", "B200_4096_poly64"):
        e, thresholds = experiment(shim, name, 6)
        eng = e._get_engine()
        np.random.seed(11)
        times = {"before": [], "after": []}
        diff = []

        def new_call(scene, point):
            res = eng.compute_rt(scene, point)
            return {k: res[k].cpu().numpy() for k in ("sample", "reference")}

        for point in range(6):
            new_membrane(e, point + 1)
            scene = e._scene(thresholds)
            with contextlib.redirect_stdout(io.StringIO()):
                before = timed(lambda: _old_loop(e, scene, point + 1))
                old = _old_loop(e, scene, point + 1)
            after = timed(lambda: new_call(scene, point + 1))
            new = new_call(scene, point + 1)
            diff.append(max(float(np.linalg.norm(new[k].astype(np.float64) - old[k]) / np.linalg.norm(old[k]))
                            for k in ("sample", "reference")))
            if point:                                    # position 0 of the loop warms up both
                times["before"].append(before)
                times["after"].append(after)
        out[name] = dict(energies=len(e.mySource.mySpectrum),
                         ms_per_position={k: round(float(np.median(v)), 3) for k, v in times.items()},
                         all_ms={k: [round(x, 3) for x in v] for k, v in times.items()},
                         image_rel_l2_new_vs_before=max(diff))
        del eng, e
        geometry.drop_device_tables()
        torch.cuda.empty_cache()
    return dict(card=card(0), workload="sample made of Lung, noise off, positions 2..6 after one warm-up", grids=out)


def scaling(shim, rank, world):
    positions = 5
    e, thresholds = experiment(shim, "B200_4096_poly64", positions)
    eng = e._get_engine()
    reduce_events = []
    np.random.seed(777)                                  # the same membrane positions on every rank

    def job(points, events):
        pending = None
        for point in points:
            new_membrane(e, point)
            nxt = shard.compute_rt_energy_sharded(eng, e._scene(thresholds), point, owner=0, reduce_events=events, defer=True)
            if pending is not None:
                pending.finish()
            pending = nxt
        pending.finish()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    job([1], None)                                       # warm-up
    barrier()
    ms = timed(lambda: job(range(2, positions + 1), reduce_events))
    barrier()
    red = sum(a.elapsed_time(b) for a, b in reduce_events)
    t = torch.tensor([ms, red], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total, red = float(t[0]), float(t[1])
    n_e, timed_positions = len(e.mySource.mySpectrum), positions - 1
    return dict(card=card(rank), n_gpus=world, experiment="B200_4096_poly64, sample made of Lung", model="RayT", energies=n_e,
                energies_per_rank=[len(shard.energies_of(list(range(n_e)), r, world)) for r in range(world)],
                timed_positions=timed_positions, ms_per_position=round(total / timed_positions, 3),
                reduce_ms_per_position=round(red / timed_positions, 4), reduces=len(reduce_events),
                timing="CUDA events around positions 2..5 (membrane cut included), max over ranks")


def main():
    mode, out = sys.argv[1], os.path.abspath(sys.argv[2])
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    workspace.enter(workspace.make_workspace(tempfile.mkdtemp()))
    import Experiment as shim
    res = single(shim) if mode == "single" else scaling(shim, rank, world)
    if world > 1:
        dist.destroy_process_group()
    if rank != 0:
        return
    key = "single" if mode == "single" else "scaling_%d" % world
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
