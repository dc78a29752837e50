"""Cost of samples with more materials than a hop takes (paresis_mix_maps, engine.ImageFormation.mixed_sample).

    python tools/mix_bench.py [out.json]

1. Kernel time of paresis_mix_maps at 8192^2 with 2, 6 and 13 material maps, both outputs (phase and attenuation map): CUDA
   events around 50 launches after 10 warm-up launches.  The inputs (268 MB a map) exceed the 126 MB L2, so each launch
   reads them from HBM.  Algorithmic traffic = (n_maps + 2) x 4 bytes a pixel; its rate is stated against the measured
   copy bandwidth of BASELINE.md section 4 (6 539.5 GB/s, read + write).
2. Time per membrane position of B200_2048_mono (2048^2, mono) through compute_rt_positions (20 positions, 4 per launch, as
   bench.py runs it) with its one-material sample and with a six-material sample (five maps and a flat one) on the same
   grid; the mixed maps are made in the warm-up call, as they are once per engine.  Three alternating repeats, median.
The card's name and power limit are read in the same run.
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
sys.path.insert(0, ROOT)
from paresis_b200 import engine, geometry, workspace  # noqa: E402
from paresis_b200 import _cabi as abi  # noqa: E402
import torch  # noqa: E402

COPY_GBS = 6539.5     # BASELINE.md section 4: measured device copy bandwidth (read + write), B200


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or "nvidia-smi unavailable"


def kernel_times(n=8192, launches=50, warmup=10):
    out = []
    p_map = torch.empty((n, n), device="cuda")
    b_map = torch.empty_like(p_map)
    for n_maps in (2, 6, 13):
        maps = [torch.rand((n, n), device="cuda") * 1e-3 for _ in range(n_maps)]
        w = [[1.0 / (m + 1) for m in range(n_maps)], [1.0 / (m + 2) for m in range(n_maps)]]
        for _ in range(warmup):
            abi.mix_maps(maps, w, [0.0, 1e-6], [p_map, b_map])
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(launches):
            abi.mix_maps(maps, w, [0.0, 1e-6], [p_map, b_map])
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / launches
        gbs = (n_maps + 2) * 4.0 * n * n / (ms * 1e-3) / 1e9
        out.append(dict(n_maps=n_maps, pixels=n * n, ms=round(ms, 4), algorithmic_GBs=round(gbs, 1),
                        fraction_of_copy_bandwidth=round(gbs / COPY_GBS, 3)))
        del maps
    return out


def position_times(n_pos=20, repeats=3):
    ws = workspace.make_workspace(tempfile.mkdtemp())
    workspace.enter(ws)
    import Experiment as shim
    from paresis_b200.hostio import tables
    d = dict(experimentName="B200_2048_mono", filepath="x/", overSampling=2, nbExpPoints=n_pos, simulation_type="RayT",
             expID="m", poissonNoise=False, returnDisplacement=False)
    with contextlib.redirect_stdout(io.StringIO()):
        e = shim.Experiment(d)
    n = int(e.exp_dict["studyDimensions"][0])
    mem = e.myMembrane
    thresholds = list(e._open_bins(0))
    single = e._scene(thresholds, per_position_membrane=True)
    six = e._scene(thresholds, per_position_membrane=True)
    energy = e.mySource.mySpectrum[0][0]
    pix = e.exp_dict["studyPixelSize"]
    yy, xx = np.meshgrid(np.arange(n), np.arange(n))
    six.sample = []
    for m, (name, cx, cy, r) in enumerate([("Muscle", .5, .5, .45), ("Adipose", .35, .4, .2), ("Bone", .6, .62, .12),
                                           ("PMMA", .3, .75, .15), ("Nylon", .7, .25, .1), ("SolidWater", 0, 0, 0)]):
        (dl, bl), = tables.interpolate(name, [energy])
        if r == 0:
            t = torch.full((n, n), 40e-6, device="cuda")
        else:
            h = 2 * np.sqrt(np.maximum((r * n) ** 2 - (xx - cx * n) ** 2 - (yy - cy * n) ** 2, 0.0)) * pix * 1e-6
            t = torch.as_tensor(h.astype(np.float32), device="cuda")
        six.sample.append(engine.Layer(t, {energy: dl}, {energy: bl}))
    eng = e._get_engine()
    assert eng.sample_fits(single, with_membrane=True) and not eng.sample_fits(six, with_membrane=True)
    plan = geometry.MembranePlan(mem, n, n, mem.membranePixelSize)
    np.random.seed(0)
    offsets = [plan.draw_offsets() for _ in range(n_pos)]
    points = list(range(1, n_pos + 1))

    def run(scene):
        eng.compute_rt_positions(scene, plan, offsets, points, n_slots=4, per_launch=4, want_means=False)

    times = {"single": [], "six": []}
    for name, scene in (("single", single), ("six", six)):
        run(scene)                      # warm-up (and, for six, the mixed maps of the energy)
    torch.cuda.synchronize()
    for _ in range(repeats):
        for name, scene in (("single", single), ("six", six)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run(scene)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / n_pos)
    eng.check_flag()
    return dict(grid=n, positions=n_pos, per_launch=4,
                ms_per_position={k: round(float(np.median(v)), 4) for k, v in times.items()},
                all_ms_per_position={k: [round(x, 4) for x in v] for k, v in times.items()})


def main():
    out = os.path.abspath(sys.argv[1]) if len(sys.argv) > 1 else None     # position_times() changes directory
    torch.cuda.set_device(0)
    res = dict(card=card(), copy_bandwidth_GBs=COPY_GBS, kernel=kernel_times())
    torch.cuda.empty_cache()
    res["positions"] = position_times()
    line = json.dumps(res)
    print(line)
    if out:
        with open(out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
