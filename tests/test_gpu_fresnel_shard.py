"""The Fresnel model as one library call per position (paresis_fresnel_run) and spread over GPUs by energy
(shard.compute_fresnel_energy_sharded).

Checked here:
  - argument checks of paresis_fresnel_run, before any CUDA call;
  - compute_fresnel against the per-energy loop it replaces, restated below with the stand-alone pieces (transmit_wave,
    FresnelPlan.convolve, mean), noise off: images, mean_energy, and the per-energy sums of the reference beam that the
    propagation now forms itself (against fp64 sums, and exactly against the accumulator of a lone energy);
  - the same images against the fp64 oracle;
  - the energy-sharded call against the single call at world size 1 (in process) and 2 (NCCL, two GPUs).
Cases: one energy, two detector bins of three energies, a sample of six materials (mixed maps), and a grid whose line
length takes the cuFFT path of the propagator instead of the in-shared-memory transform.
"""
import ctypes
import importlib
import os
import socket

import numpy as np
import pytest

import paresis_oracle as po
from conftest import rel_l2

torch = pytest.importorskip("torch")

TOL_OLD = 1e-6     # against the loop it replaces: only the global phase of the intensity-only hops differs (fp32 rounding)
TOL_ORACLE = 1e-5
CASES = ["Small_sphere_mono", "B200_small_poly3", "Small_six_materials_poly3", "cufft_grid"]


# ------------------------------------------------------------------ argument checks (no device)
def _host_job(abi, n_membrane=1, n_sample=1, plan=16, kernels=16, membrane=True):
    vp = ctypes.c_void_p
    mem = (abi.WaveLayer * max(n_membrane, 1))()
    for m in mem:
        m.thickness = 16
    en = (abi.FresnelEnergy * 1)()
    en[0].membrane_host = mem if membrane else None
    en[0].n_membrane = n_membrane
    for m in range(min(n_sample, abi.MAX_LAYERS)):
        en[0].sample[m].thickness = 16
    en[0].n_sample = n_sample
    en[0].reference = en[0].to_object = en[0].to_detector = kernels
    job = abi.FresnelJob()
    job.plan = plan
    job.n_energies, job.energies_host = 1, en
    job.wave_a = job.wave_b = job.acc_sample = job.acc_ref = vp(16).value
    return job, (mem, en)


def test_fresnel_run_rejects_bad_arguments():
    from paresis_b200 import _cabi as abi
    lib = abi.lib

    def rejects(job, msg):
        assert lib.paresis_fresnel_run(ctypes.byref(job) if job is not None else None, None) == 2
        assert msg in lib.paresis_last_error(), lib.paresis_last_error()

    rejects(None, b"null job")
    job, keep = _host_job(abi, plan=None)
    rejects(job, b"null plan")
    job, keep = _host_job(abi, membrane=False)
    rejects(job, b"no membrane layer")
    job, keep = _host_job(abi, n_membrane=0)
    rejects(job, b"no membrane layer")
    job, keep = _host_job(abi)
    keep[0][0].thickness = None
    rejects(job, b"null membrane map")
    job, keep = _host_job(abi, n_sample=0)
    rejects(job, b"sample layers")
    job, keep = _host_job(abi, n_sample=abi.MAX_LAYERS + 1)
    rejects(job, b"sample layers")
    job, keep = _host_job(abi)
    keep[1][0].sample[0].thickness = None
    rejects(job, b"null sample map")
    job, keep = _host_job(abi, kernels=None)
    rejects(job, b"null transfer kernel")
    job, keep = _host_job(abi)
    job.wave_b = None
    rejects(job, b"null wave or accumulator")
    job, keep = _host_job(abi)
    job.first_point = 1
    rejects(job, b"null wave or accumulator")            # position 0 needs the propagation accumulator
    job, keep = _host_job(abi)
    job.out_sample = 16
    rejects(job, b"incomplete detector outputs")
    job, keep = _host_job(abi)
    job.energies_host, job.n_energies = None, 1
    rejects(job, b"no energies")


@pytest.mark.gpu
def test_fresnel_run_rejects_a_kernel_of_another_plan():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from paresis_b200 import _cabi as abi, hostmath as hm
    plan, other = abi.FresnelPlan(64, 64, 15), abi.FresnelPlan(48, 48, 15)
    hx, hy, _ = hm.fresnel_vectors(48, 48, 15, (48, 48), 1.0, 1.0, 52.0, 1.5)
    kern = other.kernel(torch.as_tensor(hx, device="cuda"), torch.as_tensor(hy, device="cuda"))
    job, keep = _host_job(abi, plan=plan._h.value, kernels=kern._h.value)
    assert abi.lib.paresis_fresnel_run(ctypes.byref(job), None) == 2
    assert b"prepared for a plan of another size" in abi.lib.paresis_last_error()


# ------------------------------------------------------------------ scenes
def _blob(shape, cx, cy, r_px, pix_um):
    x = np.arange(shape[0])[:, None] - cx
    y = np.arange(shape[1])[None, :] - cy
    return 2 * np.sqrt(np.maximum(r_px ** 2 - x ** 2 - y ** 2, 0.0)) * pix_um * 1e-6


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from paresis_b200 import workspace
    from paresis_b200.hostio import imageio
    from test_gpu_many_materials import MATERIALS, _six_maps
    ws = workspace.make_workspace(str(tmp_path_factory.mktemp("ws_fresnel")))
    folder = os.path.join(ws, "Samples", "ManyMaterials")
    os.makedirs(folder)
    pix = 6.0 / 2 / (145.2 / 141.6)
    for m, t in enumerate(_six_maps((192, 256), pix)):
        imageio.write_tiff(os.path.join(folder, "m%d_%s.tif" % (m, MATERIALS[m])), t)
    old = os.getcwd()
    workspace.enter(ws)
    yield importlib.import_module("Experiment")
    os.chdir(old)


class Case:
    """A scene, the engine that runs it, and the oracle on the same (fp32-rounded) maps, for membrane positions 0, 1."""

    def __init__(self, shim, name, noise=False):
        self.name = name
        if name == "cufft_grid":
            self._synthetic(noise)
            return
        d = dict(experimentName=name, filepath="unused/", overSampling=2, nbExpPoints=2, simulation_type="Fresnel",
                 expID="t", poissonNoise=noise, seed=11)
        self.e = e = shim.Experiment(d)
        self.thresholds = list(e._open_bins(0))
        self.eng = e._get_engine()
        self.scene = None

    def _synthetic(self, noise):
        """100 x 90 study grid: convolution lengths 200 and 180 (not powers of two), so both axes take the cuFFT path."""
        from paresis_b200 import engine
        self.e = None
        det, os_, det_pix = (50, 45), 2, 6.0
        self.setup = s = po.Setup(140.0, 1.6, 3.6, det, det_pix, os_, 30000.0, [(40.0, 0.5), (52.0, 0.3), (60.0, 0.2)],
                                  50.0, 1.2, energy_sampling=1, bin_thresholds=[45.0])
        self.shape = s.study_dims
        rng = np.random.default_rng(4)
        self.energies = [en for en, _ in s.spectrum]
        self.mem_db = {en: ([5.97e-7 * (52 / en) ** 2, 9.85e-8 * (52 / en) ** 2], [5.37e-9 * (52 / en) ** 3, 3.16e-12])
                       for en in self.energies}
        self.smp_db = {en: ([9.85e-8 * (52 / en) ** 2], [3.16e-12 * (52 / en) ** 3]) for en in self.energies}
        self.noise = noise
        # grain maps of two positions: 40 caps of 3-8 pixels at random centres
        self.mem_maps = [sum(_blob(self.shape, *rng.uniform((0, 0), self.shape), rng.uniform(3, 8), s.study_pixel_um)
                             for _ in range(40)).astype(np.float32) for _ in range(2)]
        self.smp_map = _blob(self.shape, 48, 41, 35, s.study_pixel_um).astype(np.float32)
        dev = dict(device="cuda", dtype=torch.float32)
        self.eng = engine.ImageFormation(self.shape, os_, det, seed=11, poisson=noise)
        smp = [engine.Layer(torch.as_tensor(self.smp_map, **dev), *self._coeffs(self.smp_db, 0))]
        self._smp_layers = smp
        self.thresholds = list(s.thresholds)
        self._scene_for = None

    def _coeffs(self, db, m):
        return {en: db[en][0][m] for en in self.energies}, {en: db[en][1][m] for en in self.energies}

    def position(self, point):
        """New membrane for ``point`` (main.py:63-71); -> the scene."""
        from paresis_b200 import engine
        if self.e is None:
            grains = self.mem_maps[point % 2]
            dev = dict(device="cuda", dtype=torch.float32)
            membrane = [engine.Layer(torch.as_tensor(grains, **dev), *self._coeffs(self.mem_db, 0)),
                        engine.Layer(6e-3, *self._coeffs(self.mem_db, 1))]
            s = self.setup
            self.scene = engine.Scene(s.study_dims, s.study_pixel_um, s.os, s.det_dims, s.det_pixel_um, s.psf_sigma, s.d1, s.d2,
                                      s.d3, s.mean_shot_count, s.spectrum, s.source_size_um, s.energy_sampling,
                                      self.thresholds, membrane, self._smp_layers)
            return self.scene
        np.random.seed(21 + point)
        mem = self.e.myMembrane
        mem.myGeometry = []
        mem.getMyGeometry(self.e.exp_dict['studyDimensions'], mem.membranePixelSize, 2, point, 2)
        self.scene = self.e._scene(self.thresholds)
        return self.scene

    def oracle(self, point):
        if self.e is None:
            grains = self.mem_maps[point % 2].astype(np.float64)
            mem_t = np.array([grains, np.full(self.shape, 6e-3)])
            return po.compute_fresnel(self.setup, mem_t, self.mem_db, self.smp_map[None].astype(np.float64), self.smp_db, point)
        e = self.e
        det, src = e.myDetector.det_param, e.mySource.source_dict
        setup = po.Setup(e.exp_dict['distSourceToMembrane'], e.exp_dict['distMembraneToObject'],
                         e.exp_dict['distObjectToDetector'], det['myDimensions'], det['myPixelSize'], 2,
                         e.exp_dict['meanShotCount'], list(e.mySource.mySpectrum), src["mySize"], det['myPSF'],
                         energy_sampling=src["myEnergySampling"], bin_thresholds=self.thresholds[:-1])
        energies = [en for en, _ in e.mySource.mySpectrum]

        def db(obj):
            return {en: ([dict(obj.delta[m]).get(en, 0.0) for m in range(len(obj.delta))],
                         [dict(obj.beta[m]).get(en, 0.0) for m in range(len(obj.beta))]) for en in energies}
        mem, smp = e.myMembrane, e.mySampleofInterest
        return po.compute_fresnel(setup, np.asarray(mem.myGeometry).astype(np.float64), db(mem),
                                  np.asarray(smp.myGeometry).astype(np.float64), db(smp), point)


def _old_chain(eng, s, point_num, sums=True):
    """The per-energy loop compute_fresnel ran before paresis_fresnel_run (Experiment.py:279-405), from the stand-alone
    pieces.  Noise off.  -> images (device), mean_energy, fp64 sum of each energy's |reference beam|^2 (``sums``: one
    more propagation per energy, which the loop itself did not run; else None)."""
    from paresis_b200 import _cabi as abi, hostmath as hm
    from paresis_b200.engine import IMAGES
    eng._fresnel_setup()
    first = point_num == 0
    f32 = dict(device=eng.device, dtype=torch.float32)
    acc = {k: torch.zeros((eng.nx, eng.ny), **f32) for k in IMAGES}
    one = torch.empty((eng.nx, eng.ny), **f32) if sums else None
    w_a, w_b = (torch.empty((eng.nx, eng.ny), device=eng.device, dtype=torch.complex64) for _ in range(2))
    nb = len(s.thresholds)
    out = {k: torch.empty((nb, eng.det_x, eng.det_y), **f32) for k in IMAGES[:4 if first else 2]}
    means = torch.zeros(len(s.spectrum), device=eng.device, dtype=torch.float64)
    per_energy = []
    mag_mem_obj = (s.d1 + s.d2) / s.d1
    ibin, white_sum, bin_starts = 0, 0.0, {0}
    fits = eng.sample_fits(s, with_membrane=False)
    for ie, (energy, flux) in enumerate(s.spectrum):
        k = hm.wavenumber(energy * 1000)
        i0 = s.mean_shot_count / s.os ** 2 * flux * s.common_factor(energy)
        amp = float(np.sqrt(i0 * s.plate_factor(energy)))
        mem_maps, mem_ub, _ = eng._split(s.membrane, energy)
        smp_maps = eng._sample_layers(s, energy, fits)
        abi.transmit_wave(None, amp * np.exp(-k * mem_ub), [t for t, _, _ in mem_maps], [k * b for _, _, b in mem_maps],
                          [k * d for _, d, _ in mem_maps], w_a)
        eng.propagate(s, w_a, s.d3 + s.d2, energy, s.magnification, intensity_acc=acc["reference"])
        if sums:
            one.zero_()
            eng.propagate(s, w_a, s.d3 + s.d2, energy, s.magnification, intensity_acc=one)
            per_energy.append(float(one.cpu().numpy().astype(np.float64).sum()))
        eng.propagate(s, w_a, s.d2, energy, mag_mem_obj, wave_out=w_b)
        abi.transmit_wave(w_b, 0.0, [t for t, _, _ in smp_maps], [k * b for _, _, b in smp_maps],
                          [k * d for _, d, _ in smp_maps], w_b)
        eng.propagate(s, w_b, s.d3, energy, s.magnification, intensity_acc=acc["sample"])
        abi.mean(acc["reference"], means[ie:ie + 1])
        if first:
            abi.transmit_wave(None, amp, [t for t, _, _ in smp_maps], [k * b for _, _, b in smp_maps],
                              [k * d for _, d, _ in smp_maps], w_b)
            eng.propagate(s, w_b, s.d3, energy, s.magnification, intensity_acc=acc["propag"])
            white_sum += amp * amp
        if energy > s.thresholds[ibin] - s.energy_sampling / 2:
            fwhm = s.effective_source_fwhm()
            abi.fill(acc["white"], white_sum)
            for name in out:
                eng.detect(acc[name], fwhm, s.psf_sigma, 0, out[name][ibin])
            ibin += 1
            for a in acc.values():
                a.zero_()
            white_sum = 0.0
            bin_starts.add(ie + 1)
    r = means.cpu().numpy()
    per = r.copy()
    for i in range(1, len(per)):
        if i not in bin_starts:
            per[i] = r[i] - r[i - 1]
    energies = [e for e, _ in s.spectrum]
    return out, (float(np.dot(per, energies)), float(per.sum())), np.array(per_energy) if sums else None


# ------------------------------------------------------------------ one call per position
@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_single_call_matches_the_loop_and_the_oracle(shim, name):
    c = Case(shim, name)
    eng = c.eng
    n_e = None
    for point in (0, 1):
        scene = c.position(point)
        n_e = len(scene.spectrum)
        old, old_me, old_sums = _old_chain(eng, scene, point)
        got = eng.compute_fresnel(scene, point)
        sums = eng.means[:n_e].cpu().numpy()
        want = c.oracle(point)
        images = ("sample", "reference") + (("propag", "white") if point == 0 else ())
        for i, k in enumerate(images):
            a = got[k].cpu().numpy()
            b = old[k].cpu().numpy()
            assert a.shape == b.shape == want[i].shape
            assert rel_l2(a, b) < TOL_OLD, (k, point)
            assert rel_l2(a, want[i]) < TOL_ORACLE, (k, point)
        assert np.allclose(got["mean_energy"], old_me, rtol=1e-6, atol=0), point
        # the fused per-energy sums against fp64 sums of each energy's reference intensity
        assert np.allclose(sums, old_sums, rtol=1e-6, atol=0), point
        assert scene.thresholds == c.thresholds
    # a lone energy starts from a zero accumulator, so the accumulator holds exactly the fp32 values the sum is formed
    # from: the two agree to the fp64 summation order
    for point in (0, 1):
        scene = c.position(point)
        for ie in range(n_e):
            m = eng.accumulate_fresnel(scene, point, [ie])
            fused = float(m[0]) * eng.nx * eng.ny
            acc = eng.acc["reference"].cpu().numpy().astype(np.float64).sum()
            assert abs(fused / acc - 1) < 1e-11, (point, ie, fused, acc)


# ------------------------------------------------------------------ energy sharding
def _close(a, b, noise, what):
    if noise:
        # same Philox stream and the same expectations up to fp32 summation order: at most a few draws move
        assert np.mean(a != b) < 2e-3 and rel_l2(a, b) < 1e-3, what
    else:
        assert rel_l2(a, b) < 1e-6, what


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["B200_small_poly3", "Small_six_materials_poly3", "cufft_grid"])
@pytest.mark.parametrize("noise", [False, True])
def test_world1_matches_single_call(shim, name, noise):
    from paresis_b200 import shard
    c = Case(shim, name, noise=noise)
    eng = c.eng
    for point in (0, 1):
        scene = c.position(point)
        got = shard.compute_fresnel_energy_sharded(eng, scene, point)       # first on a fresh engine, as on a rank > 0
        ref = eng.compute_fresnel(scene, point)
        images = ("sample", "reference") + (("propag", "white") if point == 0 else ())
        for k in images:
            a, b = got[k].cpu().numpy(), ref[k].cpu().numpy()
            assert a.shape == b.shape
            _close(a, b, noise, (k, point))
        assert np.allclose(got["mean_energy"], ref["mean_energy"], rtol=1e-7, atol=0)
        later = shard.compute_fresnel_energy_sharded(eng, scene, point, defer=True)
        assert "mean_energy" not in later._out
        fin = later.finish()
        assert fin is later.finish()
        for k in images:
            _close(fin[k].cpu().numpy(), ref[k].cpu().numpy(), noise, (k, point, "deferred"))
        assert np.allclose(fin["mean_energy"], ref["mean_energy"], rtol=1e-7, atol=0)


def _rank_main(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import tempfile
    import torch.distributed as dist
    from paresis_b200 import shard, workspace
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    workspace.enter(workspace.make_workspace(tempfile.mkdtemp()))
    shim = importlib.import_module("Experiment")
    c = Case(shim, "B200_small_poly3")
    out = {}
    for point in (0, 1):
        scene = c.position(point)
        res = shard.compute_fresnel_energy_sharded(c.eng, scene, point)
        later = shard.compute_fresnel_energy_sharded(c.eng, scene, point, defer=True).finish()      # every rank, same order
        if rank == 0:
            single = c.eng.compute_fresnel(scene, point)
            keys = ("sample", "reference") + (("propag", "white") if point == 0 else ())
            out[point] = ({k: res[k].cpu().numpy() for k in keys}, {k: later[k].cpu().numpy() for k in keys},
                          {k: single[k].cpu().numpy() for k in keys}, res["mean_energy"], later["mean_energy"],
                          single["mean_energy"])
        else:
            assert res is None and later is None
    if rank == 0:
        q.put(out)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_world2_nccl_matches_single_gpu():
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_main, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = q.get(timeout=600)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for point in (0, 1):
        sharded, deferred, single, me_s, me_d, me_1 = out[point]
        for k in single:
            # the two ranks' partial images are added after the linear detector: fp32 sums in another order
            assert rel_l2(sharded[k], single[k]) < 1e-6, (k, point)
            assert rel_l2(deferred[k], single[k]) < 1e-6, (k, point)
        assert np.allclose(me_s, me_1, rtol=1e-6, atol=0) and np.allclose(me_d, me_1, rtol=1e-6, atol=0)
