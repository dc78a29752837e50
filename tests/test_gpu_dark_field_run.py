"""Scattering (dark-field) samples as one library call per membrane position (paresis_df_run), and on the energy-sharded path.

A sample material with a dark-field model (Lung, or every material of the sample named 'cylinder_beeds'; Sample.py:322-343)
sends the sample beam through fastRefractionDF (refractionFileNumba2.py:88-196).  Checked here, at positions 0 and 1 of
five cases (a Lung sphere, three energies in two bins, six materials of which one is Lung so that the hops see mixed maps,
two materials that both scatter, air + plate + scintillator):
  - argument rejection, host only;
  - compute_rt against the per-energy Python loop it replaced (restated below), against an fp64 oracle loop, and each
    energy's reference sum against the fp64 sum of its reference image;
  - the energy-sharded call at world size 1 (noise off and on, immediate and deferred) and 2 (NCCL) against compute_rt;
  - the many-positions call refusing a scattering scene.
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

CASES = ["sphere_lung", "poly3_lung", "six_lung", "beeds", "plate_lung"]
ORACLE_CASES = ["sphere_lung", "poly3_lung", "six_lung", "beeds"]     # the oracle loop has no air, plate or scintillator
SIX = ["Muscle", "Adipose", "Bone", "PMMA", "Nylon", "SolidWater"]


# ------------------------------------------------------------------ fixtures
def _blob(shape, cx, cy, r_px, pix_um):
    x = np.arange(shape[0])[:, None] - cx
    y = np.arange(shape[1])[None, :] - cy
    return 2 * np.sqrt(np.maximum(r_px ** 2 - x ** 2 - y ** 2, 0.0)) * pix_um * 1e-6


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return _workspace(str(tmp_path_factory.mktemp("ws_df")))


def _workspace(root):
    """A workspace with the images of the six-material sample (loadSampleGeometryFromImages)."""
    from paresis_b200 import workspace
    from paresis_b200.hostio import imageio
    ws = workspace.make_workspace(root)
    folder = os.path.join(ws, "Samples", "ManyMaterials")
    os.makedirs(folder, exist_ok=True)
    shape, pix = (192, 256), 6.0 / 2 / (145.2 / 141.6)
    centres = [(0.5, 0.5, 0.45), (0.35, 0.4, 0.2), (0.6, 0.62, 0.12), (0.3, 0.75, 0.15), (0.7, 0.25, 0.1)]
    maps = [_blob(shape, cx * shape[0], cy * shape[1], r * shape[0], pix) for cx, cy, r in centres] + [np.full(shape, 40e-6)]
    for m, t in enumerate(maps):
        imageio.write_tiff(os.path.join(folder, "m%d_%s.tif" % (m, SIX[m])), t.astype(np.float32))
    workspace.enter(ws)
    return importlib.import_module("Experiment")


def _experiment(shim, case, noise=False):
    """The experiment of a case, its scene (bins closed) and engine; the membrane of position 0 is drawn.  Use _at() for
    the scene of another position."""
    name = {"sphere_lung": "Small_sphere_mono", "poly3_lung": "B200_small_poly3", "six_lung": "Small_six_materials_poly3",
            "beeds": "Small_sphere_mono", "plate_lung": "Small_sphere_air_plate_CsI"}[case]
    d = dict(experimentName=name, filepath="unused/", overSampling=2, nbExpPoints=2, simulation_type="RayT", expID="t",
             poissonNoise=noise, seed=11)
    e = shim.Experiment(d)
    smp = e.mySampleofInterest
    if case == "six_lung":
        smp.myMaterials = list(smp.myMaterials)
        smp.myMaterials[1] = "Lung"
    elif case == "beeds":
        t0 = np.asarray(smp.myGeometry)[0].astype(np.float64)
        smp.myGeometry = np.stack([t0, 0.6 * np.roll(t0, (30, 50), axis=(0, 1))])
        smp.myMaterials = ["PMMA", "Nylon"]
        smp.myName = "cylinder_beeds"
    else:
        smp.myMaterials = ["Lung"] + list(smp.myMaterials[1:])
    smp.delta, smp.beta = [], []
    smp.getDeltaBeta(e.mySource.mySpectrum)
    _membrane(e, 0)
    thresholds = list(e._open_bins(0))
    return e, e._scene(thresholds), e._get_engine()


def _membrane(e, point):
    np.random.seed(31 + point)
    mem = e.myMembrane
    mem.myGeometry = []
    mem.getMyGeometry(e.exp_dict['studyDimensions'], mem.membranePixelSize, 2, point, 2)


def _at(e, scene, point):
    """The membrane of ``point`` and the scene that holds it."""
    _membrane(e, point)
    return e._scene(scene.thresholds)


# ------------------------------------------------------------------ the loop paresis_df_run replaced, restated
def _old_loop(e, scene, point_num):
    """The per-energy Python loop that ran a scattering sample before paresis_df_run: about ten library calls and two
    fp64 reductions per energy, the reference beam in a hop of its own.  Returns the images, the per-energy reference
    sums, the dark-field map and the displacement maps."""
    from paresis_b200 import _cabi as abi, darkfield, engine, hostmath as hm
    eng = e._get_engine()
    s = scene
    first = point_num == 0
    nx, ny = eng.nx, eng.ny
    f32 = dict(device=eng.device, dtype=torch.float32)
    bins = eng.bins(s)
    nbins = len(s.thresholds)
    out = eng._new_outputs(nbins, first)
    closing = {b[-1] for b in bins[:nbins]}
    for a in eng.acc.values():
        a.zero_()
    smp = e.mySampleofInterest
    plain, scat, clean, moved, df_px = (torch.empty((nx, ny), **f32) for _ in range(5))
    df_total = torch.zeros((nx, ny), **f32)
    g2 = hm.refraction_gradient_scale(s.d2, s.magnification, s.study_pixel_um)
    g3 = hm.refraction_gradient_scale(s.d3, s.magnification, s.study_pixel_um)
    to_px = s.d3 / (s.study_pixel_um * 1e-6 * s.magnification)
    sums, ibin, white = [], 0, 0.0
    fwhm = s.effective_source_fwhm()
    fits = eng.sample_fits(s, with_membrane=True)
    for ie, (energy, flux) in enumerate(s.spectrum):
        k = hm.wavenumber(energy * 1000)
        i0 = s.mean_shot_count / s.os ** 2 * flux * s.common_factor(energy)
        plate = s.plate_factor(energy)
        mem_maps, mem_ub, _ = eng._split(s.membrane, energy)
        smp_maps, _, _ = eng._split(s.sample, energy)
        smp_layers, fractions, have_df = [], [], False
        for imat, (t, d, b) in enumerate(smp_maps):
            model = darkfield.model_of(smp, imat)
            fraction = 1.0
            if model is not None:
                coeff, fraction = hm.angle_coefficient(d, hm.MODELS[model]), hm.MODELS[model][1]
                abi.df_angle(t, coeff * to_px, df_px)
                have_df = True
            smp_layers.append((t, d * fraction, b * fraction))
            fractions.append(fraction)
        if not have_df:
            df_px.zero_()
        if not fits:
            smp_layers = eng.mixed_sample(s.sample, energy, fractions)
        eng.i_bs.zero_()
        abi.refract_layers(None, i0 * np.exp(-2 * k * mem_ub) * plate, [(t, d * g2, 0.0, 2 * k * b) for t, d, b in mem_maps],
                           eng.i_bs, flag=eng.flag)
        hop = [(t, d * g3, d * g3, 0.0) for t, d, b in mem_maps] + [(t, d * g3, 0.0, 2 * k * b) for t, d, b in smp_layers]
        before = eng.acc["reference"].double().sum()
        abi.refract_layers(eng.i_bs, 0.0, [(t, gr, 0.0, 0.0) for t, go, gr, at in hop if gr != 0.0], eng.acc["reference"],
                           flag=eng.flag)
        sums.append(eng.acc["reference"].double().sum() - before)
        abi.df_split(eng.i_bs, 0.0, df_px, nx / 4, plain, scat, clean)
        obj = [(t, go, 0.0, at) for t, go, gr, at in hop]
        abi.refract_layers(plain, 0.0, obj, eng.acc["sample"], flag=eng.flag)
        moved.zero_()
        abi.refract_layers(scat, 0.0, obj, moved, flag=eng.flag)
        abi.df_scatter(moved, clean, eng.acc["sample"])
        if first:
            prop = [(t, d * g3, 0.0, 2 * k * b) for t, d, b in smp_layers]
            abi.df_split(None, i0 * plate, df_px, nx / 4, plain, scat, clean)
            abi.refract_layers(plain, 0.0, prop, eng.acc["propag"], flag=eng.flag)
            moved.zero_()
            abi.refract_layers(scat, 0.0, prop, moved, flag=eng.flag)
            abi.df_scatter(moved, clean, eng.acc["propag"])
            abi.axpy(df_total, df_px, flux / to_px)
            white += i0 * plate
        if ie in closing:
            seq = eng.sequence(point_num) + 4 * ibin
            names = engine.IMAGES[:4 if first else 2]
            if first:
                abi.fill(eng.acc["white"], white)
            src = eng._gauss(fwhm / 2.355) if fwhm != 0 else None
            psf = eng._gauss(s.psf_sigma) if s.psf_sigma != 0 else None
            abi.detect_counts_multi([eng.acc[n] for n in names], eng.os, eng.det_x, eng.det_y, src, psf, eng.work,
                                    [out[n][ibin] for n in names], eng.poisson, eng.seed, [seq + k_ for k_ in range(len(names))])
            ibin += 1
            if ie + 1 < len(s.spectrum):
                for a in eng.acc.values():
                    a.zero_()
                white = 0.0
    eng._i_bs_dirty = True
    eng.check_flag()
    res = {k: out[k].cpu().numpy() for k in engine.IMAGES[:4 if first else 2]}
    res["sums"] = torch.stack(sums).cpu().numpy()
    if first:
        res["dark_field"] = df_total.cpu().numpy()
        res["dx"], res["dy"] = darkfield._displacement_maps(eng, smp_layers, g3, df_px)
    return res


def _images(first):
    return ("sample", "reference") + (("propag", "white") if first else ())


# ------------------------------------------------------------------ host-only argument checks
def test_df_run_rejects_bad_arguments():
    """Every argument check happens before the first CUDA call: bogus device addresses are never touched."""
    from paresis_b200 import _cabi as abi
    vp = 4096

    def job(n_hop2=2, scatter=True, **over):
        en = (abi.RtEnergy * 1)()
        en[0].n_hop1, en[0].n_hop2, en[0].n_propag, en[0].close_bin = 1, n_hop2, 1, 1
        for lay, n in ((en[0].hop1, 1), (en[0].hop2, n_hop2), (en[0].propag, 1)):
            for m in range(min(n, abi.MAX_LAYERS)):
                lay[m].thickness = vp
        df = (abi.DfEnergy * 1)()
        df[0].scatter_map = vp if scatter else None
        df[0].angle_coeff = 1.0
        j = abi.DfJob()
        r = j.rt
        r.nx, r.ny, r.oversampling, r.det_x, r.det_y = 64, 64, 2, 32, 32
        r.first_point, r.n_energies, r.energies_host = 1, 1, en
        r.i_bs = r.acc_sample = r.acc_ref = r.acc_propag = r.acc_white = vp
        r.out_sample = r.out_ref = r.out_propag = r.out_white = vp
        j.energies_df_host = df
        j.angle = j.plain = j.scattered = j.clean = j.moved = vp
        for key, value in over.items():
            target = r if hasattr(r, key) and key not in ("angle", "plain", "scattered", "clean", "moved", "dark_field") else j
            setattr(target, key, value)
        return j, (en, df)

    cases = [
        (dict(i_bs=None), b"null object-plane buffer"),
        (dict(acc_propag=None), b"null object-plane buffer"),
        (dict(moved=None), b"null dark-field scratch"),
        (dict(angle=None), b"null dark-field scratch"),
        (dict(out_white=None), b"incomplete detector outputs"),
        (dict(acc_white=None), b"incomplete detector outputs"),
        (dict(first_point=0, dark_field=vp), b"belongs to position 0"),
        (dict(n_hop2=abi.MAX_LAYERS + 1), b"mix the sample's maps"),
        (dict(n_hop2=0), b"object hop"),
        (dict(scatter=False), b"no scattering map"),
        (dict(n_energies=0), b"no energies"),
        (dict(nx=2), b"bad frame"),
    ]
    for over, msg in cases:
        n_hop2, scatter = over.pop("n_hop2", 2), over.pop("scatter", True)
        j, keep = job(n_hop2, scatter, **over)
        assert abi.lib.paresis_df_run(ctypes.byref(j), None) == 2, msg
        assert msg in abi.lib.paresis_last_error(), (msg, abi.lib.paresis_last_error())
    assert abi.lib.paresis_df_run(None, None) == 2


# ------------------------------------------------------------------ the single call
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_single_call_matches_old_loop(shim, case):
    e, scene, eng = _experiment(shim, case)
    assert eng.scatters(scene)
    if case == "six_lung":
        assert not eng.sample_fits(scene, with_membrane=True)
    energies = np.array([en for en, _ in scene.spectrum])
    for point in (0, 1):
        scene = _at(e, scene, point)
        old = _old_loop(e, scene, point)
        got = eng.compute_rt(scene, point, want_displacement=True)
        for k in _images(point == 0):
            assert rel_l2(got[k].cpu().numpy(), old[k]) < 3e-6, (k, point)
        m = old["sums"] / float(eng.nx * eng.ny)
        assert np.allclose(got["mean_energy"], (float(np.dot(m, energies)), float(m.sum())), rtol=1e-6)
        if point == 0:
            assert np.abs(old["dark_field"]).max() > 0
            assert rel_l2(got["dark_field"].cpu().numpy(), old["dark_field"]) < 1e-6
            assert eng.dx_pad.shape == old["dx"].shape
            assert rel_l2(eng.dx_pad.cpu().numpy(), old["dx"]) < 1e-6 and rel_l2(eng.dy_pad.cpu().numpy(), old["dy"]) < 1e-6
        else:
            assert "dark_field" not in got


def _db(obj, energies):
    return {en: ([dict(obj.delta[m]).get(en, 0.0) for m in range(len(obj.delta))],
                 [dict(obj.beta[m]).get(en, 0.0) for m in range(len(obj.beta))]) for en in energies}


def _oracle_df(e, point):
    """Experiment.py:407-526 with fastRefractionDF in fp64 (vacuum, no plate or scintillator), from the oracle's pieces."""
    from paresis_b200 import darkfield
    det, src = e.myDetector.det_param, e.mySource.source_dict
    s = po.Setup(e.exp_dict['distSourceToMembrane'], e.exp_dict['distMembraneToObject'], e.exp_dict['distObjectToDetector'],
                 det['myDimensions'], det['myPixelSize'], 2, e.exp_dict['meanShotCount'], list(e.mySource.mySpectrum),
                 src["mySize"], det['myPSF'], energy_sampling=src["myEnergySampling"],
                 bin_thresholds=det["myBinsThersholds"][:-1])
    mem, smp = e.myMembrane, e.mySampleofInterest
    energies = [en for en, _ in s.spectrum]
    mem_t, mem_db = np.asarray(mem.myGeometry).astype(np.float64), _db(mem, energies)
    smp_t, smp_db = np.asarray(smp.myGeometry).astype(np.float64), _db(smp, energies)
    models = [darkfield.model_of(smp, m) for m in range(smp_t.shape[0])]
    n, first = s.study_dims, point == 0
    zeros = np.zeros(n)
    acc = {k: np.zeros(n) for k in ("sample", "reference", "propag", "white")}
    images = {k: [] for k in acc}
    dark, ibin, fwhm = np.zeros(n), 0, s.effective_source_fwhm()
    args = lambda energy: (s.d3, energy, s.magnification, s.study_pixel_um)
    for energy, flux in s.spectrum:
        inc = np.ones(n) * (s.mean_shot_count / s.os ** 2) * flux
        i_m, phi_m = po.set_wave_rt(inc, zeros, mem_t, *mem_db[energy], energy)
        i_bs, _, _ = po.fast_refraction(np.abs(i_m), phi_m, s.d2, energy, s.magnification, s.study_pixel_um)
        i_s, phi_s, df = po.set_wave_rt_df(i_bs, phi_m, smp_t, *smp_db[energy], energy, models)
        acc["sample"] += po.fast_refraction_df(np.abs(i_s), phi_s, *args(energy), df)[0]
        acc["reference"] += po.fast_refraction(np.abs(i_bs), phi_m, *args(energy))[0]
        if first:
            i_p, phi_p, df_p = po.set_wave_rt_df(inc, zeros, smp_t, *smp_db[energy], energy, models)
            acc["propag"] += po.fast_refraction_df(np.abs(i_p), phi_p, *args(energy), df_p)[0]
            acc["white"] += inc
            dark += df_p * flux
        if energy > s.thresholds[ibin] - s.energy_sampling / 2:
            for k in acc:
                images[k].append(po.detection(acc[k], fwhm, s.os, s.det_dims, s.psf_sigma))
                acc[k] = np.zeros(n)
            ibin += 1
    return {k: np.stack(v) for k, v in images.items()}, dark


@pytest.mark.gpu
@pytest.mark.parametrize("case", ORACLE_CASES)
def test_single_call_matches_oracle(shim, case):
    e, scene, eng = _experiment(shim, case)
    for point in (0, 1):
        scene = _at(e, scene, point)
        got = eng.compute_rt(scene, point)
        want, dark = _oracle_df(e, point)
        for k in _images(point == 0):
            assert rel_l2(got[k].cpu().numpy(), want[k]) < 1e-5, (k, point)
        if point == 0:
            assert rel_l2(got["dark_field"].cpu().numpy(), dark) < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["sphere_lung", "poly3_lung", "six_lung", "beeds"])
def test_reference_sums_are_each_energys_own(shim, case):
    """means[e] of one energy = the fp64 sum of that energy's reference image (both object hops add to it)."""
    e, scene, eng = _experiment(shim, case)
    for point in (0, 1):
        for i in range(len(scene.spectrum)):
            mean = float(eng.accumulate_rt(scene, point, [i])[0])
            want = float(eng.acc["reference"].double().sum()) / (eng.nx * eng.ny)
            assert abs(mean / want - 1) < 1e-6, (point, i)


@pytest.mark.gpu
def test_many_positions_call_refuses_scattering_scenes(shim):
    e, scene, eng = _experiment(shim, "sphere_lung")
    with pytest.raises(NotImplementedError):
        eng.compute_rt_positions(scene, None, [[0, 0]], [0])


# ------------------------------------------------------------------ the energy-sharded call
def _agree(a, b, noise, what):
    if noise:
        # same Philox stream; expectations agree to an ulp, so only draws on a decision boundary may move
        assert np.mean(a != b) < 2e-3 and rel_l2(a, b) < 1e-3, what
    else:
        assert rel_l2(a, b) < 3e-6, what


@pytest.mark.gpu
@pytest.mark.parametrize("noise", [False, True])
@pytest.mark.parametrize("case", ["sphere_lung", "poly3_lung", "six_lung"])
def test_sharded_world1_matches_single_call(shim, case, noise):
    from paresis_b200 import shard
    e, scene, eng = _experiment(shim, case, noise)
    for point in (0, 1):
        ref = eng.compute_rt(scene, point)
        got = shard.compute_rt_energy_sharded(eng, scene, point)
        later = shard.compute_rt_energy_sharded(eng, scene, point, defer=True)
        assert "mean_energy" not in later._out
        fin = later.finish()
        for res in (got, fin):
            for k in _images(point == 0):
                a, b = res[k].cpu().numpy(), ref[k].cpu().numpy()
                assert a.shape == b.shape
                _agree(a, b, noise, (k, point))
            assert np.allclose(res["mean_energy"], ref["mean_energy"], rtol=1e-6)
            if point == 0:
                assert rel_l2(res["dark_field"].cpu().numpy(), ref["dark_field"].cpu().numpy()) < 1e-6
            else:
                assert "dark_field" not in res


def _rank_main(rank, world, port, root, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from paresis_b200 import shard
    shim = _workspace(os.path.join(root, "rank%d" % rank))
    out = {}
    for noise in (False, True):
        e, scene, eng = _experiment(shim, "poly3_lung", noise)
        for point in (0, 1):
            res = shard.compute_rt_energy_sharded(eng, scene, point)
            later = shard.compute_rt_energy_sharded(eng, scene, point, defer=True).finish()
            if rank == 0:
                single = eng.compute_rt(scene, point)
                keys = _images(point == 0) + (("dark_field",) if point == 0 else ())
                out[noise, point] = ({k: res[k].cpu().numpy() for k in keys}, {k: later[k].cpu().numpy() for k in keys},
                                     {k: single[k].cpu().numpy() for k in keys}, res["mean_energy"], single["mean_energy"])
            else:
                assert res is None and later is None
    if rank == 0:
        q.put(out)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_sharded_world2_nccl_matches_single_call(tmp_path):
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_main, args=(r, 2, port, str(tmp_path), q)) for r in range(2)]
    for p in procs:
        p.start()
    out = q.get(timeout=900)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for (noise, point), (sharded, later, single, me_s, me_1) in out.items():
        for k in single:
            if k == "dark_field":
                assert rel_l2(sharded[k], single[k]) < 1e-6 and rel_l2(later[k], single[k]) < 1e-6
                continue
            _agree(sharded[k], single[k], noise, (k, noise, point))
            _agree(later[k], single[k], noise, (k, noise, point))
        assert np.allclose(me_s, me_1, rtol=1e-6)
