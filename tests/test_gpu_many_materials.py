"""Samples of any number of materials, and uniform sample layers, on every GPU path.

A hop takes at most PARESIS_MAX_LAYERS thickness maps; a sample that does not fit (or has a uniform layer) reaches the
hops as two maps per energy, mixed by paresis_mix_maps (engine.ImageFormation.mixed_sample).  Checked here:
  - the kernel against numpy in fp64 (within one fp32 rounding) and its argument checks;
  - a six-material sample (five images and a flat map, loadSampleGeometryFromImages) against the fp64 oracle with the
    same maps, ray tracing (mono and three energies in one bin) and Fresnel, at the 1e-5 bound; the other ray-tracing
    drivers (positions in one call, energy sharding) against the position-by-position call;
  - uniform sample layers (the your_own_geometry template; a mapped sample plus a uniform Layer) against the oracle;
  - invariance: splitting a sample's maps into parts of the same material leaves the images unchanged (dark field too);
  - stand-alone setWave / setWaveRT of six materials against the oracle.
"""
import importlib
import os

import numpy as np
import pytest

import paresis_oracle as po
from conftest import rel_l2

torch = pytest.importorskip("torch")

TOL = 1e-5
MATERIALS = ["Muscle", "Adipose", "Bone", "PMMA", "Nylon", "SolidWater"]


def _blob(shape, cx, cy, r_px, pix_um):
    """Projected thickness (metres) of a sphere of radius r_px pixels centred at (cx, cy)."""
    x = np.arange(shape[0])[:, None] - cx
    y = np.arange(shape[1])[None, :] - cy
    return 2 * np.sqrt(np.maximum(r_px ** 2 - x ** 2 - y ** 2, 0.0)) * pix_um * 1e-6


def _six_maps(shape, pix_um):
    nx, ny = shape
    maps = [_blob(shape, nx * 0.5, ny * 0.5, 0.45 * nx, pix_um),              # Muscle: the body
            _blob(shape, nx * 0.35, ny * 0.4, 0.2 * nx, pix_um),              # Adipose
            _blob(shape, nx * 0.6, ny * 0.62, 0.12 * nx, pix_um),             # Bone
            _blob(shape, nx * 0.3, ny * 0.75, 0.15 * nx, pix_um),             # PMMA
            _blob(shape, nx * 0.7, ny * 0.25, 0.1 * nx, pix_um)]              # Nylon
    maps.append(np.full(shape, 40e-6))                                        # SolidWater: a flat 40 um layer
    return [m.astype(np.float32) for m in maps]


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from paresis_b200 import workspace
    from paresis_b200.hostio import imageio
    ws = workspace.make_workspace(str(tmp_path_factory.mktemp("ws_many")))
    folder = os.path.join(ws, "Samples", "ManyMaterials")
    os.makedirs(folder)
    # study grid of the small_96x128_psf detector at oversampling 2; one image per material, named in material order
    pix = 6.0 / 2 / (145.2 / 141.6)
    for m, t in enumerate(_six_maps((192, 256), pix)):
        imageio.write_tiff(os.path.join(folder, "m%d_%s.tif" % (m, MATERIALS[m])), t)
    old = os.getcwd()
    workspace.enter(ws)
    yield importlib.import_module("Experiment")
    os.chdir(old)


def _experiment(shim, name, model, points=2):
    d = dict(experimentName=name, filepath="unused/", overSampling=2, nbExpPoints=points, simulation_type=model,
             expID="t", poissonNoise=False)
    return shim.Experiment(d)


def _membrane(e, point, seed=21):
    np.random.seed(seed + point)
    mem = e.myMembrane
    mem.myGeometry = []
    mem.getMyGeometry(e.exp_dict['studyDimensions'], mem.membranePixelSize, 2, point, 2)


def _db(obj, energies):
    return {en: ([dict(obj.delta[m]).get(en, 0.0) for m in range(len(obj.delta))],
                 [dict(obj.beta[m]).get(en, 0.0) for m in range(len(obj.beta))]) for en in energies}


def _setup(e):
    det, src = e.myDetector.det_param, e.mySource.source_dict
    return po.Setup(e.exp_dict['distSourceToMembrane'], e.exp_dict['distMembraneToObject'], e.exp_dict['distObjectToDetector'],
                    det['myDimensions'], det['myPixelSize'], 2, e.exp_dict['meanShotCount'], list(e.mySource.mySpectrum),
                    src["mySize"], det['myPSF'], energy_sampling=src["myEnergySampling"])


def _oracle(e, model, point, sample_t=None, sample_db=None):
    energies = [en for en, _ in e.mySource.mySpectrum]
    mem, smp = e.myMembrane, e.mySampleofInterest
    sample_t = np.asarray(smp.myGeometry).astype(np.float64) if sample_t is None else sample_t
    sample_db = _db(smp, energies) if sample_db is None else sample_db
    fn = po.compute_rt if model == "RayT" else po.compute_fresnel
    return fn(_setup(e), np.asarray(mem.myGeometry).astype(np.float64), _db(mem, energies), sample_t, sample_db, point)


def _run(e, model, point):
    if model == "RayT":
        return e.computeSampleAndReferenceImages_RT(point)
    return e.computeSampleAndReferenceImages_Fresnel(point)


# ------------------------------------------------------------------ the kernel
def test_mix_maps_rejects_bad_arguments():
    """Argument checks happen before any CUDA call (no device needed)."""
    import ctypes
    from paresis_b200 import _cabi as abi
    vp = ctypes.c_void_p
    one = (vp * 1)(vp(16))
    w = (ctypes.c_double * 2)(1.0, 1.0)
    outs = (vp * 2)(vp(16), vp(32))
    cases = [((None, 1, w, None, 1, outs), b"null pointer"), ((one, 1, None, None, 1, outs), b"null pointer"),
             ((one, 1, w, None, 1, None), b"null pointer"), ((one, 0, w, None, 1, outs), b"n_maps >= 1"),
             ((one, 1, w, None, 0, outs), b"n_out must be 1 or 2"), ((one, 1, w, None, 3, outs), b"n_out must be 1 or 2"),
             (((vp * 1)(None), 1, w, None, 1, outs), b"null material map 0"),
             ((one, 1, w, None, 2, (vp * 2)(vp(16), None)), b"null output map 1")]
    for (maps, n_maps, weights, bias, n_out, out), msg in cases:
        assert abi.lib.paresis_mix_maps(maps, n_maps, weights, bias, n_out, out, 100, None) == 2
        assert msg in abi.lib.paresis_last_error(), msg


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(130, 291), (64, 64)])
@pytest.mark.parametrize("n_maps", [1, 2, 7, 13, 40])
@pytest.mark.parametrize("n_out", [1, 2])
@pytest.mark.parametrize("with_bias", [False, True])
def test_mix_maps_matches_fp64(shape, n_maps, n_out, with_bias):
    """out[k] = bias[k] + sum_m w[k][m] maps[m] within one fp32 rounding of the fp64 value (130 x 291: n % 4 != 0; 40 maps:
    two chunks of the shared-memory table)."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from paresis_b200 import _cabi as abi
    rng = np.random.default_rng(n_maps * 10 + n_out)
    maps = [rng.uniform(0, 1e-3, shape).astype(np.float32) for _ in range(n_maps)]
    weights = rng.uniform(0.01, 1.0, (n_out, n_maps))
    bias = rng.uniform(0, 1e-4, n_out) if with_bias else None
    want = np.einsum("km,mxy->kxy", weights, np.stack(maps).astype(np.float64))
    if with_bias:
        want += bias[:, None, None]
    d_maps = [torch.as_tensor(m, device="cuda") for m in maps]
    outs = [torch.full(shape, np.nan, device="cuda") for _ in range(n_out)]
    abi.mix_maps(d_maps, weights.tolist(), bias.tolist() if with_bias else None, outs)
    for k in range(n_out):
        got = outs[k].cpu().numpy().astype(np.float64)
        assert (np.abs(got - want[k]) <= np.spacing(np.abs(want[k]).astype(np.float32)).astype(np.float64)).all()
    # maps that are not 16-byte aligned take the scalar loads
    base = torch.as_tensor(np.concatenate([np.zeros(1, np.float32), maps[0].ravel()]), device="cuda")
    out = torch.empty(maps[0].size, device="cuda")
    abi.mix_maps([base[1:]], [[0.5]], None, [out])
    assert np.array_equal(out.cpu().numpy(), (maps[0].ravel().astype(np.float64) * 0.5).astype(np.float32))


# ------------------------------------------------------------------ six materials against the oracle
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["Small_six_materials_mono", "Small_six_materials_poly3"])
def test_six_materials_ray_tracing_matches_oracle(shim, name):
    e = _experiment(shim, name, "RayT")
    st = np.asarray(e.mySampleofInterest.myGeometry)
    assert st.shape == (6, 192, 256) and e.mySampleofInterest.myMaterials == MATERIALS
    for point in (0, 1):
        _membrane(e, point)
        if point == 0:
            scene = e._scene(list(e.myDetector.det_param["myBinsThersholds"]) + [e.mySource.mySpectrum[-1][0]])
            assert not e._get_engine().sample_fits(scene, with_membrane=True)
        res = _run(e, "RayT", point)
        want = _oracle(e, "RayT", point)
        for k, img in enumerate(("sample", "reference", "propag", "white")[:4 if point == 0 else 2]):
            assert rel_l2(res[k], want[k]) < TOL, img
        if point == 0:
            # displacement of the sample-only beam at the last energy (fp32 phase map of the mixed materials)
            s = _setup(e)
            energy = e.mySource.mySpectrum[-1][0]
            sd, sb = _db(e.mySampleofInterest, [energy])[energy]
            i_p, phi_p = po.set_wave_rt(np.ones(s.study_dims), np.zeros(s.study_dims), st.astype(np.float64), sd, sb, energy)
            _, dx, dy = po.fast_refraction(i_p, phi_p, s.d3, energy, s.magnification, s.study_pixel_um)
            assert res[4].shape == dx.shape
            assert rel_l2(res[4], dx) < 5e-5 and rel_l2(res[5], dy) < 5e-5


@pytest.mark.gpu
def test_six_materials_fresnel_matches_oracle(shim):
    e = _experiment(shim, "Small_six_materials_mono", "Fresnel")
    for point in (0, 1):
        _membrane(e, point)
        res = _run(e, "Fresnel", point)
        want = _oracle(e, "Fresnel", point)
        for k, img in enumerate(("sample", "reference", "propag", "white")[:4 if point == 0 else 2]):
            assert rel_l2(res[k], want[k]) < TOL, img


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["Small_six_materials_mono", "Small_six_materials_poly3"])
def test_six_materials_other_drivers(shim, name):
    """paresis_rt_run_positions (1 or 3 streams, 3 positions per launch) and the energy-sharded call at world size 1 give
    the images of the position-by-position call."""
    from paresis_b200 import geometry, shard
    e = _experiment(shim, name, "RayT", points=3)
    mem = e.myMembrane
    dims = e.exp_dict['studyDimensions']
    np.random.seed(77)
    single = []
    for point in range(3):
        mem.myGeometry = []
        mem.getMyGeometry(dims, mem.membranePixelSize, 2, point, 3)
        res = e.computeSampleAndReferenceImages_RT(point)
        single.append([np.array(r) for r in res[:4]])
    thresholds = e.myDetector.det_param["myBinsThersholds"]
    eng = e._get_engine()
    # energy sharding at world size 1 against the single call, on the last membrane
    scene = e._scene(thresholds)
    for point in (0, 1):
        ref = eng.compute_rt(scene, point)
        got = shard.compute_rt_energy_sharded(eng, scene, point)
        for k in ("sample", "reference") + (("propag", "white") if point == 0 else ()):
            assert rel_l2(got[k].cpu().numpy(), ref[k].cpu().numpy()) < 3e-6, k
    scene = e._scene(thresholds, per_position_membrane=True)
    plan = geometry.MembranePlan(mem, dims[0], dims[1], mem.membranePixelSize)
    np.random.seed(77)
    offsets = [plan.draw_offsets() for _ in range(3)]
    for slots, per in ((1, 0), (3, 0), (3, 3)):
        out = eng.compute_rt_positions(scene, plan, offsets, [0, 1, 2], n_slots=slots, per_launch=per)
        torch.cuda.synchronize()
        eng.check_flag()
        for p in range(3):
            assert rel_l2(out["sample"][p].cpu().numpy(), single[p][0]) < 1e-6, (slots, per, p)
            assert rel_l2(out["reference"][p].cpu().numpy(), single[p][1]) < 1e-6, (slots, per, p)
        assert rel_l2(out["propag"][0].cpu().numpy(), single[0][2]) < 1e-6
        assert rel_l2(out["white"][0].cpu().numpy(), single[0][3]) < 1e-6


# ------------------------------------------------------------------ uniform sample layers
@pytest.mark.gpu
@pytest.mark.parametrize("model", ["RayT", "Fresnel"])
def test_your_own_geometry_template(shim, model):
    """The bundled template: one flat 5 um Muscle layer."""
    e = _experiment(shim, "Small_your_own_geometry", model, points=1)
    _membrane(e, 0)
    res = _run(e, model, 0)
    want = _oracle(e, model, 0)
    for k in range(4):
        assert rel_l2(res[k], want[k]) < TOL, k


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["RayT", "Fresnel"])
def test_uniform_sample_layer(shim, model):
    """A scene whose sample holds a mapped material and a uniform Layer (thickness as a number): the uniform layer only
    attenuates, through the bias of the mixed attenuation map."""
    from paresis_b200 import engine
    e = _experiment(shim, "Small_sphere_mono", model, points=1)
    _membrane(e, 0)
    energy = e.mySource.mySpectrum[-1][0]
    thresholds = e._open_bins(0)
    scene = e._scene(thresholds)
    from paresis_b200.hostio import tables
    (d_bone, b_bone), = tables.interpolate("Bone", [energy])
    scene.sample.append(engine.Layer(300e-6, {energy: d_bone}, {energy: b_bone}))
    eng = e._get_engine()
    assert not eng.sample_fits(scene, with_membrane=False)
    out = eng.compute_rt(scene, 0) if model == "RayT" else eng.compute_fresnel(scene, 0)
    torch.cuda.synchronize()
    smp = e.mySampleofInterest
    st = np.asarray(smp.myGeometry).astype(np.float64)
    sample_t = np.concatenate([st, np.full((1,) + st.shape[1:], 300e-6)])
    sd, sb = _db(smp, [energy])[energy]
    want = _oracle(e, model, 0, sample_t, {energy: (sd + [d_bone], sb + [b_bone])})
    for k, img in enumerate(engine.IMAGES):
        assert rel_l2(out[img].cpu().numpy(), want[k]) < TOL, img
    # an empty sample still has nothing to image
    scene.sample = []
    with pytest.raises(NotImplementedError):
        eng.compute_rt(scene, 0) if model == "RayT" else eng.compute_fresnel(scene, 0)


# ------------------------------------------------------------------ invariance under splitting a material
def _split_parts(t, n_parts, seed):
    """n_parts maps of the same material that add up to t (smooth, non-flat weights)."""
    rng = np.random.default_rng(seed)
    x = np.linspace(0, 1, t.shape[0])[:, None]
    y = np.linspace(0, 1, t.shape[1])[None, :]
    w = np.stack([1.0 + 0.5 * np.sin(2 * np.pi * (rng.uniform(0.5, 2) * x + rng.uniform(0.5, 2) * y + rng.uniform()))
                  for _ in range(n_parts)])
    w /= w.sum(axis=0)
    return [t * w[k] for k in range(n_parts)]


@pytest.mark.gpu
@pytest.mark.parametrize("model,first", [("RayT", "Lung"), ("RayT", "Nylon"), ("Fresnel", "Nylon")])
def test_splitting_materials_changes_nothing(shim, model, first):
    """Two materials (today's path; with Lung the dark-field model, pinned by the goldens) against the same object as five
    materials: the first kept whole (the Lung angle map comes from its own thickness), the PMMA split in four parts."""
    images = {}
    for split in (False, True):
        e = _experiment(shim, "Small_sphere_mono", model, points=1)
        smp = e.mySampleofInterest
        t0 = np.asarray(smp.myGeometry)[0].astype(np.float64)
        t1 = 0.6 * np.roll(t0, (30, 50), axis=(0, 1))
        geom = [t0] + (_split_parts(t1, 4, 3) if split else [t1])
        smp.myMaterials = [first] + ["PMMA"] * (len(geom) - 1)
        smp.myGeometry = np.stack(geom)
        smp.delta, smp.beta = [], []
        smp.getDeltaBeta(e.mySource.mySpectrum)
        _membrane(e, 0)
        images[split] = _run(e, model, 0)
    assert images[False][0].shape == images[True][0].shape
    for k in range(4):
        assert rel_l2(images[True][k], images[False][k]) < TOL, k
    if model == "RayT":
        assert rel_l2(images[True][6], images[False][6]) < 1e-6         # dark-field map
        if first == "Lung":
            assert np.abs(images[False][6]).max() > 0


# ------------------------------------------------------------------ stand-alone transmission
@pytest.mark.gpu
def test_stand_alone_set_wave_six_materials(shim):
    Sample = importlib.import_module("Sample")
    from paresis_b200.hostio import tables
    shape, E, pix = (70, 111), 52.0, 2.9
    s = Sample.AnalyticalSample()
    s.myType, s.myName, s.myMaterials = "sample_of_interest", "six", MATERIALS
    coeffs = [tables.interpolate(m, [E])[0] for m in MATERIALS]        # (delta, beta) per material at E
    s.delta = [[(E, d)] for d, _ in coeffs]
    s.beta = [[(E, b)] for _, b in coeffs]
    t = np.stack(_six_maps(shape, pix)).astype(np.float64)
    s.myGeometry = t
    deltas, betas = [d for d, _ in coeffs], [b for _, b in coeffs]
    rng = np.random.default_rng(2)
    i_in = rng.uniform(0.8, 1.2, shape) * 7500
    phi_in = rng.uniform(-3, 3, shape)
    i_out, phi_out, df = s.setWaveRT(i_in, E, phi_in)
    t32 = t.astype(np.float32).astype(np.float64)
    want_i, want_phi = po.set_wave_rt(i_in.astype(np.float32).astype(np.float64), phi_in, t32, deltas, betas, E)
    assert df == 0
    assert rel_l2(i_out, want_i) < 1e-6 and rel_l2(phi_out, want_phi) < 1e-6
    assert phi_out.dtype == np.float64
    wave0 = np.sqrt(i_in) * np.exp(1j * phi_in)
    got = s.setWave(wave0, E)
    want = po.set_wave(wave0.astype(np.complex64).astype(np.complex128), t32, deltas, betas, E)
    assert np.abs(got - want).max() / np.abs(want).max() < 2e-5
    assert rel_l2(np.abs(got) ** 2, np.abs(want) ** 2) < 1e-6
