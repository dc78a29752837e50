"""Many membrane positions of the Fresnel model in one library call (paresis_fresnel_run_positions,
engine.ImageFormation.compute_fresnel_positions).

Checked here:
  - argument checks, before any CUDA call (host only, and on the GPU those that need a real plan);
  - the call against the position-by-position compute_fresnel on maps cut at the same offsets: thickness maps and images
    bit for bit, noise off and on, at 1, 2 and 3 slots, with position 0 first and not first; the per-energy sums to the
    fp64 atomicAdd order;
  - the images against the fp64 oracle;
  - a membrane without a sphere field (rasterised per position) against the field path.
Cases: one energy; two detector bins of three energies; a sample of six materials (mixed maps); uniform layers with a
plate and a scintillator; a 100 x 90 grid whose line lengths take the cuFFT path; the 2048^2 benchmark grid, whose two
axes take the in-shared-memory line transform.
"""
import copy
import ctypes
import importlib
import os

import numpy as np
import pytest

from conftest import rel_l2

torch = pytest.importorskip("torch")

ERR_ARG = 2


# ------------------------------------------------------------------ argument checks (no device)
def _args(abi, n_pos=1, n_slots=1, first=0):
    """A well-formed call on fake pointers (nothing is dereferenced before the checks fail)."""
    from test_gpu_fresnel_shard import _host_job
    job, keep = _host_job(abi)
    job.oversampling, job.det_x, job.det_y = 2, 4, 4
    mem = abi.Membrane()
    mem.field, mem.field_x, mem.field_y, mem.n_layers = 16, 64, 64, 1
    offs = (ctypes.c_int64 * 2)(0, 0)
    pos = (abi.RtPosition * n_pos)()
    for p in pos:
        p.offsets_host = ctypes.cast(offs, ctypes.POINTER(ctypes.c_int64))
        p.thickness = p.out_sample = p.out_ref = 16
        p.first_point = first
    slots = (abi.FresnelSlot * n_slots)()
    for k, sl in enumerate(slots):
        sl.plan = 16 * (k + 1)
        sl.wave_a = sl.wave_b = sl.acc_sample = sl.acc_ref = sl.acc_propag = sl.acc_white = 16
    return job, mem, pos, slots, (keep, offs)


def _call(abi, job, mem, pos, slots, n_pos=None, n_slots=None):
    return abi.lib.paresis_fresnel_run_positions(
        ctypes.byref(job) if job is not None else None, ctypes.byref(mem) if mem is not None else None, pos,
        len(pos) if n_pos is None else n_pos, slots, len(slots) if n_slots is None else n_slots, None)


def test_run_positions_rejects_bad_arguments():
    from paresis_b200 import _cabi as abi

    def rejects(msg, *args, **kw):
        assert _call(abi, *args, **kw) == ERR_ARG
        err = abi.lib.paresis_last_error()
        assert err.startswith(b"paresis_fresnel_run_positions") and msg in err, err

    job, mem, pos, slots, keep = _args(abi)
    rejects(b"null job, membrane, positions or slots", None, mem, pos, slots)
    rejects(b"null job, membrane, positions or slots", job, None, pos, slots)
    rejects(b"null job, membrane, positions or slots", job, mem, None, slots, n_pos=1)
    rejects(b"null job, membrane, positions or slots", job, mem, pos, None, n_slots=1)
    rejects(b"n_slots >= 1", job, mem, pos, slots, n_slots=0)
    rejects(b"n_positions >= 0", job, mem, pos, slots, n_pos=-1)
    # nothing to do is fine
    assert _call(abi, job, mem, pos, slots, n_pos=0) == 0

    job, mem, pos, slots, keep = _args(abi)
    job.energies_host = None
    rejects(b"no energies", job, mem, pos, slots)
    job, mem, pos, slots, keep = _args(abi)
    mem.field = None
    rejects(b"neither a sphere field nor spheres", job, mem, pos, slots)
    job, mem, pos, slots, keep = _args(abi)
    job.det_x = 0
    rejects(b"bad detector geometry", job, mem, pos, slots)

    # positions
    for field in ("offsets_host", "thickness"):
        job, mem, pos, slots, keep = _args(abi)
        setattr(pos[0], field, None)
        rejects(b"position 0 lacks offsets or a thickness buffer", job, mem, pos, slots)
    for field in ("out_sample", "out_ref"):
        job, mem, pos, slots, keep = _args(abi)
        setattr(pos[0], field, None)
        rejects(b"position 0 has incomplete detector outputs", job, mem, pos, slots)
    job, mem, pos, slots, keep = _args(abi, first=1)
    rejects(b"position 0 has incomplete detector outputs", job, mem, pos, slots)      # position 0 needs propag, white
    pos[0].out_propag = 16
    rejects(b"position 0 has incomplete detector outputs", job, mem, pos, slots)
    for field in ("probe_start", "probe_end"):
        job, mem, pos, slots, keep = _args(abi)
        setattr(pos[0], field, 16)
        rejects(b"position 0 has probe events", job, mem, pos, slots)

    # slots
    job, mem, pos, slots, keep = _args(abi, n_slots=2)
    slots[1].plan = None
    rejects(b"slot 1 has no plan", job, mem, pos, slots)
    for field in ("wave_a", "wave_b", "acc_sample", "acc_ref", "acc_propag", "acc_white"):
        job, mem, pos, slots, keep = _args(abi, n_slots=2)
        setattr(slots[1], field, None)
        rejects(b"slot 1 lacks a wave or an accumulator", job, mem, pos, slots)
    job, mem, pos, slots, keep = _args(abi, n_slots=3)
    slots[2].plan = slots[0].plan
    rejects(b"slot 2 shares its plan with another slot", job, mem, pos, slots)

    # the per-energy checks of paresis_fresnel_run
    job, mem, pos, slots, keep = _args(abi)
    keep[0][1][0].n_membrane = 0
    rejects(b"energy 0: no membrane layer", job, mem, pos, slots)
    job, mem, pos, slots, keep = _args(abi)
    keep[0][1][0].membrane_host = None
    rejects(b"energy 0: no membrane layer", job, mem, pos, slots)
    for n in (0, abi.MAX_LAYERS + 1):
        job, mem, pos, slots, keep = _args(abi)
        keep[0][1][0].n_sample = n
        rejects(b"energy 0: need 1 .. PARESIS_MAX_LAYERS sample layers", job, mem, pos, slots)
    job, mem, pos, slots, keep = _args(abi)
    keep[0][1][0].sample[0].thickness = None
    rejects(b"energy 0: null sample map", job, mem, pos, slots)
    for field in ("reference", "to_object", "to_detector"):
        job, mem, pos, slots, keep = _args(abi)
        setattr(keep[0][1][0], field, None)
        rejects(b"energy 0: null transfer kernel", job, mem, pos, slots)

    # a NULL membrane map stands for the position's map here only: paresis_fresnel_run still refuses it
    job, mem, pos, slots, keep = _args(abi)
    keep[0][0][0].thickness = None
    assert abi.lib.paresis_fresnel_run(ctypes.byref(job), None) == ERR_ARG
    assert b"null membrane map" in abi.lib.paresis_last_error()


@pytest.mark.gpu
def test_run_positions_rejects_plans_that_do_not_fit():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from paresis_b200 import _cabi as abi, hostmath as hm
    plan, other = abi.FresnelPlan(64, 64, 15), abi.FresnelPlan(48, 48, 15)
    hx, hy, _ = hm.fresnel_vectors(64, 64, 15, (64, 64), 1.0, 1.0, 52.0, 1.5)
    kern = plan.kernel(torch.as_tensor(hx, device="cuda"), torch.as_tensor(hy, device="cuda"))
    torch.cuda.synchronize()

    def rejects(msg, job, mem, pos, slots):
        assert _call(abi, job, mem, pos, slots) == ERR_ARG
        assert msg in abi.lib.paresis_last_error(), abi.lib.paresis_last_error()

    def args(n_slots):
        job, mem, pos, slots, keep = _args(abi, n_slots=n_slots)
        en = keep[0][1][0]
        en.reference = en.to_object = en.to_detector = kern._h.value
        for sl in slots:
            sl.plan = plan._h.value
        return job, mem, pos, slots, keep

    # a slot whose plan is of another size than the transfer kernels
    job, mem, pos, slots, keep = args(2)
    slots[1].plan = other._h.value
    rejects(b"energy 0: a transfer kernel was prepared for a plan of another size", job, mem, pos, slots)
    # two slots on one plan
    job, mem, pos, slots, keep = args(2)
    rejects(b"slot 1 shares its plan with another slot", job, mem, pos, slots)
    # no sphere field: every slot needs the raster work
    job, mem, pos, slots, keep = args(1)
    mem.field, mem.spheres, mem.n_spheres, mem.pix_um, mem.margin = None, 16, 100, 1.0, 4
    slots[0].raster_work, slots[0].raster_work_bytes = 16, 0
    rejects(b"slot 0: the membrane has no sphere field and the raster work is smaller", job, mem, pos, slots)


# ------------------------------------------------------------------ cases
@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from paresis_b200 import workspace
    from paresis_b200.hostio import imageio
    from test_gpu_many_materials import MATERIALS, _six_maps
    ws = workspace.make_workspace(str(tmp_path_factory.mktemp("ws_fresnel_positions")))
    folder = os.path.join(ws, "Samples", "ManyMaterials")
    os.makedirs(folder)
    pix = 6.0 / 2 / (145.2 / 141.6)
    for m, t in enumerate(_six_maps((192, 256), pix)):
        imageio.write_tiff(os.path.join(folder, "m%d_%s.tif" % (m, MATERIALS[m])), t)
    old = os.getcwd()
    workspace.enter(ws)
    yield importlib.import_module("Experiment")
    os.chdir(old)


class Scan:
    """A Fresnel scene whose membrane is cut per position (Layer(PER_POSITION)), its engine, the membrane plan and three
    positions' offsets drawn from one seed."""

    def __init__(self, shim, name, noise=False, n_pos=3):
        from paresis_b200 import engine, geometry
        from test_gpu_fresnel_shard import Case
        self.name = name
        if name == "cufft_grid":
            # 100 x 90 study grid: convolution lengths 200 and 180, both axes on the cuFFT path; the membrane of a
            # shipped experiment cut at that size
            c = Case(shim, "cufft_grid", noise=noise)
            host = Case(shim, "Small_sphere_mono").e.myMembrane
            s = c.setup
            self.eng = c.eng
            self.plan = geometry.MembranePlan(host, 100, 90, host.membranePixelSize)
            membrane = [engine.Layer(engine.PER_POSITION, *c._coeffs(c.mem_db, 0)), engine.Layer(6e-3, *c._coeffs(c.mem_db, 1))]
            self.scene = engine.Scene(s.study_dims, s.study_pixel_um, s.os, s.det_dims, s.det_pixel_um, s.psf_sigma, s.d1, s.d2,
                                      s.d3, s.mean_shot_count, s.spectrum, s.source_size_um, s.energy_sampling,
                                      list(s.thresholds), membrane, c._smp_layers)
            self.case = None
        else:
            self.case = c = Case(shim, name, noise=noise)
            e = c.e
            mem = e.myMembrane
            dims = e.exp_dict['studyDimensions']
            self.eng = c.eng
            self.plan = geometry.MembranePlan(mem, dims[0], dims[1], mem.membranePixelSize)
            self.scene = e._scene(c.thresholds, per_position_membrane=True)
        assert self.plan.field() is not None
        np.random.seed(77)
        self.offsets = [self.plan.draw_offsets() for _ in range(n_pos)]

    def scene_with(self, grains):
        """The scene with the position's map in place of PER_POSITION (what compute_fresnel takes)."""
        from paresis_b200 import engine
        s = copy.copy(self.scene)
        s.membrane = [engine.Layer(grains, L.delta, L.beta) if L.map is engine.PER_POSITION else L for L in self.scene.membrane]
        return s

    def one_by_one(self, p, point):
        """Position p at point number ``point`` through the per-position API: -> thickness, images, sums (numpy)."""
        from paresis_b200 import geometry
        eng = self.eng
        grains = torch.empty((eng.nx, eng.ny), device=eng.device, dtype=torch.float32)
        geometry._cut_membrane(self.plan, self.offsets[p], self.plan.pix, grains)
        out = eng.compute_fresnel(self.scene_with(grains), point)
        n_e = len(self.scene.spectrum)
        keys = ("sample", "reference") + (("propag", "white") if point == 0 else ())
        return grains.cpu().numpy(), {k: out[k].cpu().numpy() for k in keys}, eng.means[:n_e].cpu().numpy().copy()


POSITION_CASES = ["Small_sphere_mono", "B200_small_poly3", "Small_six_materials_poly3", "Small_sphere_air_plate_CsI",
                  "cufft_grid", "B200_2048_mono"]


# ------------------------------------------------------------------ one call against the position-by-position API
@pytest.mark.gpu
@pytest.mark.parametrize("noise", [False, True])
@pytest.mark.parametrize("name", POSITION_CASES)
def test_positions_in_one_call_match_one_by_one(shim, name, noise):
    sc = Scan(shim, name, noise=noise)
    eng = sc.eng
    orders = ([0, 1, 2], [1, 0, 2])
    single = {}
    for points in orders:
        for p, point in enumerate(points):
            if (p, point) not in single:
                single[(p, point)] = sc.one_by_one(p, point)
    for slots in (1, 2, 3):
        for points in orders:
            out = eng.compute_fresnel_positions(sc.scene, sc.plan, sc.offsets, points, n_slots=slots)
            torch.cuda.synchronize()
            what = (name, noise, slots, points)
            assert out["firsts"] == [points.index(0)], what
            for p, point in enumerate(points):
                thick, imgs, sums = single[(p, point)]
                assert np.array_equal(out["thickness"][p].cpu().numpy(), thick), what + (p, "thickness")
                assert np.array_equal(out["sample"][p].cpu().numpy(), imgs["sample"]), what + (p, "sample")
                assert np.array_equal(out["reference"][p].cpu().numpy(), imgs["reference"]), what + (p, "reference")
                # fp64 atomicAdd order of the reference beam's sum
                assert np.allclose(out["sums"][p].cpu().numpy(), sums, rtol=1e-12, atol=0), what + (p, "sums")
                if point == 0:
                    assert np.array_equal(out["propag"][0].cpu().numpy(), imgs["propag"]), what + (p, "propag")
                    assert np.array_equal(out["white"][0].cpu().numpy(), imgs["white"]), what + (p, "white")


@pytest.mark.gpu
def test_positions_reuse_buffers_and_skip_sums(shim):
    """``buffers`` of an earlier call are written in place; want_means=False leaves the sums alone."""
    sc = Scan(shim, "B200_small_poly3")
    first = sc.eng.compute_fresnel_positions(sc.scene, sc.plan, sc.offsets, [0, 1, 2])
    want = {k: first[k].cpu().numpy() for k in ("sample", "reference", "propag", "white", "sums")}
    bufs = first["buffers"]
    for t in bufs.values():
        t.fill_(-1.0)
    again = sc.eng.compute_fresnel_positions(sc.scene, sc.plan, sc.offsets, [0, 1, 2], want_means=False, buffers=bufs)
    assert again["buffers"] is bufs
    for k in ("sample", "reference", "propag", "white"):
        assert np.array_equal(again[k].cpu().numpy(), want[k]), k
    assert (again["sums"].cpu().numpy() == -1.0).all()


# ------------------------------------------------------------------ against the fp64 oracle
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["Small_sphere_mono", "B200_small_poly3"])
def test_positions_match_the_oracle(shim, name):
    sc = Scan(shim, name, n_pos=2)
    out = sc.eng.compute_fresnel_positions(sc.scene, sc.plan, sc.offsets, [0, 1])
    torch.cuda.synchronize()
    e = sc.case.e
    support = np.full(out["thickness"].shape[1:], e.myMembrane.myPMMAThickness * 1e-6)
    for p in (0, 1):
        e.myMembrane.myGeometry = np.array([out["thickness"][p].cpu().numpy().astype(np.float64), support])
        want = sc.case.oracle(p)
        got = [out["sample"][p], out["reference"][p]] + ([out["propag"][0], out["white"][0]] if p == 0 else [])
        for i, g in enumerate(got):
            g = g.cpu().numpy()
            assert g.shape == want[i].shape
            assert rel_l2(g, want[i]) < 1e-5, (name, p, i)


# ------------------------------------------------------------------ a membrane without a sphere field
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["Small_sphere_mono", "B200_small_poly3"])
def test_raster_fallback_matches_the_field(shim, name):
    from paresis_b200 import geometry
    sc = Scan(shim, name)
    field = sc.eng.compute_fresnel_positions(sc.scene, sc.plan, sc.offsets, [0, 1, 2], n_slots=2)
    field = {k: field[k].cpu().numpy() for k in ("thickness", "sample", "reference", "propag", "white", "sums")}
    raster_plan = geometry.MembranePlan(sc.case.e.myMembrane, sc.plan.dim_x, sc.plan.dim_y, sc.plan.pix)
    raster_plan.field = lambda: None          # paresis_membrane.field = NULL: each position is rasterised
    assert sc.eng._membrane(raster_plan)[0].field is None
    raster = sc.eng.compute_fresnel_positions(sc.scene, raster_plan, sc.offsets, [0, 1, 2], n_slots=2)
    torch.cuda.synchronize()
    for k in ("thickness", "sample", "reference", "propag", "white"):
        got = raster[k].cpu().numpy()
        assert got.shape == field[k].shape
        for p in range(got.shape[0]):
            assert rel_l2(got[p], field[k][p]) < 1e-6, (name, k, p)
    assert np.allclose(raster["sums"].cpu().numpy(), field["sums"], rtol=1e-6, atol=0)


@pytest.mark.gpu
def test_compute_fresnel_refuses_a_per_position_membrane(shim):
    """A PER_POSITION map only has a meaning inside a many-positions call: the single call reports it as a NULL map."""
    from paresis_b200 import _cabi as abi
    sc = Scan(shim, "Small_sphere_mono", n_pos=1)
    with pytest.raises(abi.ParesisError, match="null membrane map"):
        sc.eng.compute_fresnel(sc.scene, 1)
