"""Many membrane positions of a scattering (dark-field) sample in one library call (paresis_df_run_positions,
engine.ImageFormation.compute_df_positions).

Checked here:
  - argument checks, all before any CUDA call (host only: bogus device addresses are never touched);
  - the call against the position-by-position compute_rt on maps cut at the same offsets, at 1, 2 and 3 slots, with
    position 0 first and not first: thickness maps bit for bit; with noise off, images and the dark-field map to 1e-6
    relative L2 (the many-positions hops use full-height tiles, so their fp32 atomics add in another order); with noise
    on, the same Philox stream; the per-energy sums to rtol 1e-6;
  - the images and the dark-field map against the fp64 oracle;
  - a membrane without a sphere field (rasterised per position) against the field path;
  - reused output buffers, and the refusals of compute_df_positions / compute_rt_positions.
Cases: the five of test_gpu_dark_field_run (a Lung sphere, three energies in two bins, six materials with one Lung so
that the hops see mixed maps, two materials that both scatter, air + plate + scintillator) and the 2048^2 benchmark grid
with its sample made of Lung.
"""
import contextlib
import copy
import ctypes
import io
import os

import numpy as np
import pytest

from conftest import rel_l2
from test_gpu_dark_field_run import _agree, _experiment, _oracle_df, _workspace

torch = pytest.importorskip("torch")

ERR_ARG = 2
WHO = b"paresis_df_run_positions"


# ------------------------------------------------------------------ argument checks (no device)
def _args(abi, n_pos=1, n_slots=1, first=0):
    """A well-formed call on fake, distinct pointers (nothing is dereferenced before the checks fail)."""
    vp = 1 << 20
    en = (abi.RtEnergy * 1)()
    en[0].n_hop1, en[0].n_hop2, en[0].n_propag, en[0].close_bin = 1, 2, 1, 1
    en[0].hop1[0].thickness = None                      # the position's membrane map
    en[0].hop2[0].thickness, en[0].hop2[1].thickness = None, vp
    en[0].propag[0].thickness = vp
    df = (abi.DfEnergy * 1)()
    df[0].scatter_map, df[0].angle_coeff = vp, 1.0
    job = abi.DfJob()
    r = job.rt
    r.nx, r.ny, r.oversampling, r.det_x, r.det_y = 64, 64, 2, 32, 32
    r.n_energies, r.energies_host = 1, en
    job.energies_df_host = df
    mem = abi.Membrane()
    mem.field, mem.field_x, mem.field_y, mem.n_layers = vp, 128, 128, 1
    offs = (ctypes.c_int64 * 2)(0, 0)
    pos = (abi.DfPosition * n_pos)()
    for p in pos:
        p.rt.offsets_host = ctypes.cast(offs, ctypes.POINTER(ctypes.c_int64))
        p.rt.thickness = p.rt.out_sample = p.rt.out_ref = vp
        p.rt.first_point = first
        if first:
            p.rt.out_propag = p.rt.out_white = p.dark_field = vp
    slots = (abi.DfSlot * n_slots)()
    for k, sl in enumerate(slots):
        for i, name in enumerate(SLOT_IMAGES):
            setattr(sl, name, vp * (2 + k) + 4096 * i)
    return job, mem, pos, slots, (en, df, offs)


SLOT_IMAGES = ("i_bs", "acc_sample", "acc_ref", "acc_propag", "acc_white", "angle", "plain", "scattered", "clean", "moved",
               "detect_work")


def _call(abi, job, mem, pos, slots, n_pos=None, n_slots=None):
    return abi.lib.paresis_df_run_positions(
        ctypes.byref(job) if job is not None else None, ctypes.byref(mem) if mem is not None else None, pos,
        len(pos) if n_pos is None else n_pos, slots, len(slots) if n_slots is None else n_slots, None)


def test_run_positions_rejects_bad_arguments():
    from paresis_b200 import _cabi as abi

    def rejects(msg, *args, **kw):
        assert _call(abi, *args, **kw) == ERR_ARG, msg
        err = abi.lib.paresis_last_error()
        assert err.startswith(WHO) and msg in err, (msg, err)

    job, mem, pos, slots, keep = _args(abi)
    rejects(b"null job, membrane, positions or slots", None, mem, pos, slots)
    rejects(b"null job, membrane, positions or slots", job, None, pos, slots)
    rejects(b"null job, membrane, positions or slots", job, mem, None, slots, n_pos=1)
    rejects(b"null job, membrane, positions or slots", job, mem, pos, None, n_slots=1)
    rejects(b"n_slots >= 1", job, mem, pos, slots, n_slots=0)
    rejects(b"n_positions >= 0", job, mem, pos, slots, n_pos=-1)
    assert _call(abi, job, mem, pos, slots, n_pos=0) == 0        # nothing to do is fine

    def fresh(**kw):
        return _args(abi, **kw)

    job, mem, pos, slots, keep = fresh()
    job.rt.energies_host = None
    rejects(b"no energies", job, mem, pos, slots)
    job, mem, pos, slots, keep = fresh()
    job.energies_df_host = None
    rejects(b"no energies", job, mem, pos, slots)
    job, mem, pos, slots, keep = fresh()
    job.rt.nx = 2
    rejects(b"bad frame", job, mem, pos, slots)
    job, mem, pos, slots, keep = fresh()
    mem.field = None
    rejects(b"neither a sphere field nor spheres", job, mem, pos, slots)
    job, mem, pos, slots, keep = fresh()
    job.rt.det_x = 0
    rejects(b"bad detector geometry", job, mem, pos, slots)

    # positions
    for field in ("offsets_host", "thickness"):
        job, mem, pos, slots, keep = fresh()
        setattr(pos[0].rt, field, None)
        rejects(b"position 0 lacks offsets or a thickness buffer", job, mem, pos, slots)
    for field in ("out_sample", "out_ref"):
        job, mem, pos, slots, keep = fresh()
        setattr(pos[0].rt, field, None)
        rejects(b"position 0 has incomplete detector outputs", job, mem, pos, slots)
    for field in ("out_propag", "out_white"):
        job, mem, pos, slots, keep = fresh(first=1)
        setattr(pos[0].rt, field, None)
        rejects(b"position 0 has incomplete detector outputs", job, mem, pos, slots)
    for field in ("probe_start", "probe_end"):
        job, mem, pos, slots, keep = fresh()
        setattr(pos[0].rt, field, 16)
        rejects(b"position 0 has probe events", job, mem, pos, slots)
    job, mem, pos, slots, keep = fresh(n_pos=2)
    pos[1].dark_field = 1 << 30
    rejects(b"position 1: the dark-field map belongs to position 0", job, mem, pos, slots)

    # slots
    for field in ("i_bs", "acc_sample", "acc_ref", "acc_propag", "acc_white"):
        job, mem, pos, slots, keep = fresh(n_slots=2)
        setattr(slots[1], field, None)
        rejects(b"slot 1 lacks an object-plane buffer or an accumulator", job, mem, pos, slots)
    for field in ("angle", "plain", "scattered", "clean", "moved"):
        job, mem, pos, slots, keep = fresh(n_slots=2)
        setattr(slots[1], field, None)
        rejects(b"slot 1 lacks a dark-field scratch image", job, mem, pos, slots)
    # an image of one slot handed to another, as the same image or as another one: slots run concurrently
    for mine, theirs in (("moved", "moved"), ("angle", "clean"), ("i_bs", "i_bs"), ("acc_ref", "acc_sample"),
                         ("detect_work", "detect_work")):
        job, mem, pos, slots, keep = fresh(n_slots=3)
        setattr(slots[2], mine, getattr(slots[0], theirs))
        rejects(b"slot 2 shares an image buffer with another slot", job, mem, pos, slots)
    job, mem, pos, slots, keep = fresh(n_slots=2)
    for sl in slots:
        sl.detect_work = None                           # no detector work of its own is not a shared buffer
    mem.field, mem.spheres, mem.n_spheres, mem.pix_um, mem.margin = None, 16, 100, 1.0, 4
    rejects(b"slot 0: the membrane has no sphere field and the raster work is smaller", job, mem, pos, slots)

    # the per-energy checks of paresis_df_run; NULL hop1 / hop2 maps (the position's membrane) pass them
    for field, n, msg in (("n_hop1", 0, b"energy 0: need 1 .. PARESIS_MAX_LAYERS membrane maps"),
                          ("n_hop2", abi.MAX_LAYERS + 1, b"energy 0: need 1 .. PARESIS_MAX_LAYERS membrane + sample maps"),
                          ("n_hop2", 0, b"energy 0: need 1 .. PARESIS_MAX_LAYERS membrane + sample maps")):
        job, mem, pos, slots, keep = fresh()
        setattr(keep[0][0], field, n)
        rejects(msg, job, mem, pos, slots)
    job, mem, pos, slots, keep = fresh(first=1)
    keep[0][0].n_propag = 0
    rejects(b"energy 0: need 1 .. PARESIS_MAX_LAYERS sample maps in the sample-only hop", job, mem, pos, slots)
    job, mem, pos, slots, keep = fresh(first=1)
    keep[0][0].propag[0].thickness = None
    rejects(b"energy 0: null sample map", job, mem, pos, slots)
    job, mem, pos, slots, keep = fresh()
    keep[1][0].scatter_map = None
    rejects(b"energy 0: no scattering map", job, mem, pos, slots)
    # too little raster work is the first thing wrong here: the NULL membrane maps were accepted
    job, mem, pos, slots, keep = fresh(first=1)
    mem.field, mem.spheres, mem.n_spheres, mem.pix_um, mem.margin = None, 16, 100, 1.0, 4
    slots[0].raster_work, slots[0].raster_work_bytes = 1 << 30, 0
    rejects(b"slot 0: the membrane has no sphere field and the raster work is smaller", job, mem, pos, slots)

    # a NULL membrane map stands for the position's map here only: paresis_df_run still refuses it
    for hop, msg in (("hop1", b"null membrane map"), ("hop2", b"null object-hop map")):
        job, mem, pos, slots, keep = fresh()
        r = job.rt
        r.i_bs = r.acc_sample = r.acc_ref = r.acc_propag = r.acc_white = 1 << 20
        job.angle = job.plain = job.scattered = job.clean = job.moved = 1 << 20
        other = "hop2" if hop == "hop1" else "hop1"
        getattr(keep[0][0], other)[0].thickness = 1 << 20
        assert abi.lib.paresis_df_run(ctypes.byref(job), None) == ERR_ARG
        err = abi.lib.paresis_last_error()
        assert err.startswith(b"paresis_df_run:") and msg in err, err


# ------------------------------------------------------------------ cases
@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    old = os.getcwd()
    yield _workspace(str(tmp_path_factory.mktemp("ws_df_positions")))
    os.chdir(old)


def _lung_grid(shim, noise):
    """B200_2048_mono with its sample made of Lung (as tools/df_bench.py runs it)."""
    with contextlib.redirect_stdout(io.StringIO()):
        e = shim.Experiment(dict(experimentName="B200_2048_mono", filepath="unused/", overSampling=2, nbExpPoints=3,
                                 simulation_type="RayT", expID="t", poissonNoise=noise, seed=11))
        smp = e.mySampleofInterest
        smp.myMaterials = ["Lung"] * len(smp.myMaterials)
        smp.delta, smp.beta = [], []
        smp.getDeltaBeta(e.mySource.mySpectrum)
    return e, list(e._open_bins(0))


class Scan:
    """A scattering scene whose membrane is cut per position (Layer(PER_POSITION)), its engine, the membrane plan and
    the offsets of ``n_pos`` positions drawn from one seed."""

    def __init__(self, shim, name, noise=False, n_pos=3):
        from paresis_b200 import geometry
        if name == "B200_2048_mono":
            self.e, thresholds = _lung_grid(shim, noise)
        else:
            self.e, scene, _ = _experiment(shim, name, noise)
            thresholds = scene.thresholds
        e = self.e
        self.eng = e._get_engine()
        mem = e.myMembrane
        dims = e.exp_dict['studyDimensions']
        self.plan = geometry.MembranePlan(mem, dims[0], dims[1], mem.membranePixelSize)
        self.scene = e._scene(thresholds, per_position_membrane=True)
        assert self.eng.scatters(self.scene)
        assert self.plan.field() is not None
        np.random.seed(77)
        self.offsets = [self.plan.draw_offsets() for _ in range(n_pos)]

    def scene_with(self, grains):
        """The scene with the position's map in place of PER_POSITION (what compute_rt takes)."""
        from paresis_b200 import engine
        s = copy.copy(self.scene)
        s.membrane = [engine.Layer(grains, L.delta, L.beta) if L.map is engine.PER_POSITION else L for L in self.scene.membrane]
        return s

    def one_by_one(self, p, point):
        """Position p at point number ``point`` through compute_rt: -> thickness, images (+ dark_field), sums (numpy)."""
        from paresis_b200 import geometry
        eng = self.eng
        grains = torch.empty((eng.nx, eng.ny), device=eng.device, dtype=torch.float32)
        geometry._cut_membrane(self.plan, self.offsets[p], self.plan.pix, grains)
        out = eng.compute_rt(self.scene_with(grains), point)
        n_e = len(self.scene.spectrum)
        keys = ("sample", "reference") + (("propag", "white", "dark_field") if point == 0 else ())
        return grains.cpu().numpy(), {k: out[k].cpu().numpy() for k in keys}, eng.means[:n_e].cpu().numpy().copy()


POSITION_CASES = ["sphere_lung", "poly3_lung", "six_lung", "beeds", "plate_lung", "B200_2048_mono"]


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
            out = eng.compute_df_positions(sc.scene, sc.plan, sc.offsets, points, n_slots=slots)
            torch.cuda.synchronize()
            what = (name, noise, slots, points)
            first = points.index(0)
            assert out["firsts"] == [first], what
            assert out["dark_field"].shape == (1, eng.nx, eng.ny), what
            for p, point in enumerate(points):
                thick, imgs, sums = single[(p, point)]
                assert np.array_equal(out["thickness"][p].cpu().numpy(), thick), what + (p, "thickness")
                got = {"sample": out["sample"][p], "reference": out["reference"][p]}
                if point == 0:
                    got.update(propag=out["propag"][0], white=out["white"][0])
                for k, g in got.items():
                    g = g.cpu().numpy()
                    assert g.shape == imgs[k].shape, what + (p, k)
                    if noise:
                        _agree(g, imgs[k], True, what + (p, k))
                    else:
                        assert rel_l2(g, imgs[k]) < 1e-6, what + (p, k)
                assert np.allclose(out["sums"][p].cpu().numpy(), sums, rtol=1e-6, atol=0), what + (p, "sums")
                if point == 0:
                    assert np.abs(imgs["dark_field"]).max() > 0
                    assert rel_l2(out["dark_field"][0].cpu().numpy(), imgs["dark_field"]) < 1e-6, what + (p, "dark_field")


@pytest.mark.gpu
def test_positions_reuse_buffers_and_skip_sums(shim):
    """``buffers`` of an earlier call are written in place, the dark-field map zeroed first; want_means=False leaves the
    sums alone."""
    sc = Scan(shim, "poly3_lung")
    first = sc.eng.compute_df_positions(sc.scene, sc.plan, sc.offsets, [0, 1, 2])
    keys = ("sample", "reference", "propag", "white", "dark_field")
    want = {k: first[k].cpu().numpy() for k in keys}
    bufs = first["buffers"]
    for t in bufs.values():
        t.fill_(-1.0)
    again = sc.eng.compute_df_positions(sc.scene, sc.plan, sc.offsets, [0, 1, 2], want_means=False, buffers=bufs)
    assert again["buffers"] is bufs
    for k in keys:
        assert rel_l2(again[k].cpu().numpy(), want[k]) < 1e-6, k
    assert (again["sums"].cpu().numpy() == -1.0).all()


# ------------------------------------------------------------------ against the fp64 oracle
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sphere_lung", "poly3_lung"])
def test_positions_match_the_oracle(shim, name):
    sc = Scan(shim, name, n_pos=2)
    out = sc.eng.compute_df_positions(sc.scene, sc.plan, sc.offsets, [0, 1])
    torch.cuda.synchronize()
    e = sc.e
    support = np.full(out["thickness"].shape[1:], e.myMembrane.myPMMAThickness * 1e-6)
    for p in (0, 1):
        e.myMembrane.myGeometry = np.array([out["thickness"][p].cpu().numpy().astype(np.float64), support])
        want, dark = _oracle_df(e, p)
        got = {"sample": out["sample"][p], "reference": out["reference"][p]}
        if p == 0:
            got.update(propag=out["propag"][0], white=out["white"][0])
        for k, g in got.items():
            g = g.cpu().numpy()
            assert g.shape == want[k].shape
            assert rel_l2(g, want[k]) < 1e-5, (name, p, k)
        if p == 0:
            assert rel_l2(out["dark_field"][0].cpu().numpy(), dark) < 1e-5, (name, "dark_field")


# ------------------------------------------------------------------ a membrane without a sphere field
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sphere_lung", "poly3_lung"])
def test_raster_fallback_matches_the_field(shim, name):
    from paresis_b200 import geometry
    sc = Scan(shim, name)
    keys = ("thickness", "sample", "reference", "propag", "white", "dark_field")
    field = sc.eng.compute_df_positions(sc.scene, sc.plan, sc.offsets, [0, 1, 2], n_slots=2)
    field = {k: field[k].cpu().numpy() for k in keys + ("sums",)}
    raster_plan = geometry.MembranePlan(sc.e.myMembrane, sc.plan.dim_x, sc.plan.dim_y, sc.plan.pix)
    raster_plan.field = lambda: None          # paresis_membrane.field = NULL: each position is rasterised
    assert sc.eng._membrane(raster_plan)[0].field is None
    raster = sc.eng.compute_df_positions(sc.scene, raster_plan, sc.offsets, [0, 1, 2], n_slots=2)
    torch.cuda.synchronize()
    for k in keys:
        got = raster[k].cpu().numpy()
        assert got.shape == field[k].shape
        for p in range(got.shape[0]):
            assert rel_l2(got[p], field[k][p]) < 1e-6, (name, k, p)
    assert np.allclose(raster["sums"].cpu().numpy(), field["sums"], rtol=1e-6, atol=0)


# ------------------------------------------------------------------ refusals
@pytest.mark.gpu
def test_each_many_positions_call_refuses_the_other_kind_of_scene(shim):
    from paresis_b200 import engine
    sc = Scan(shim, "sphere_lung", n_pos=1)
    with pytest.raises(NotImplementedError, match="compute_df_positions"):
        sc.eng.compute_rt_positions(sc.scene, sc.plan, sc.offsets, [1])
    plain = copy.copy(sc.scene)
    plain.sample = [engine.Layer(L.map, L.delta, L.beta) for L in sc.scene.sample]
    assert not sc.eng.scatters(plain)
    with pytest.raises(NotImplementedError, match="compute_rt_positions"):
        sc.eng.compute_df_positions(plain, sc.plan, sc.offsets, [1])
