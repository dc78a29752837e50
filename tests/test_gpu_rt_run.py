"""The ray-tracing run entries (paresis_rt_run, paresis_rt_run_positions, engine.ImageFormation.compute_rt_positions).

Checked here:
  - argument checks of both entries, all before any CUDA call (host only: bogus device addresses are never touched).
    Each case sits where an entry that checked as it went would already have launched: after a good energy or
    position, with a dirty I_bs, on the slot path and on the several-positions-per-launch path;
  - slots with a detector kernel wide enough for the work-buffer passes (PSF half-width >= 50 at oversampling 2), at 2
    and 3 slots, against position-by-position compute_rt: every slot has a work buffer of its own;
  - probe events (detector and membrane cut, at 1 and 2 slots) leave the images as they are and time something.
"""
import copy
import ctypes
import os

import numpy as np
import pytest

from conftest import rel_l2

torch = pytest.importorskip("torch")

ERR_ARG = 2
VP = 1 << 20                                            # a fake device address: never dereferenced


# ------------------------------------------------------------------ argument checks (no device)
def _energies(abi, first_maps=True):
    """Two energies, each closing a bin: hop1 = [map], hop2 = [map, sample], propag = [sample].  ``first_maps``: the
    membrane maps are real pointers (paresis_rt_run); otherwise NULL, the position's map (paresis_rt_run_positions)."""
    en = (abi.RtEnergy * 2)()
    for e in en:
        e.n_hop1, e.n_hop2, e.n_propag, e.close_bin = 1, 2, 1, 1
        e.hop1[0].thickness = VP if first_maps else None
        e.hop2[0].thickness, e.hop2[1].thickness = (VP if first_maps else None), VP + 4096
        e.propag[0].thickness = VP + 4096
        e.intensity_membrane = e.intensity_propag = 1.0
    return en


def _job(abi, first=1, outputs=True, maps=True):
    """A paresis_rt_run job on fake, distinct pointers, with I_bs dirty (its memsets would be the first CUDA calls)."""
    en = _energies(abi, maps)
    job = abi.RtJob()
    job.nx, job.ny, job.oversampling, job.det_x, job.det_y = 64, 64, 2, 32, 32
    job.first_point, job.n_energies, job.energies_host = first, 2, en
    for i, name in enumerate(("i_bs", "acc_sample", "acc_ref", "acc_propag", "acc_white")):
        setattr(job, name, VP * 2 + 4096 * i)
    if outputs:
        for i, name in enumerate(("out_sample", "out_ref", "out_propag", "out_white")):
            setattr(job, name, VP * 3 + 4096 * i)
    job.i_bs_dirty = 1
    return job, en


SLOT_IMAGES = ("i_bs", "acc_sample", "acc_ref", "acc_propag", "acc_white", "detect_work")


def _positions_args(abi, n_pos=2, n_slots=2, first=0, per_launch=0):
    """A paresis_rt_run_positions call on fake, distinct pointers; position 0 is the first point if ``first``."""
    job, en = _job(abi, first=0, outputs=False, maps=False)
    job.positions_per_launch = per_launch
    mem = abi.Membrane()
    mem.field, mem.field_x, mem.field_y, mem.n_layers = VP, 128, 128, 1
    offs = (ctypes.c_int64 * 2)(0, 0)
    pos = (abi.RtPosition * n_pos)()
    for p, ps in enumerate(pos):
        ps.offsets_host = ctypes.cast(offs, ctypes.POINTER(ctypes.c_int64))
        ps.thickness, ps.out_sample, ps.out_ref = VP * (8 + p), VP * (8 + p) + 4096, VP * (8 + p) + 8192
        if first and p == 0:
            ps.first_point, ps.out_propag, ps.out_white = 1, VP * 7, VP * 7 + 4096
    slots = (abi.RtSlot * n_slots)()
    for k, sl in enumerate(slots):
        for i, name in enumerate(SLOT_IMAGES):
            setattr(sl, name, VP * (32 + k) + 4096 * i)
        sl.i_bs_dirty = 1
    return job, mem, pos, slots, (en, offs)


def _rejects(abi, rc, who, msg):
    assert rc == ERR_ARG, (msg, rc, abi.lib.paresis_last_error())
    err = abi.lib.paresis_last_error()
    assert err.startswith(who) and msg in err, (msg, err)


def test_run_rejects_bad_arguments():
    from paresis_b200 import _cabi as abi

    def rejects(msg, job):
        _rejects(abi, abi.lib.paresis_rt_run(ctypes.byref(job) if job is not None else None, None), b"paresis_rt_run:", msg)

    rejects(b"null job", None)
    job, en = _job(abi)
    job.energies_host = None
    rejects(b"no energies", job)
    job, en = _job(abi)
    job.n_energies = 0
    rejects(b"no energies", job)
    job, en = _job(abi)
    job.ny = 2
    rejects(b"bad frame 64 x 2", job)
    for name in ("i_bs", "acc_sample", "acc_ref", "acc_propag"):
        job, en = _job(abi)
        setattr(job, name, None)
        rejects(b"null object-plane buffer or accumulator", job)
    # outputs: all of them or none; acc_white with outputs at position 0
    for first, name in ((0, "out_sample"), (0, "out_ref"), (1, "out_propag"), (1, "out_white"), (1, "acc_white")):
        job, en = _job(abi, first=first)
        setattr(job, name, None)
        rejects(b"incomplete detector outputs (all of them, or none to accumulate only)", job)
    job, en = _job(abi, first=0, outputs=False)
    job.out_ref = VP
    rejects(b"incomplete detector outputs", job)
    for name in ("oversampling", "det_x", "det_y"):
        job, en = _job(abi)
        setattr(job, name, 0)
        rejects(b"bad detector geometry", job)
    for name in ("dx_pad", "dy_pad"):
        job, en = _job(abi)
        setattr(job, name, VP * 5)
        rejects(b"dx_pad and dy_pad come together", job)
    job, en = _job(abi)
    job.i_bs_group[1] = VP * 6                             # after a NULL entry
    rejects(b"an i_bs_group entry follows a NULL one", job)

    # per energy: energy 1 is wrong, energy 0 would already have run
    for field, n, msg in (("n_hop1", 0, b"energy 1: need 1 .. PARESIS_MAX_LAYERS membrane maps"),
                          ("n_hop1", abi.MAX_LAYERS + 1, b"energy 1: need 1 .. PARESIS_MAX_LAYERS membrane maps"),
                          ("n_hop2", 0, b"energy 1: need 1 .. PARESIS_MAX_LAYERS membrane + sample maps"),
                          ("n_hop2", abi.MAX_LAYERS + 1, b"energy 1: need 1 .. PARESIS_MAX_LAYERS membrane + sample maps"),
                          ("n_propag", 0, b"energy 1: need 1 .. PARESIS_MAX_LAYERS sample maps in the sample-only hop"),
                          ("n_propag", abi.MAX_LAYERS + 1, b"energy 1: need 1 .. PARESIS_MAX_LAYERS sample maps")):
        job, en = _job(abi)
        setattr(en[1], field, n)
        rejects(msg, job)
    for hop, msg in (("hop1", b"energy 1: null membrane map"), ("hop2", b"energy 1: null object-hop map"),
                     ("propag", b"energy 1: null sample map")):
        job, en = _job(abi)
        getattr(en[1], hop)[0].thickness = None
        rejects(msg, job)
    # accumulate only (no outputs) keeps the per-energy checks
    job, en = _job(abi, outputs=False)
    en[1].hop2[1].thickness = None
    rejects(b"energy 1: null object-hop map", job)


def test_run_positions_rejects_bad_arguments():
    from paresis_b200 import _cabi as abi
    who = b"paresis_rt_run_positions:"

    def call(job, mem, pos, slots, n_pos=None, n_slots=None):
        return abi.lib.paresis_rt_run_positions(
            ctypes.byref(job) if job is not None else None, ctypes.byref(mem) if mem is not None else None, pos,
            len(pos) if n_pos is None else n_pos, slots, len(slots) if n_slots is None else n_slots, None)

    def rejects(msg, *args, **kw):
        _rejects(abi, call(*args, **kw), who, msg)

    job, mem, pos, slots, keep = _positions_args(abi)
    rejects(b"null job, membrane, positions or slots", None, mem, pos, slots)
    rejects(b"null job, membrane, positions or slots", job, None, pos, slots)
    rejects(b"null job, membrane, positions or slots", job, mem, None, slots, n_pos=1)
    rejects(b"null job, membrane, positions or slots", job, mem, pos, None, n_slots=1)
    rejects(b"n_slots >= 1", job, mem, pos, slots, n_slots=0)
    rejects(b"n_positions >= 0", job, mem, pos, slots, n_pos=-1)
    assert call(job, mem, pos, slots, n_pos=0) == 0       # nothing to do is fine

    # on the slot path and on the several-positions-per-launch path
    for per in (0, 2):
        def fresh(**kw):
            return _positions_args(abi, per_launch=per, **kw)

        job, mem, pos, slots, keep = fresh()
        job.energies_host = None
        rejects(b"no energies", job, mem, pos, slots)
        job, mem, pos, slots, keep = fresh()
        job.nx = 2
        rejects(b"bad frame", job, mem, pos, slots)
        job, mem, pos, slots, keep = fresh()
        mem.field = None
        rejects(b"neither a sphere field nor spheres", job, mem, pos, slots)
        job, mem, pos, slots, keep = fresh()
        job.det_y = 0
        rejects(b"bad detector geometry", job, mem, pos, slots)

        # positions: position 1 is wrong, position 0 would already have run
        for field in ("offsets_host", "thickness"):
            job, mem, pos, slots, keep = fresh()
            setattr(pos[1], field, None)
            rejects(b"position 1 lacks offsets or a thickness buffer", job, mem, pos, slots)
        for field in ("out_sample", "out_ref"):
            job, mem, pos, slots, keep = fresh()
            setattr(pos[1], field, None)
            rejects(b"position 1 has incomplete detector outputs", job, mem, pos, slots)
        job, mem, pos, slots, keep = fresh(n_pos=3)
        pos[1].first_point = 1                             # position 0 runs in a group first, then position 1 alone
        rejects(b"position 1 has incomplete detector outputs", job, mem, pos, slots)

        # slots
        for field in ("i_bs", "acc_sample", "acc_ref", "acc_propag", "acc_white"):
            job, mem, pos, slots, keep = fresh()
            setattr(slots[1], field, None)
            rejects(b"slot 1 lacks an object-plane buffer or an accumulator", job, mem, pos, slots)
        job, mem, pos, slots, keep = fresh()
        slots[1].i_bs_group[1] = VP * 60                   # after a NULL entry
        rejects(b"slot 1: an i_bs_group entry follows a NULL one", job, mem, pos, slots)
        # an image of one slot handed to another, as the same image or as another one: slots run concurrently
        for mine, theirs in (("i_bs", "i_bs"), ("acc_ref", "acc_sample"), ("acc_white", "acc_propag"),
                             ("detect_work", "detect_work"), ("detect_work", "i_bs"), ("group", "i_bs"), ("group", "group")):
            job, mem, pos, slots, keep = fresh(n_slots=3)
            for sl in slots:
                sl.i_bs_group[0] = sl.i_bs + 65536
            src = slots[0].i_bs_group[0] if theirs == "group" else getattr(slots[0], theirs)
            if mine == "group":
                slots[2].i_bs_group[0] = src
            else:
                setattr(slots[2], mine, src)
            rejects(b"slot 2 shares an image buffer with another slot", job, mem, pos, slots)

        # per energy: energy 1 is wrong; the NULL hop1 / hop2 maps (the position's membrane) pass
        for field, n, msg in (("n_hop1", 0, b"energy 1: need 1 .. PARESIS_MAX_LAYERS membrane maps"),
                              ("n_hop2", abi.MAX_LAYERS + 1, b"energy 1: need 1 .. PARESIS_MAX_LAYERS membrane + sample maps")):
            job, mem, pos, slots, keep = fresh()
            setattr(keep[0][1], field, n)
            rejects(msg, job, mem, pos, slots)
        # the sample-only hop is checked when a position is the first point
        job, mem, pos, slots, keep = fresh(first=1)
        keep[0][1].n_propag = 0
        rejects(b"energy 1: need 1 .. PARESIS_MAX_LAYERS sample maps in the sample-only hop", job, mem, pos, slots)
        job, mem, pos, slots, keep = fresh(first=1)
        keep[0][1].propag[0].thickness = None              # never the position's map
        rejects(b"energy 1: null sample map", job, mem, pos, slots)

    # without a sphere field the membrane is rasterised: every slot needs raster work (the NULL maps were accepted)
    job, mem, pos, slots, keep = _positions_args(abi)
    mem.field, mem.spheres, mem.n_spheres, mem.pix_um, mem.margin = None, 16, 100, 1.0, 4
    slots[0].raster_work, slots[0].raster_work_bytes = 1 << 30, 1 << 40
    rejects(b"slot 1: the membrane has no sphere field and the raster work is smaller", job, mem, pos, slots)


# ------------------------------------------------------------------ on the GPU
@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from paresis_b200 import workspace
    import importlib
    ws = workspace.make_workspace(str(tmp_path_factory.mktemp("ws_rt_run")))
    old = os.getcwd()
    workspace.enter(ws)
    yield importlib.import_module("Experiment")
    os.chdir(old)


class Scan:
    """A plain (non-scattering) scene whose membrane is cut per position, its engine, the membrane plan and the offsets of
    ``n_pos`` positions drawn from one seed.  ``psf_sigma``: the detector PSF in its place (None: the experiment's)."""

    def __init__(self, shim, name="Small_sphere_mono", n_pos=4, psf_sigma=None):
        from paresis_b200 import geometry
        e = shim.Experiment(dict(experimentName=name, filepath="unused/", overSampling=2, nbExpPoints=n_pos,
                                 simulation_type="RayT", expID="t", poissonNoise=False, seed=11))
        self.eng = e._get_engine()
        mem = e.myMembrane
        dims = e.exp_dict['studyDimensions']
        self.plan = geometry.MembranePlan(mem, dims[0], dims[1], mem.membranePixelSize)
        self.scene = e._scene(list(e._open_bins(0)), per_position_membrane=True)
        if psf_sigma is not None:
            self.scene = copy.copy(self.scene)
            self.scene.psf_sigma = float(psf_sigma)
        assert not self.eng.scatters(self.scene)
        np.random.seed(77)
        self.offsets = [self.plan.draw_offsets() for _ in range(n_pos)]

    def one_by_one(self, p, point):
        """Position p at point number ``point`` through compute_rt -> {image name: numpy array}."""
        from paresis_b200 import engine, geometry
        eng = self.eng
        grains = torch.empty((eng.nx, eng.ny), device=eng.device, dtype=torch.float32)
        geometry._cut_membrane(self.plan, self.offsets[p], self.plan.pix, grains)
        s = copy.copy(self.scene)
        s.membrane = [engine.Layer(grains, L.delta, L.beta) if L.map is engine.PER_POSITION else L for L in self.scene.membrane]
        out = eng.compute_rt(s, point)
        keys = ("sample", "reference") + (("propag", "white") if point == 0 else ())
        return {k: out[k].cpu().numpy() for k in keys}

    def check(self, out, points, single, what):
        for p, point in enumerate(points):
            got = {"sample": out["sample"][p], "reference": out["reference"][p]}
            if point == 0:
                got.update(propag=out["propag"][0], white=out["white"][0])
            for k, g in got.items():
                assert rel_l2(g.cpu().numpy(), single[p][k]) < 1e-6, what + (p, k)


@pytest.mark.gpu
def test_slots_with_a_wide_psf_match_one_by_one(shim):
    """A PSF half-width of 51 at oversampling 2 takes the detector's separable passes through its work buffer; positions
    on 2 and 3 slots run them concurrently, each slot through a buffer of its own."""
    from paresis_b200 import hostmath as hm
    sc = Scan(shim, psf_sigma=17.0)
    assert hm.gaussian_half_width(sc.scene.psf_sigma) >= 50 and sc.eng.os == 2
    points = list(range(len(sc.offsets)))
    single = [sc.one_by_one(p, point) for p, point in enumerate(points)]
    for slots in (2, 3):
        out = sc.eng.compute_rt_positions(sc.scene, sc.plan, sc.offsets, points, n_slots=slots)
        torch.cuda.synchronize()
        sc.eng.check_flag()
        sc.check(out, points, single, ("wide psf", slots))


@pytest.mark.gpu
@pytest.mark.parametrize("label", ["detect", "raster_spheres"])
def test_probe_events_leave_the_images_alone(shim, label):
    """Probe events (paresis_rt_position.probe_start / probe_end) time one kernel of a position, which then runs alone;
    the images are those of the same call without them."""
    sc = Scan(shim)
    points = list(range(len(sc.offsets)))
    plain = sc.eng.compute_rt_positions(sc.scene, sc.plan, sc.offsets, points, n_slots=2)
    torch.cuda.synchronize()
    single = [{k: plain[k][p].cpu().numpy() for k in ("sample", "reference")} for p in points]
    single[0].update(propag=plain["propag"][0].cpu().numpy(), white=plain["white"][0].cpu().numpy())
    for slots, probed in ((1, points), (2, [1])):
        events = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) if p in probed else None
                  for p in points]
        out = sc.eng.compute_rt_positions(sc.scene, sc.plan, sc.offsets, points, n_slots=slots, probe_label=label,
                                          probe_events=events)
        torch.cuda.synchronize()
        sc.eng.check_flag()
        sc.check(out, points, single, (label, slots))
        for p in probed:
            e0, e1 = events[p]
            assert e0.elapsed_time(e1) > 0, (label, slots, p)
