"""ctypes binding of ``libparesis_b200.so`` (the C ABI declared in ``include/paresis_b200.h``).

There is no fallback: if the library is missing or does not load, importing this module
raises.  PyTorch is used only for device memory and streams; tensors cross the boundary as
raw ``data_ptr()`` values.
"""
import ctypes
import os

import numpy as np
import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
# PARESIS_B200_LIB: another build of the same library in the package directory (the bounds-checked debug build)
LIB_PATH = os.path.join(_PKG, os.path.basename(os.environ.get("PARESIS_B200_LIB", "libparesis_b200.so")))

OK = 0
FLAG_NONFINITE = 1
MAX_LAYERS = 4
MAX_HOP_BATCH = 8      # membrane positions that can share one strip-hop launch (paresis_refract_hop_batch)
MAX_GROUP = 4          # energies of a detector bin that can share one object hop (paresis_refract_group)
REFRACTION_MARGIN = 15   # refractionFileNumba2.py:50
REFRACTION_MARGIN_V1 = 10  # refractionFileNumba.py:36

EXPORTS = (
    "paresis_version", "paresis_last_error", "paresis_set_tuning", "paresis_trim", "paresis_splat", "paresis_refract_phi", "paresis_refract_layers",
    "paresis_transmit_rt", "paresis_transmit_wave", "paresis_mix_maps", "paresis_fresnel_plan_create", "paresis_fresnel_plan_destroy",
    "paresis_fresnel_plan_bytes", "paresis_fresnel_propagate", "paresis_fresnel_kernel_create", "paresis_fresnel_kernel_destroy",
    "paresis_fresnel_convolve", "paresis_fresnel_spectrum", "paresis_fresnel_from_spectrum", "paresis_fresnel_run", "paresis_fresnel_run_positions", "paresis_df_run", "paresis_detect_work_floats", "paresis_detect",
    "paresis_detect_counts", "paresis_detect_counts_multi",
    "paresis_poisson", "paresis_bin_sum", "paresis_raster_work_bytes", "paresis_raster_spheres", "paresis_sphere_map", "paresis_cylinder_map",
    "paresis_fill", "paresis_axpy", "paresis_mean", "paresis_sum_scaled", "paresis_rt_run", "paresis_rt_run_positions",
    "paresis_refract_layers_ex", "paresis_raster_field", "paresis_membrane_from_field",
    "paresis_two_sphere_phantom", "paresis_df_angle", "paresis_df_split", "paresis_df_scatter",
    "paresis_refract_group", "paresis_refract_tile_batch", "paresis_membrane_from_field_batch", "paresis_refract_hop_batch", "paresis_refract_hop_work_bytes", "paresis_transfer_lane_create", "paresis_transfer_lane_destroy", "paresis_transfer_d2h", "paresis_transfer_wait",
)


class ParesisError(RuntimeError):
    pass


class Layer(ctypes.Structure):
    _fields_ = [("thickness", ctypes.c_void_p), ("grad_obj", ctypes.c_float), ("grad_ref", ctypes.c_float),
                ("atten", ctypes.c_float)]


class RtEnergy(ctypes.Structure):
    _fields_ = [("intensity_membrane", ctypes.c_float), ("intensity_propag", ctypes.c_float),
                ("hop1", Layer * MAX_LAYERS), ("n_hop1", ctypes.c_int),
                ("hop2", Layer * MAX_LAYERS), ("n_hop2", ctypes.c_int),
                ("propag", Layer * MAX_LAYERS), ("n_propag", ctypes.c_int),
                ("close_bin", ctypes.c_int)]


class RtJob(ctypes.Structure):
    _fields_ = [("nx", ctypes.c_int), ("ny", ctypes.c_int), ("oversampling", ctypes.c_int), ("det_x", ctypes.c_int),
                ("det_y", ctypes.c_int), ("first_point", ctypes.c_int), ("n_energies", ctypes.c_int),
                ("energies_host", ctypes.POINTER(RtEnergy)),
                ("i_bs", ctypes.c_void_p), ("acc_sample", ctypes.c_void_p), ("acc_ref", ctypes.c_void_p),
                ("acc_propag", ctypes.c_void_p), ("acc_white", ctypes.c_void_p), ("means", ctypes.c_void_p),
                ("detect_work", ctypes.c_void_p), ("src_kernel", ctypes.c_void_p), ("src_half", ctypes.c_int),
                ("psf_kernel", ctypes.c_void_p), ("psf_half", ctypes.c_int), ("noise", ctypes.c_int),
                ("seed", ctypes.c_uint64), ("sequence", ctypes.c_uint64),
                ("out_sample", ctypes.c_void_p), ("out_ref", ctypes.c_void_p), ("out_propag", ctypes.c_void_p),
                ("out_white", ctypes.c_void_p), ("dx_pad", ctypes.c_void_p), ("dy_pad", ctypes.c_void_p),
                ("flag", ctypes.c_void_p), ("probe", ctypes.c_int), ("probe_start", ctypes.c_void_p),
                ("probe_end", ctypes.c_void_p), ("i_bs_dirty", ctypes.c_int), ("i_bs_group", ctypes.c_void_p * (MAX_GROUP - 1)),
                ("positions_per_launch", ctypes.c_int), ("throughput", ctypes.c_int)]


class DfEnergy(ctypes.Structure):
    _fields_ = [("scatter_map", ctypes.c_void_p), ("angle_coeff", ctypes.c_double), ("dark_field_weight", ctypes.c_double)]


class DfJob(ctypes.Structure):
    _fields_ = [("rt", RtJob), ("energies_df_host", ctypes.POINTER(DfEnergy)), ("angle", ctypes.c_void_p),
                ("plain", ctypes.c_void_p), ("scattered", ctypes.c_void_p), ("clean", ctypes.c_void_p), ("moved", ctypes.c_void_p),
                ("dark_field", ctypes.c_void_p)]


class GroupEnergy(ctypes.Structure):
    _fields_ = [("layers", Layer * MAX_LAYERS), ("n_layers", ctypes.c_int), ("intensity_in", ctypes.c_void_p),
                ("intensity_scale", ctypes.c_float), ("sum_ref", ctypes.c_void_p)]


class RtPosition(ctypes.Structure):
    _fields_ = [("offsets_host", ctypes.POINTER(ctypes.c_int64)), ("thickness", ctypes.c_void_p),
                ("out_sample", ctypes.c_void_p), ("out_ref", ctypes.c_void_p), ("out_propag", ctypes.c_void_p),
                ("out_white", ctypes.c_void_p), ("means", ctypes.c_void_p), ("sequence", ctypes.c_uint64),
                ("first_point", ctypes.c_int), ("probe_start", ctypes.c_void_p), ("probe_end", ctypes.c_void_p)]


class RtSlot(ctypes.Structure):
    _fields_ = [("i_bs", ctypes.c_void_p), ("acc_sample", ctypes.c_void_p), ("acc_ref", ctypes.c_void_p),
                ("acc_propag", ctypes.c_void_p), ("acc_white", ctypes.c_void_p), ("raster_work", ctypes.c_void_p),
                ("raster_work_bytes", ctypes.c_size_t), ("stream", ctypes.c_void_p), ("i_bs_dirty", ctypes.c_int),
                ("i_bs_group", ctypes.c_void_p * (MAX_GROUP - 1))]


class Membrane(ctypes.Structure):
    _fields_ = [("spheres", ctypes.c_void_p), ("n_spheres", ctypes.c_int), ("pix_um", ctypes.c_double),
                ("n_layers", ctypes.c_int), ("margin", ctypes.c_int), ("field", ctypes.c_void_p),
                ("field_x", ctypes.c_int), ("field_y", ctypes.c_int)]


class RefractExtras(ctypes.Structure):
    _fields_ = [("zero_fill", ctypes.c_void_p * 3), ("clear_input", ctypes.c_int), ("zero_scalar", ctypes.c_void_p),
                ("sum_ref", ctypes.c_void_p), ("intensity_scale", ctypes.c_float), ("mode", ctypes.c_int), ("reach", ctypes.c_int), ("throughput", ctypes.c_int)]


class HopItem(ctypes.Structure):
    _fields_ = [("intensity_in", ctypes.c_void_p), ("thickness", ctypes.c_void_p * MAX_LAYERS), ("out_obj", ctypes.c_void_p),
                ("out_ref", ctypes.c_void_p), ("sum_ref", ctypes.c_void_p)]


class C32(ctypes.Structure):
    _fields_ = [("re", ctypes.c_float), ("im", ctypes.c_float)]


class WaveLayer(ctypes.Structure):
    _fields_ = [("thickness", ctypes.c_void_p), ("atten", ctypes.c_double), ("phase", ctypes.c_double)]


class FresnelEnergy(ctypes.Structure):
    _fields_ = [("amplitude_membrane", ctypes.c_float), ("amplitude_propag", ctypes.c_float), ("white", ctypes.c_double),
                ("membrane_host", ctypes.POINTER(WaveLayer)), ("n_membrane", ctypes.c_int),
                ("sample", WaveLayer * MAX_LAYERS), ("n_sample", ctypes.c_int),
                ("reference", ctypes.c_void_p), ("phase_reference", C32),
                ("to_object", ctypes.c_void_p), ("phase_to_object", C32),
                ("to_detector", ctypes.c_void_p), ("phase_to_detector", C32),
                ("close_bin", ctypes.c_int)]


class FresnelJob(ctypes.Structure):
    _fields_ = [("plan", ctypes.c_void_p), ("oversampling", ctypes.c_int), ("det_x", ctypes.c_int), ("det_y", ctypes.c_int),
                ("first_point", ctypes.c_int), ("n_energies", ctypes.c_int), ("energies_host", ctypes.POINTER(FresnelEnergy)),
                ("wave_a", ctypes.c_void_p), ("wave_b", ctypes.c_void_p),
                ("acc_sample", ctypes.c_void_p), ("acc_ref", ctypes.c_void_p), ("acc_propag", ctypes.c_void_p),
                ("acc_white", ctypes.c_void_p), ("means", ctypes.c_void_p), ("detect_work", ctypes.c_void_p),
                ("src_kernel", ctypes.c_void_p), ("src_half", ctypes.c_int), ("psf_kernel", ctypes.c_void_p), ("psf_half", ctypes.c_int),
                ("noise", ctypes.c_int), ("seed", ctypes.c_uint64), ("sequence", ctypes.c_uint64),
                ("out_sample", ctypes.c_void_p), ("out_ref", ctypes.c_void_p), ("out_propag", ctypes.c_void_p),
                ("out_white", ctypes.c_void_p)]


class FresnelSlot(ctypes.Structure):
    _fields_ = [("plan", ctypes.c_void_p), ("wave_a", ctypes.c_void_p), ("wave_b", ctypes.c_void_p),
                ("acc_sample", ctypes.c_void_p), ("acc_ref", ctypes.c_void_p), ("acc_propag", ctypes.c_void_p),
                ("acc_white", ctypes.c_void_p), ("detect_work", ctypes.c_void_p), ("raster_work", ctypes.c_void_p),
                ("raster_work_bytes", ctypes.c_size_t), ("stream", ctypes.c_void_p)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "paresis_b200: %s not found. Build it with `python -m paresis_b200.build` "
            "(nvcc, sm_100a). There is no CPU or PyTorch fallback for this path." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
    missing = [n for n in EXPORTS if not hasattr(lib, n)]
    if missing:
        raise ImportError("paresis_b200: %s lacks symbols %s" % (LIB_PATH, missing))
    vp, ci, cd, cf, sz, u64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_float, ctypes.c_size_t, ctypes.c_uint64
    lib.paresis_version.restype = ci
    lib.paresis_last_error.restype = ctypes.c_char_p
    sig = {
        "paresis_set_tuning": [ci, ci],
        "paresis_splat": [vp, vp, vp, vp, ci, ci, ci, ci, vp, vp],
        "paresis_refract_phi": [vp, vp, vp, vp, vp, ci, ci, ci, cd, cd, cd, cd, cd, vp, vp],
        "paresis_refract_layers": [vp, cf, ctypes.POINTER(Layer), ci, vp, vp, vp, vp, ci, ci, ci, vp, vp],
        "paresis_transmit_rt": [vp, vp, ctypes.POINTER(vp), ctypes.POINTER(cd), ctypes.POINTER(cd), ci, vp, vp, sz, vp],
        "paresis_transmit_wave": [vp, cf, ctypes.POINTER(vp), ctypes.POINTER(cd), ctypes.POINTER(cd), ci, vp, sz, vp],
        "paresis_mix_maps": [ctypes.POINTER(vp), ci, ctypes.POINTER(cd), ctypes.POINTER(cd), ci, ctypes.POINTER(vp), sz, vp],
        "paresis_fresnel_plan_create": [ci, ci, ci, ctypes.POINTER(vp)],
        "paresis_fresnel_plan_destroy": [vp],
        "paresis_fresnel_propagate": [vp, vp, vp, vp, C32, vp, vp, vp],
        "paresis_fresnel_kernel_create": [vp, vp, vp, vp, ctypes.POINTER(vp)],
        "paresis_fresnel_kernel_destroy": [vp],
        "paresis_fresnel_convolve": [vp, vp, vp, C32, vp, vp, vp],
        "paresis_fresnel_spectrum": [vp, vp, vp],
        "paresis_fresnel_from_spectrum": [vp, vp, vp, C32, vp, vp, vp],
        "paresis_fresnel_run": [ctypes.POINTER(FresnelJob), vp],
        "paresis_fresnel_run_positions": [ctypes.POINTER(FresnelJob), ctypes.POINTER(Membrane), ctypes.POINTER(RtPosition), ci,
                                          ctypes.POINTER(FresnelSlot), ci, vp],
        "paresis_detect": [vp, ci, ci, ci, ci, ci, vp, ci, vp, ci, vp, vp, vp],
        "paresis_detect_counts": [vp, ci, ci, ci, ci, ci, vp, ci, vp, ci, vp, vp, ci, u64, u64, vp],
        "paresis_detect_counts_multi": [ctypes.POINTER(vp), ctypes.POINTER(vp), ctypes.POINTER(u64), ci, ci, ci, ci, ci, ci, vp, ci,
                                        vp, ci, vp, ci, u64, vp],
        "paresis_poisson": [vp, vp, sz, u64, u64, vp],
        "paresis_bin_sum": [vp, ci, ci, ci, ci, vp, vp],
        "paresis_raster_spheres": [vp, ci, cd, ctypes.POINTER(ctypes.c_int64), ci, ci, ci, ci, vp, vp, sz, vp],
        "paresis_raster_field": [vp, ci, cd, ci, ci, vp, vp, sz, vp],
        "paresis_membrane_from_field": [vp, ci, ci, ctypes.POINTER(ctypes.c_int64), ci, ci, ci, ci, vp, vp],
        "paresis_sphere_map": [cd, ci, ci, cd, vp, vp],
        "paresis_cylinder_map": [cd, cd, ci, ci, cd, vp, vp],
        "paresis_fill": [vp, cf, sz, vp],
        "paresis_axpy": [vp, vp, cf, sz, vp],
        "paresis_mean": [vp, sz, vp, vp],
        "paresis_sum_scaled": [vp, sz, cd, vp, vp],
        "paresis_rt_run": [ctypes.POINTER(RtJob), vp],
        "paresis_df_run": [ctypes.POINTER(DfJob), vp],
        "paresis_two_sphere_phantom": [ci, ci, ci, cd, vp, vp],
        "paresis_df_angle": [vp, cd, vp, sz, vp],
        "paresis_df_split": [vp, cf, vp, cf, vp, vp, vp, sz, vp],
        "paresis_df_scatter": [vp, vp, vp, ci, ci, vp],
        "paresis_refract_group": [ctypes.POINTER(GroupEnergy), ci, vp, vp, ci, ci, vp, vp],
        "paresis_refract_hop_batch": [ctypes.POINTER(HopItem), ci, ctypes.POINTER(Layer), ci, cf, cf, ci, ci, ci, ci, vp, sz, vp, vp],
        "paresis_transfer_lane_create": [ctypes.POINTER(vp)],
        "paresis_transfer_lane_destroy": [vp],
        "paresis_transfer_d2h": [vp, vp, vp, sz, vp],
        "paresis_transfer_wait": [vp],
        "paresis_rt_run_positions": [ctypes.POINTER(RtJob), ctypes.POINTER(Membrane), ctypes.POINTER(RtPosition), ci,
                                     ctypes.POINTER(RtSlot), ci, vp],
        "paresis_refract_layers_ex": [vp, cf, ctypes.POINTER(Layer), ci, vp, vp, vp, vp, ci, ci, ci, vp,
                                      ctypes.POINTER(RefractExtras), vp],
    }
    for name, argtypes in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = ci
    lib.paresis_detect_work_floats.argtypes = [ci, ci, ci, ci, ci]
    lib.paresis_detect_work_floats.restype = sz
    lib.paresis_fresnel_plan_bytes.argtypes = [vp]
    lib.paresis_fresnel_plan_bytes.restype = sz
    lib.paresis_refract_hop_work_bytes.argtypes = [ci, ci, ci, ci, ci, ci, ci]
    lib.paresis_refract_hop_work_bytes.restype = sz
    lib.paresis_raster_work_bytes.argtypes = [ci, ci, ci, ci]
    lib.paresis_raster_work_bytes.restype = sz
    return lib


lib = _load()

# Every call below is one (or a few) of OUR kernels; the bench reports this counter.
launches = 0


def _check(rc, what):
    if rc != OK:
        raise ParesisError("%s failed (%d): %s" % (what, rc, lib.paresis_last_error().decode()))


_stream_override = None


def _stream():
    if _stream_override is not None:
        return _stream_override
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


class on_stream:
    """Resolve torch's current stream once for a batch of library calls (the lookup costs ~20 us)."""

    def __enter__(self):
        global _stream_override
        self.prev = _stream_override
        _stream_override = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def __exit__(self, *exc):
        global _stream_override
        _stream_override = self.prev


# probe kinds of paresis_rt_run
PROBE = {"refract_membrane_hop": 1, "refract_sample_ref_hop": 2, "detect": 3, "raster_spheres": 4}


def rt_run(job, launches_in_job, probe=None):
    """paresis_rt_run; `probe` = (kind label, start Event, end Event) records one kernel of the call."""
    if probe is not None:
        label, e0, e1 = probe
        for e in (e0, e1):
            if not e.cuda_event:
                e.record()          # materialise the underlying cudaEvent_t
        job.probe, job.probe_start, job.probe_end = PROBE[label], e0.cuda_event, e1.cuda_event
    else:
        job.probe = 0
    _check(lib.paresis_rt_run(ctypes.byref(job), _stream()), "paresis_rt_run")
    _count(launches_in_job)


def fresnel_run(job, launches_in_job):
    """paresis_fresnel_run: one membrane position of the Fresnel model (a FresnelJob)."""
    _check(lib.paresis_fresnel_run(ctypes.byref(job), _stream()), "paresis_fresnel_run")
    _count(launches_in_job)


def fresnel_run_positions(job, membrane, positions, slots, launches_in_job):
    """paresis_fresnel_run_positions: `positions` / `slots` are ctypes arrays of RtPosition / FresnelSlot."""
    _check(lib.paresis_fresnel_run_positions(ctypes.byref(job), ctypes.byref(membrane), positions, len(positions), slots,
                                             len(slots), _stream()), "paresis_fresnel_run_positions")
    _count(launches_in_job)


def df_run(job, launches_in_job):
    """paresis_df_run: one membrane position of the ray-tracing model with a scattering sample (a DfJob)."""
    _check(lib.paresis_df_run(ctypes.byref(job), _stream()), "paresis_df_run")
    _count(launches_in_job)


def rt_run_positions(job, membrane, positions, slots, launches_in_job, probe_label=None):
    """paresis_rt_run_positions: `positions` / `slots` are ctypes arrays of RtPosition / RtSlot."""
    job.probe = PROBE[probe_label] if probe_label in PROBE else 0
    _check(lib.paresis_rt_run_positions(ctypes.byref(job), ctypes.byref(membrane), positions, len(positions), slots,
                                        len(slots), _stream()), "paresis_rt_run_positions")
    _count(launches_in_job)


def _ptr(t, dtype=None):
    if t is None:
        return None
    if not t.is_cuda or not t.is_contiguous():
        raise ParesisError("expected a contiguous CUDA tensor")
    if dtype is not None and t.dtype != dtype:
        raise ParesisError("expected dtype %s, got %s" % (dtype, t.dtype))
    return ctypes.c_void_p(t.data_ptr())


def _count(n=1):
    global launches
    launches += n


# Optional CUDA-event timing of library calls (used by bench.py): None = off, "*" = every call
# (events stored as (label, start, end)), or one label (stored as (start, end)).
profile_only = None
profile_events = []


def _timed(label, call):
    if profile_only is None or (profile_only != "*" and profile_only != label):
        return call()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    rc = call()
    e1.record()
    profile_events.append((label, e0, e1) if profile_only == "*" else (e0, e1))
    return rc


def set_tuning(key, value):
    _check(lib.paresis_set_tuning(int(key), int(value)), "paresis_set_tuning")


if os.environ.get("PARESIS_TILE_CONFIG"):     # development knob: -1 = direct-to-L2 hop kernel, 0 / 1 = tile shapes
    set_tuning(2, int(os.environ["PARESIS_TILE_CONFIG"]))


if os.environ.get("PARESIS_LEAN_ROWS"):        # development knob: source rows per block of the tile hops (0 = automatic)
    set_tuning(3, int(os.environ["PARESIS_LEAN_ROWS"]))
if os.environ.get("PARESIS_ROWS"):            # development knob: source rows per warp of the hop kernels
    set_tuning(1, int(os.environ["PARESIS_ROWS"]))


def splat(intensity, dx, dy, out, margin=0, variant=2, flag=None):
    nx, ny = intensity.shape
    _check(lib.paresis_splat(_ptr(intensity, torch.float32), _ptr(dx, torch.float32), _ptr(dy, torch.float32),
                             _ptr(out, torch.float32), nx, ny, margin, variant, _ptr(flag, torch.int32), _stream()),
           "paresis_splat")
    _count()


def refract_phi(intensity, phi, out, distance, energy_kev, magnification, pixel_um, margin=REFRACTION_MARGIN,
                dx_pad=None, dy_pad=None, flag=None, clamp_px=0.0):
    nx, ny = intensity.shape
    _check(lib.paresis_refract_phi(_ptr(intensity, torch.float32), _ptr(phi, torch.float64), _ptr(out, torch.float32),
                                   _ptr(dx_pad, torch.float32), _ptr(dy_pad, torch.float32), nx, ny, margin,
                                   float(distance), float(energy_kev), float(magnification), float(pixel_um),
                                   float(clamp_px), _ptr(flag, torch.int32), _stream()), "paresis_refract_phi")
    _count()


def refract_layers(intensity_in, intensity_uniform, layers, out_obj, out_ref=None, margin=REFRACTION_MARGIN, flag=None,
                   dx_pad=None, dy_pad=None, zero_fill=(), clear_input=False, zero_scalar=None, sum_ref=None,
                   intensity_scale=0.0, mode=0, reach=0):
    """layers: list of (thickness tensor, grad_obj, grad_ref, atten); the keyword extras are
    paresis_refract_extras (zero_fill: up to 3 float32 images; zero_scalar / sum_ref: float64 scalars;
    mode 0: out += through the round-1 kernels, 1: out = / 2: out += through the owner-computes strip kernels)."""
    n = len(layers)
    arr = (Layer * n)()
    for k, (t, go, gr, at) in enumerate(layers):
        arr[k].thickness = t.data_ptr()
        arr[k].grad_obj, arr[k].grad_ref, arr[k].atten = float(go), float(gr), float(at)
        _ptr(t, torch.float32)
    nx, ny = out_obj.shape
    label = "refract_sample_ref_hop" if out_ref is not None else "refract_membrane_hop"
    extras = RefractExtras()
    for k, z in enumerate(zero_fill):
        extras.zero_fill[k] = z.data_ptr()
        _ptr(z, torch.float32)
    extras.clear_input = 1 if clear_input else 0
    extras.zero_scalar = zero_scalar.data_ptr() if zero_scalar is not None else None
    extras.sum_ref = sum_ref.data_ptr() if sum_ref is not None else None
    extras.intensity_scale = float(intensity_scale)
    extras.mode, extras.reach = int(mode), int(reach)
    _check(_timed(label, lambda: lib.paresis_refract_layers_ex(
        _ptr(intensity_in, torch.float32), float(intensity_uniform), arr, n, _ptr(out_obj, torch.float32),
        _ptr(out_ref, torch.float32), _ptr(dx_pad, torch.float32), _ptr(dy_pad, torch.float32), nx, ny, margin,
        _ptr(flag, torch.int32), ctypes.byref(extras), _stream())), "paresis_refract_layers_ex")
    _count()


def refract_hop_batch(items, coeffs, intensity_uniform, intensity_scale, accumulate=False, reach=12, work=None, flag=None):
    """paresis_refract_hop_batch.  items: list of dicts {intensity_in (tensor | None), thickness (list of tensors),
    out_obj, out_ref (tensor | None), sum_ref (float64 tensor | None)}; coeffs: list of (grad_obj, grad_ref, atten)."""
    n = len(items)
    arr = (HopItem * n)()

    def addr(t, dtype):
        _ptr(t, dtype)
        return t.data_ptr() if t is not None else None

    for k, it in enumerate(items):
        arr[k].intensity_in = addr(it.get("intensity_in"), torch.float32)
        for m, t in enumerate(it["thickness"]):
            arr[k].thickness[m] = addr(t, torch.float32)
        arr[k].out_obj = addr(it["out_obj"], torch.float32)
        arr[k].out_ref = addr(it.get("out_ref"), torch.float32)
        arr[k].sum_ref = addr(it.get("sum_ref"), torch.float64)
    lay = (Layer * len(coeffs))()
    for m, (go, gr, at) in enumerate(coeffs):
        lay[m].grad_obj, lay[m].grad_ref, lay[m].atten = float(go), float(gr), float(at)
    nx, ny = items[0]["out_obj"].shape
    _check(lib.paresis_refract_hop_batch(arr, n, lay, len(coeffs), float(intensity_uniform), float(intensity_scale),
                                         1 if accumulate else 0, int(reach), nx, ny, _ptr(work), work.numel() * work.element_size() if work is not None else 0,
                                         _ptr(flag, torch.int32), _stream()), "paresis_refract_hop_batch")
    _count(2)


def refract_group(energies, out_obj, out_ref, flag=None):
    """paresis_refract_group.  energies: list of (intensity image, intensity scale, layers, sum_ref tensor or None)
    with layers = [(thickness, grad_obj, grad_ref, atten), ...] on the same thickness maps."""
    n = len(energies)
    arr = (GroupEnergy * n)()
    for g, (inten, scale, layers, sum_ref) in enumerate(energies):
        for m, (t, go, gr, at) in enumerate(layers):
            arr[g].layers[m].thickness = t.data_ptr()
            arr[g].layers[m].grad_obj, arr[g].layers[m].grad_ref, arr[g].layers[m].atten = float(go), float(gr), float(at)
            _ptr(t, torch.float32)
        arr[g].n_layers = len(layers)
        arr[g].intensity_in = _ptr(inten, torch.float32)
        arr[g].intensity_scale = float(scale)
        arr[g].sum_ref = sum_ref.data_ptr() if sum_ref is not None else None
    nx, ny = out_obj.shape
    _check(_timed("refract_sample_ref_hop", lambda: lib.paresis_refract_group(
        arr, n, _ptr(out_obj, torch.float32), _ptr(out_ref, torch.float32), nx, ny, _ptr(flag, torch.int32), _stream())),
        "paresis_refract_group")
    _count()


def _layer_arrays(thickness, atten, phase):
    n = len(thickness)
    tp = (ctypes.c_void_p * max(n, 1))(*[t.data_ptr() for t in thickness])
    for t in thickness:
        _ptr(t, torch.float32)
    at = (ctypes.c_double * max(n, 1))(*[float(a) for a in atten])
    ph = (ctypes.c_double * max(n, 1))(*[float(p) for p in phase])
    return n, tp, at, ph


def _groups(n):
    """Transmission is multiplicative: more than MAX_LAYERS materials are applied MAX_LAYERS at a time, each call after the
    first working in place on the outputs of the one before (Sample.py:279, :347-348 loop over any number of materials)."""
    return [slice(g, g + MAX_LAYERS) for g in range(0, max(n, 1), MAX_LAYERS)]


def transmit_rt(intensity_in, phi_in, thickness, atten, phase, intensity_out, phi_out):
    count = (intensity_out if intensity_out is not None else phi_out).numel()
    for k, sl in enumerate(_groups(len(thickness))):
        n, tp, at, ph = _layer_arrays(thickness[sl], atten[sl], phase[sl])
        i_in, p_in = (intensity_in, phi_in) if k == 0 else (intensity_out, phi_out)
        _check(lib.paresis_transmit_rt(_ptr(i_in, torch.float32), _ptr(p_in, torch.float64), tp, at, ph, n,
                                       _ptr(intensity_out, torch.float32), _ptr(phi_out, torch.float64), count, _stream()),
               "paresis_transmit_rt")
        _count()


def transmit_wave(wave_in, amplitude_uniform, thickness, atten, phase, wave_out):
    for k, sl in enumerate(_groups(len(thickness))):
        n, tp, at, ph = _layer_arrays(thickness[sl], atten[sl], phase[sl])
        w_in = wave_in if k == 0 else wave_out
        _check(lib.paresis_transmit_wave(_ptr(w_in, torch.complex64), float(amplitude_uniform), tp, at, ph, n,
                                         _ptr(wave_out, torch.complex64), wave_out.numel(), _stream()),
               "paresis_transmit_wave")
        _count()


def mix_maps(maps, weights, bias, outs):
    """paresis_mix_maps: outs[k] = bias[k] + sum_m weights[k][m] * maps[m] (fp64 accumulation, one fp32 rounding).
    ``weights``: n_out rows of len(maps) values; ``bias``: n_out values or None (0)."""
    n_out, n_maps = len(outs), len(maps)
    for t in list(maps) + list(outs):
        _ptr(t, torch.float32)
    mp = (ctypes.c_void_p * max(n_maps, 1))(*[t.data_ptr() for t in maps])
    op = (ctypes.c_void_p * max(n_out, 1))(*[t.data_ptr() for t in outs])
    w = (ctypes.c_double * max(n_out * n_maps, 1))(*[float(v) for row in weights for v in row])
    b = (ctypes.c_double * n_out)(*[float(v) for v in bias]) if bias is not None else None
    count = outs[0].numel() if outs else 0
    if any(t.numel() != count for t in list(maps) + list(outs)):
        raise ParesisError("paresis_mix_maps: every map and output must have %d pixels" % count)
    _check(lib.paresis_mix_maps(mp, n_maps, w, b, n_out, op, count, _stream()), "paresis_mix_maps")
    _count()


class FresnelPlan:
    def __init__(self, nx, ny, margin=15):
        h = ctypes.c_void_p()
        _check(lib.paresis_fresnel_plan_create(nx, ny, margin, ctypes.byref(h)), "paresis_fresnel_plan_create")
        self._h = h
        self.nx, self.ny, self.margin = nx, ny, margin

    def bytes(self):
        return lib.paresis_fresnel_plan_bytes(self._h)

    def propagate(self, wave_in, hx, hy, phase=1.0 + 0.0j, wave_out=None, intensity_acc=None):
        ph = C32(float(np.real(phase)), float(np.imag(phase)))
        _check(lib.paresis_fresnel_propagate(self._h, _ptr(wave_in, torch.complex64), _ptr(hx, torch.complex64),
                                             _ptr(hy, torch.complex64), ph, _ptr(wave_out, torch.complex64),
                                             _ptr(intensity_acc, torch.float32), _stream()),
               "paresis_fresnel_propagate")
        _count(16)

    def kernel(self, hx, hy):
        """The convolution kernels of one transfer function (both axes), for convolve()."""
        return FresnelKernel(self, hx, hy)

    def convolve(self, wave_in, kernel, phase=1.0 + 0.0j, wave_out=None, intensity_acc=None):
        ph = C32(float(np.real(phase)), float(np.imag(phase)))
        _check(lib.paresis_fresnel_convolve(self._h, _ptr(wave_in, torch.complex64), kernel._h, ph, _ptr(wave_out, torch.complex64),
                                            _ptr(intensity_acc, torch.float32), _stream()), "paresis_fresnel_convolve")
        _count(6)

    def spectrum(self, wave_in):
        """fft2(pad(wave_in)) kept inside the plan for from_spectrum()."""
        _check(lib.paresis_fresnel_spectrum(self._h, _ptr(wave_in, torch.complex64), _stream()), "paresis_fresnel_spectrum")
        _count(2)

    def from_spectrum(self, hx, hy, phase=1.0 + 0.0j, wave_out=None, intensity_acc=None):
        ph = C32(float(np.real(phase)), float(np.imag(phase)))
        _check(lib.paresis_fresnel_from_spectrum(self._h, _ptr(hx, torch.complex64), _ptr(hy, torch.complex64), ph,
                                                 _ptr(wave_out, torch.complex64), _ptr(intensity_acc, torch.float32), _stream()),
               "paresis_fresnel_from_spectrum")
        _count(3)

    def close(self):
        if self._h:
            lib.paresis_fresnel_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class FresnelKernel:
    def __init__(self, plan, hx, hy):
        h = ctypes.c_void_p()
        _check(lib.paresis_fresnel_kernel_create(plan._h, _ptr(hx, torch.complex64), _ptr(hy, torch.complex64), _stream(),
                                                 ctypes.byref(h)), "paresis_fresnel_kernel_create")
        self._h = h
        _count(10)

    def close(self):
        if self._h:
            lib.paresis_fresnel_kernel_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def detect_work_floats(nx, ny, oversampling, det_x, det_y):
    return lib.paresis_detect_work_floats(nx, ny, oversampling, det_x, det_y)


def detect(image, oversampling, det_x, det_y, src_kernel, psf_kernel, work, expect_out):
    nx, ny = image.shape
    sh = 0 if src_kernel is None else (src_kernel.numel() - 1) // 2
    ph = 0 if psf_kernel is None else (psf_kernel.numel() - 1) // 2
    _check(_timed("detect", lambda: lib.paresis_detect(
        _ptr(image, torch.float32), nx, ny, oversampling, det_x, det_y, _ptr(src_kernel, torch.float32), sh,
        _ptr(psf_kernel, torch.float32), ph, _ptr(work, torch.float32), _ptr(expect_out, torch.float32), _stream())),
        "paresis_detect")
    _count(4 if ph else 3)


def detect_counts(image, oversampling, det_x, det_y, src_kernel, psf_kernel, work, out, noise, seed=0, sequence=0):
    nx, ny = image.shape
    sh = 0 if src_kernel is None else (src_kernel.numel() - 1) // 2
    ph = 0 if psf_kernel is None else (psf_kernel.numel() - 1) // 2
    _check(_timed("detect", lambda: lib.paresis_detect_counts(
        _ptr(image, torch.float32), nx, ny, oversampling, det_x, det_y, _ptr(src_kernel, torch.float32), sh,
        _ptr(psf_kernel, torch.float32), ph, _ptr(work, torch.float32), _ptr(out, torch.float32), 1 if noise else 0,
        int(seed) & (2 ** 64 - 1), int(sequence) & (2 ** 64 - 1), _stream())), "paresis_detect_counts")
    _count()


def detect_counts_multi(images, oversampling, det_x, det_y, src_kernel, psf_kernel, work, outs, noise, seed, sequences):
    """Up to 8 images of one detector in a single launch (paresis_detect_counts_multi); one output and one Poisson
    sequence per image."""
    n = len(images)
    if len(outs) != n or len(sequences) != n:
        raise ValueError("detect_counts_multi: %d images, %d outputs and %d sequences" % (n, len(outs), len(sequences)))
    nx, ny = images[0].shape
    sh = 0 if src_kernel is None else (src_kernel.numel() - 1) // 2
    ph = 0 if psf_kernel is None else (psf_kernel.numel() - 1) // 2
    ip = (ctypes.c_void_p * n)(*[_ptr(t, torch.float32) for t in images])
    op = (ctypes.c_void_p * n)(*[_ptr(t, torch.float32) for t in outs])
    sq = (ctypes.c_uint64 * n)(*[int(q) & (2 ** 64 - 1) for q in sequences])
    _check(_timed("detect", lambda: lib.paresis_detect_counts_multi(
        ip, op, sq, n, nx, ny, oversampling, det_x, det_y, _ptr(src_kernel, torch.float32), sh,
        _ptr(psf_kernel, torch.float32), ph, _ptr(work, torch.float32), 1 if noise else 0, int(seed) & (2 ** 64 - 1),
        _stream())), "paresis_detect_counts_multi")
    _count()


def poisson(expect, counts, seed, sequence):
    _check(_timed("poisson", lambda: lib.paresis_poisson(
        _ptr(expect, torch.float32), _ptr(counts, torch.float32), expect.numel(), int(seed) & (2 ** 64 - 1),
        int(sequence) & (2 ** 64 - 1), _stream())), "paresis_poisson")
    _count()


def bin_sum(image, size_x, size_y, out):
    nx, ny = image.shape
    _check(lib.paresis_bin_sum(_ptr(image, torch.float32), nx, ny, size_x, size_y, _ptr(out, torch.float32), _stream()),
           "paresis_bin_sum")
    _count()


_raster_work = {}


def raster_spheres(spheres, pix_um, offsets, dim_x, dim_y, margin, out):
    offs = np.ascontiguousarray(np.asarray(offsets, dtype=np.int64).reshape(-1, 2))
    need = lib.paresis_raster_work_bytes(spheres.shape[0], offs.shape[0], dim_x, dim_y)
    key = out.device.index
    work = _raster_work.get(key)
    if work is None or work.numel() < need:
        work = _raster_work[key] = torch.empty(need, device=out.device, dtype=torch.uint8)
    _check(_timed("raster_spheres", lambda: lib.paresis_raster_spheres(
        _ptr(spheres, torch.float64), spheres.shape[0], float(pix_um), offs.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)),
        offs.shape[0], dim_x, dim_y, margin, _ptr(out, torch.float32), ctypes.c_void_p(work.data_ptr()), work.numel(),
        _stream())), "paresis_raster_spheres")
    _count(2)


def raster_field(spheres, pix_um, field):
    """paresis_raster_field: the caps of the whole sphere list on its own canvas (once per experiment)."""
    fx, fy = field.shape
    need = lib.paresis_raster_work_bytes(spheres.shape[0], 1, fx, fy)
    work = torch.empty(need, device=field.device, dtype=torch.uint8)
    _check(lib.paresis_raster_field(_ptr(spheres, torch.float64), spheres.shape[0], float(pix_um), fx, fy,
                                    _ptr(field, torch.float32), ctypes.c_void_p(work.data_ptr()), work.numel(), _stream()),
           "paresis_raster_field")
    _count(2)
    torch.cuda.current_stream().synchronize()      # `work` is released when this returns


def membrane_from_field(field, offsets, margin, dim_x, dim_y, out):
    offs = np.ascontiguousarray(np.asarray(offsets, dtype=np.int64).reshape(-1, 2))
    fx, fy = field.shape
    _check(_timed("raster_spheres", lambda: lib.paresis_membrane_from_field(
        _ptr(field, torch.float32), fx, fy, offs.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), offs.shape[0], margin,
        dim_x, dim_y, _ptr(out, torch.float32), _stream())), "paresis_membrane_from_field")
    _count()


def two_sphere_phantom(kind, dim_x, dim_y, pix_um, out3):
    _check(lib.paresis_two_sphere_phantom(int(kind), dim_x, dim_y, float(pix_um), _ptr(out3, torch.float32), _stream()),
           "paresis_two_sphere_phantom")
    _count()


def df_angle(thickness, coeff, df_px):
    _check(lib.paresis_df_angle(_ptr(thickness, torch.float32), float(coeff), _ptr(df_px, torch.float32), thickness.numel(),
                                _stream()), "paresis_df_angle")
    _count()


def df_split(intensity, intensity_uniform, df_px, limit_px, i_plain, i_df, df_clean):
    _check(lib.paresis_df_split(_ptr(intensity, torch.float32), float(intensity_uniform), _ptr(df_px, torch.float32),
                                float(limit_px), _ptr(i_plain, torch.float32), _ptr(i_df, torch.float32),
                                _ptr(df_clean, torch.float32), df_px.numel(), _stream()), "paresis_df_split")
    _count()


def df_scatter(scattered, df_px, out):
    nx, ny = out.shape
    _check(lib.paresis_df_scatter(_ptr(scattered, torch.float32), _ptr(df_px, torch.float32), _ptr(out, torch.float32), nx, ny,
                                  _stream()), "paresis_df_scatter")
    _count()


def sphere_map(radius_um, dim_x, dim_y, pix_um, out):
    _check(lib.paresis_sphere_map(float(radius_um), dim_x, dim_y, float(pix_um), _ptr(out, torch.float32), _stream()),
           "paresis_sphere_map")
    _count()


def cylinder_map(radius_um, angle_deg, dim_x, dim_y, pix_um, out):
    _check(lib.paresis_cylinder_map(float(radius_um), float(angle_deg), dim_x, dim_y, float(pix_um),
                                    _ptr(out, torch.float32), _stream()), "paresis_cylinder_map")
    _count()


def fill(dst, value):
    _check(lib.paresis_fill(_ptr(dst, torch.float32), float(value), dst.numel(), _stream()), "paresis_fill")
    _count()


def axpy(dst, src, scale=1.0):
    _check(lib.paresis_axpy(_ptr(dst, torch.float32), _ptr(src, torch.float32), float(scale), dst.numel(), _stream()),
           "paresis_axpy")
    _count()


def mean(src, out):
    _check(lib.paresis_mean(_ptr(src, torch.float32), src.numel(), _ptr(out, torch.float64), _stream()), "paresis_mean")
    _count()
