"""Dark-field branch of the ray-tracing model on the GPU: the stand-alone pieces.

Reference: ``fastRefractionDF`` (refractionFileNumba2.py:88-196) and the Lung / 'cylinder_beeds' scattering
model of ``AnalyticalSample.setWaveRT`` (Sample.py:322-343).

The refraction part is the ordinary fused hop run twice -- on the rays with and without a scattering angle
(refractionFileNumba2.py:143-155) -- followed by the variable-width Gaussian scatter of the refracted
dark-field intensity (``paresis_df_scatter``; a Python double loop upstream).  A whole membrane position of a
scattering sample is one library call (``paresis_df_run``, reached through ``engine.ImageFormation.compute_rt``);
``model_of`` tells the scene which materials scatter.
"""
import numpy as np
import torch

from . import _cabi as abi
from . import hostmath as hm
from .host_api import device, to_dev, to_host, InsaneValues


def model_of(sample, imat):
    """Which scattering model applies to material ``imat`` of ``sample`` (Sample.py:322-343), or None."""
    if sample.myType != "sample_of_interest":
        return None
    model = "Lung" if sample.myMaterials[imat] == "Lung" else None
    if sample.myName == 'cylinder_beeds':
        model = "cylinder_beeds"          # upstream tests the name after the material: it wins
    return model


# ------------------------------------------------------------------ numpy-in / numpy-out pieces
def set_wave_rt(sample, geom, intensity, energy, phi, delta, beta):
    """AnalyticalSample.setWaveRT for a scattering sample: (I, phi, newDf) as host arrays."""
    k = hm.wavenumber(energy * 1000)
    shape = geom.map_shape
    maps = geom.device_entries(materialise=True)
    new_df, att, phase = 0, [], []
    for imat in range(len(maps)):
        model = model_of(sample, imat)
        fraction = 1.0
        if model is not None:
            coeff, fraction = hm.angle_coefficient(delta[imat], hm.MODELS[model]), hm.MODELS[model][1]
            df = torch.empty(shape, device=device(), dtype=torch.float32)
            abi.df_angle(maps[imat], coeff, df)
            new_df = to_host(df)
        att.append(2 * k * beta[imat] * fraction)          # the thickness is scaled by the volume fraction (:333, :344)
        phase.append(k * delta[imat] * fraction)
    i_in = to_dev(np.broadcast_to(np.asarray(intensity, dtype=np.float64), shape))
    phi_in = None
    if not (np.isscalar(phi) and phi == 0):
        phi_in = to_dev(np.broadcast_to(np.asarray(phi, dtype=np.float64), shape), torch.float64)
    i_out = torch.empty(shape, device=device(), dtype=torch.float32)
    phi_out = torch.empty(shape, device=device(), dtype=torch.float64)
    abi.transmit_rt(i_in, phi_in, maps, att, phase, i_out, phi_out)
    return to_host(i_out), to_host(phi_out), new_df


def fast_refraction_df(intensity, phi, distance, energy_kev, magnification, pixel_um, dark_field):
    """fastRefractionDF (refractionFileNumba2.py:88-196): (I3[N,N], Dx, Dy) as float64 host arrays, the
    displacement maps zero-padded by margin2 = ceil(6 max(DF))."""
    intensity = np.asarray(intensity, dtype=np.float64)
    nx, ny = intensity.shape
    df_px = np.asarray(dark_field, dtype=np.float64) * distance / (pixel_um * 1e-6 * magnification)     # :114
    margin2 = int(np.ceil(df_px.max() * 6))                                                             # :115-117
    dev = device()
    f32 = dict(device=dev, dtype=torch.float32)
    d_df = to_dev(df_px)
    plain, scat, clean = (torch.empty((nx, ny), **f32) for _ in range(3))
    abi.df_split(to_dev(intensity), 0.0, d_df, nx / 4, plain, scat, clean)
    d_phi = to_dev(phi, torch.float64)
    out, moved = torch.zeros((nx, ny), **f32), torch.zeros((nx, ny), **f32)
    dxp = torch.zeros((nx + 2 * margin2, ny + 2 * margin2), **f32)
    dyp = torch.zeros_like(dxp)
    flag = torch.zeros(1, device=dev, dtype=torch.int32)
    abi.refract_phi(plain, d_phi, out, distance, energy_kev, magnification, pixel_um, margin2, dxp, dyp, flag)
    abi.refract_phi(scat, d_phi, moved, distance, energy_kev, magnification, pixel_um, margin2, None, None, flag)
    abi.df_scatter(moved, clean, out)
    res = to_host(out)
    if int(flag.item()) & abi.FLAG_NONFINITE or not np.isfinite(res).all():
        raise InsaneValues("The calculated intensity refractive includes some nans or insane values")
    # Dx, Dy of every ray (the first call only saw the rays without a scattering angle; the maps do not depend on I)
    return res, to_host(dxp), to_host(dyp)


def _displacement_maps(eng, smp_layers, g3, df_px):
    margin2 = int(np.ceil(float(df_px.max().item()) * 6))
    f32 = dict(device=eng.device, dtype=torch.float32)
    dxp = torch.zeros((eng.nx + 2 * margin2, eng.ny + 2 * margin2), **f32)
    dyp = torch.zeros_like(dxp)
    scratch = torch.zeros((eng.nx, eng.ny), **f32)
    abi.refract_layers(None, 1.0, [(t, d * g3, 0.0, 0.0) for t, d, b in smp_layers], scratch, margin=margin2, dx_pad=dxp, dy_pad=dyp)
    return to_host(dxp), to_host(dyp)
