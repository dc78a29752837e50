"""Dark-field branch of the ray-tracing model on the GPU.

Reference: ``fastRefractionDF`` (refractionFileNumba2.py:88-196), the Lung / 'cylinder_beeds' scattering
model of ``AnalyticalSample.setWaveRT`` (Sample.py:322-343) and the places
``computeSampleAndReferenceImages_RT`` threads the dark-field map through (Experiment.py:469-473, :490-492).

The refraction part is the ordinary fused hop run twice -- on the rays with and without a scattering angle
(refractionFileNumba2.py:143-155) -- followed by the variable-width Gaussian scatter of the refracted
dark-field intensity (``paresis_df_scatter``; a Python double loop upstream).  Everything stays on the
device; this module is the per-energy loop of a position whose sample scatters.
"""
import numpy as np
import torch

from . import _cabi as abi
from . import engine
from . import hostmath as hm
from . import transfer
from .host_api import device, to_dev, to_host, InsaneValues

MODELS = {"Lung": (47.0, 0.5), "cylinder_beeds": (15.0, 0.6)}     # sphere radius (um), volume fraction (Sample.py:325-326, :336-337)


def model_of(sample, imat):
    """Which scattering model applies to material ``imat`` of ``sample`` (Sample.py:322-343), or None."""
    if sample.myType != "sample_of_interest":
        return None
    model = "Lung" if sample.myMaterials[imat] == "Lung" else None
    if sample.myName == 'cylinder_beeds':
        model = "cylinder_beeds"          # upstream tests the name after the material: it wins
    return model


def angle_coefficient(delta, model):
    """newDf = coeff * sqrt(thickness[m]) in radians (Sample.py:328-332, :339-343)."""
    radius, fraction = MODELS[model]
    n_vol = fraction * 3 / 4 / np.pi / (radius ** 3)
    return 2 * delta * np.sqrt(n_vol ** (1 / 3) * 1e6) * np.sqrt(np.log(2 / delta) + 1), fraction


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
            coeff, fraction = angle_coefficient(delta[imat], model)
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


# ------------------------------------------------------------------ one position, device resident
def compute_rt(exp, point_num):
    """Experiment.computeSampleAndReferenceImages_RT (Experiment.py:407-526) for a sample with a dark-field
    model: same 7-tuple as the reference."""
    thresholds = exp._open_bins(point_num)
    eng = exp._get_engine()
    scene = exp._scene(thresholds)
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
    smp = exp.mySampleofInterest
    plain, scat, clean, moved, df_px = (torch.empty((nx, ny), **f32) for _ in range(5))
    df_total = torch.zeros((nx, ny), **f32)
    g2 = hm.refraction_gradient_scale(s.d2, s.magnification, s.study_pixel_um)
    g3 = hm.refraction_gradient_scale(s.d3, s.magnification, s.study_pixel_um)
    to_px = s.d3 / (s.study_pixel_um * 1e-6 * s.magnification)
    sums, energies, ibin, white = [], [], 0, 0.0
    fwhm = s.effective_source_fwhm()
    fits = eng.sample_fits(s, with_membrane=True)
    for ie, (energy, flux) in enumerate(s.spectrum):
        print("Current Energy: %gkev" % energy)
        k = hm.wavenumber(energy * 1000)
        i0 = s.mean_shot_count / s.os ** 2 * flux * s.common_factor(energy)
        plate = s.plate_factor(energy)
        mem_maps, mem_ub, _ = eng._split(s.membrane, energy)
        smp_maps, _, _ = eng._split(s.sample, energy)
        # sample layers: the scattering material's thickness counts with its volume fraction; its angle map in pixels
        smp_layers, fractions, have_df = [], [], False
        for imat, (t, d, b) in enumerate(smp_maps):
            model = model_of(smp, imat)
            fraction = 1.0
            if model is not None:
                coeff, fraction = angle_coefficient(d, model)
                abi.df_angle(t, coeff * to_px, df_px)
                have_df = True
            smp_layers.append((t, d * fraction, b * fraction))
            fractions.append(fraction)
        if not have_df:
            df_px.zero_()
        if not fits:
            # more materials than a hop takes: the hops see the two mixed maps, the angle map stays the material's own
            smp_layers = eng.mixed_sample(s.sample, energy, fractions)
        # membrane -> object plane (Experiment.py:463-466)
        eng.i_bs.zero_()
        abi.refract_layers(None, i0 * np.exp(-2 * k * mem_ub) * plate, [(t, d * g2, 0.0, 2 * k * b) for t, d, b in mem_maps],
                           eng.i_bs, flag=eng.flag)
        hop = [(t, d * g3, d * g3, 0.0) for t, d, b in mem_maps] + [(t, d * g3, 0.0, 2 * k * b) for t, d, b in smp_layers]
        # reference beam (:474) and the sample beam split by scattering angle (:473 -> refractionFileNumba2.py:143-155)
        before = eng.acc["reference"].double().sum()
        abi.refract_layers(eng.i_bs, 0.0, [(t, gr, 0.0, 0.0) for t, go, gr, at in hop if gr != 0.0], eng.acc["reference"],
                           flag=eng.flag)
        sums.append(eng.acc["reference"].double().sum() - before)
        energies.append(energy)
        abi.df_split(eng.i_bs, 0.0, df_px, nx / 4, plain, scat, clean)
        obj = [(t, go, 0.0, at) for t, go, gr, at in hop]
        abi.refract_layers(plain, 0.0, obj, eng.acc["sample"], flag=eng.flag)
        moved.zero_()
        abi.refract_layers(scat, 0.0, obj, moved, flag=eng.flag)
        abi.df_scatter(moved, clean, eng.acc["sample"])
        if first:
            # the sample alone (:490-498)
            prop = [(t, d * g3, 0.0, 2 * k * b) for t, d, b in smp_layers]
            abi.df_split(None, i0 * plate, df_px, nx / 4, plain, scat, clean)
            abi.refract_layers(plain, 0.0, prop, eng.acc["propag"], flag=eng.flag)
            moved.zero_()
            abi.refract_layers(scat, 0.0, prop, moved, flag=eng.flag)
            abi.df_scatter(moved, clean, eng.acc["propag"])
            abi.axpy(df_total, df_px, flux / to_px)            # self.darkFieldPropag += DarkFieldPropag * flux (:491), radians
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
    eng._i_bs_dirty = True      # this loop does not keep paresis_rt_run's "I_bs is all zero between jobs" invariant
    try:
        eng.check_flag()
    except engine.InsaneValues as exc:
        raise Exception(str(exc))
    per = torch.stack(sums).cpu().numpy() / float(nx * ny)
    exp.exp_dict['meanEnergy'] = (exp.exp_dict['meanEnergy'] + float(np.dot(per, energies))) / float(per.sum())
    host = transfer.fetch(out["_stack"], torch.float64)
    imgs = [host[i] for i in range(host.shape[0])]
    while len(imgs) < 4:
        imgs.append(exp._zeros(imgs[0].shape))
    if first:
        exp.darkFieldPropag = to_host(df_total)
        # Dx, Dy of the sample-only beam at the last energy (:492), zero-padded by 6 * max(DF) as fastRefractionDF returns them
        exp.Dxreal, exp.Dyreal = _displacement_maps(eng, smp_layers, g3, df_px)
    print("Mean detected energy in reference image", exp.exp_dict['meanEnergy'])
    return imgs[0], imgs[1], imgs[2], imgs[3], exp.Dxreal, exp.Dyreal, exp.darkFieldPropag


def _displacement_maps(eng, smp_layers, g3, df_px):
    margin2 = int(np.ceil(float(df_px.max().item()) * 6))
    f32 = dict(device=eng.device, dtype=torch.float32)
    dxp = torch.zeros((eng.nx + 2 * margin2, eng.ny + 2 * margin2), **f32)
    dyp = torch.zeros_like(dxp)
    scratch = torch.zeros((eng.nx, eng.ny), **f32)
    abi.refract_layers(None, 1.0, [(t, d * g3, 0.0, 0.0) for t, d, b in smp_layers], scratch, margin=margin2, dx_pad=dxp, dy_pad=dyp)
    return to_host(dxp), to_host(dyp)
