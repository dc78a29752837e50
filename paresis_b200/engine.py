"""Device-resident image formation for one membrane position.

This is the B200 execution of ``Experiment.computeSampleAndReferenceImages_RT`` /
``_Fresnel`` (reference Experiment.py:407-526 / :279-405): the per-energy loop runs as a
short sequence of fused CUDA kernels on one stream, the accumulators never leave HBM, and
only the detector images come back to the host.  PyTorch provides device memory and streams;
all arithmetic is in ``libparesis_b200.so`` (C ABI, ``include/paresis_b200.h``).

The host shim (``paresis_b200/CodePython/Experiment.py``) builds a :class:`Scene` from the
XML-derived objects and calls :meth:`ImageFormation.compute_rt` / ``compute_fresnel``.
"""
import time
from types import SimpleNamespace

import numpy as np
import torch

from . import _cabi as abi
from . import hostmath as hm

IMAGES = ("sample", "reference", "propag", "white")
DF_SCRATCH = ("angle", "plain", "scattered", "clean", "moved")    # scratch images of paresis_df_run


class _PerPosition:
    """Stands for "the membrane map of the position being computed" in a batched scene."""

    def __repr__(self):
        return "PER_POSITION"


PER_POSITION = _PerPosition()


class Layer:
    """One material of an object: a device thickness map (metres) or a uniform thickness.

    ``scatter``: the dark-field model of a scattering material of the sample, (sphere radius um, volume fraction) as in
    hostmath.MODELS (Sample.py:322-343), or None.  Ray tracing scales that material's delta and beta by the fraction and
    spreads the rays by its scattering angle (paresis_df_run); the Fresnel model ignores it, as the reference does."""

    __slots__ = ("map", "uniform", "delta", "beta", "scatter")

    def __init__(self, thickness, delta, beta, scatter=None):
        # delta / beta: {energy_keV: value}
        if isinstance(thickness, torch.Tensor) or thickness is PER_POSITION:
            self.map, self.uniform = thickness, None
        else:
            self.map, self.uniform = None, float(thickness)
        self.delta, self.beta = delta, beta
        self.scatter = scatter


class Scene:
    """Everything the per-energy loop reads (products of Experiment.__init__, Experiment.py:81-100).

    ``membrane`` may mix mapped and uniform layers (the support plate is uniform: it only
    attenuates).  ``sample`` may hold any number of mapped and uniform layers: when they do not fit
    a hop, they reach it as two mixed maps per energy (ImageFormation.mixed_sample)."""

    def __init__(self, study_dims, study_pixel_um, oversampling, det_dims, det_pixel_um, psf_sigma,
                 d_source_membrane, d_membrane_object, d_object_detector, mean_shot_count,
                 spectrum, source_size_um, energy_sampling, thresholds, membrane, sample,
                 common_factor=None, plate_factor=None):
        self.study_dims = (int(study_dims[0]), int(study_dims[1]))
        self.study_pixel_um = float(study_pixel_um)
        self.os = int(oversampling)
        self.det_dims = (int(det_dims[0]), int(det_dims[1]))
        self.det_pixel_um = float(det_pixel_um)
        self.psf_sigma = float(psf_sigma)
        self.d1, self.d2, self.d3 = float(d_source_membrane), float(d_membrane_object), float(d_object_detector)
        self.magnification = (self.d1 + self.d3 + self.d2) / (self.d1 + self.d2)
        self.mean_shot_count = float(mean_shot_count)
        self.spectrum = [(float(e), float(w)) for e, w in spectrum]
        self.source_size_um = float(source_size_um)
        self.energy_sampling = float(energy_sampling)
        self.thresholds = list(thresholds)   # already closed by the last energy (Experiment.py:429)
        self.membrane = list(membrane)
        self.sample = list(sample)
        # per-energy scalar factors on the incident intensity: air volume and scintillator
        # efficiency (Experiment.py:452-459); detector protection plate (:478-480, :494-496)
        self.common_factor = common_factor or (lambda e: 1.0)
        self.plate_factor = plate_factor or (lambda e: 1.0)

    def effective_source_fwhm(self):
        """Experiment.py:503 (FWHM in oversampled pixels)."""
        return self.source_size_um * self.d3 / (self.d1 + self.d2) / self.det_pixel_um * self.os


class InsaneValues(Exception):
    pass


def _on_own_device(method):
    """Library calls launch on the CURRENT device: make the engine's device current for the duration of the call."""
    import functools

    @functools.wraps(method)
    def wrapper(self, *args, **kwargs):
        with torch.cuda.device(self.device):
            return method(self, *args, **kwargs)
    return wrapper


class ImageFormation:
    """Owns the scratch buffers of one GPU and runs membrane positions one after another."""

    def __init__(self, study_dims, oversampling, det_dims, device=None, seed=None, poisson=True):
        if not torch.cuda.is_available():
            raise RuntimeError("paresis_b200 needs a CUDA device (B200); there is no CPU path")
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.nx, self.ny = int(study_dims[0]), int(study_dims[1])
        self.os = int(oversampling)
        self.det_x, self.det_y = int(det_dims[0]), int(det_dims[1])
        self.poisson = poisson
        # Detector.py:113 seeds from the wall clock; so do we unless told otherwise
        self.seed = int(np.floor(time.time() * 100 % (2 ** 32 - 1))) if seed is None else int(seed)
        f32 = dict(device=self.device, dtype=torch.float32)
        n = (self.nx, self.ny)
        self.i_bs = torch.zeros(n, **f32)      # invariant of paresis_rt_run: all zero between jobs
        self.i_bs_group = []                   # further such buffers, made when a detector bin holds several energies
        self._i_bs_dirty = False
        self.acc = {k: torch.zeros(n, **f32) for k in IMAGES}
        self.work = torch.empty(abi.detect_work_floats(self.nx, self.ny, self.os, self.det_x, self.det_y), **f32)
        self.expect = torch.empty((self.det_x, self.det_y), **f32)
        self.flag = torch.zeros(1, device=self.device, dtype=torch.int32)
        self.means = torch.zeros(256, device=self.device, dtype=torch.float64)
        self.dx_pad = None
        self.dy_pad = None
        self._kernels = {}
        self._plan = None
        self._vectors = {}
        self._waves = None
        self._mixed = {}         # (material maps, weights) -> the mixed maps of one energy (mixed_sample)
        self._mixed_of = None    # the material maps the cached mixed maps were made from
        self._df = None          # scratch images of paresis_df_run, made with the first scattering sample

    # ------------------------------------------------------------------ helpers
    def _gauss(self, sigma):
        key = round(float(sigma), 12)
        if key not in self._kernels:
            if hm.gaussian_half_width(sigma) == 0:
                self._kernels[key] = None      # 1x1 kernel == identity (round(3*sigma) == 0, Detector.py:212)
            else:
                self._kernels[key] = torch.as_tensor(hm.gaussian_1d(sigma), device=self.device, dtype=torch.float32)
        return self._kernels[key]

    @_on_own_device
    def detect(self, image, fwhm, psf_sigma, sequence, out):
        """Detector.detection (Detector.py:79-119): device image -> ``out`` (device, detector dims)."""
        src = self._gauss(fwhm / 2.355) if fwhm != 0 else None
        psf = self._gauss(psf_sigma) if psf_sigma != 0 else None
        abi.detect_counts(image, self.os, self.det_x, self.det_y, src, psf, self.work, out, self.poisson, self.seed, sequence)

    def check_flag(self):
        """The reference's NaN / 'insane values' guard (refractionFileNumba2.py:81-82), checked lazily."""
        if int(self.flag.item()) & abi.FLAG_NONFINITE:
            self.flag.zero_()
            raise InsaneValues("The calculated intensity refractive includes some nans or insane values")

    @staticmethod
    def _split(layers, energy):
        """-> maps [(tensor, delta, beta)], sum(beta*t) and sum(delta*t) of the uniform layers."""
        maps, ub, ud = [], 0.0, 0.0
        for L in layers:
            d, b = L.delta.get(energy, 0.0), L.beta.get(energy, 0.0)   # a missing energy leaves 0 (Sample.py:303-319)
            if L.map is not None:
                maps.append((L.map, d, b))
            else:
                ub += b * L.uniform
                ud += d * L.uniform
        return maps, ub, ud

    # ------------------------------------------------------------------ samples with many materials
    @staticmethod
    def sample_fits(scene, with_membrane):
        """Whether the sample's layers go to the hops as they are: all mapped, and at most MAX_LAYERS maps per hop
        (``with_membrane``: the membrane maps share the hop, as in ray tracing)."""
        if any(L.map is None for L in scene.sample):
            return False
        used = len(scene.sample) + (sum(L.map is not None for L in scene.membrane) if with_membrane else 0)
        return used <= abi.MAX_LAYERS

    def mixed_sample(self, layers, energy, fractions=None):
        """The sample at ``energy`` as two layers [(P, delta*, 0), (B, 0, beta*)] (DESIGN.md, "Samples of any number
        of materials"): P = sum_m (delta_m / delta*) t_m, B = sum_m (beta_m / beta*) t_m + (sum of uniform beta t) / beta*,
        delta* / beta* the largest coefficients of that energy.  Everything a hop does with the sample is linear in
        thickness, so these two maps stand for all of them; a uniform layer's constant phase has no gradient and is a
        global phase of a wave, so uniform layers only enter B.  ``fractions``: per-layer factors on the thickness (the
        volume fraction of a dark-field material, Sample.py:333, :344).

        The maps depend on (sample, energy) only: they are made once and kept while the sample's maps stay the same."""
        fractions = fractions if fractions is not None else [1.0] * len(layers)
        maps, d, b, uniform, bias = [], [], [], [], 0.0
        for L, f in zip(layers, fractions):
            dl, bl = L.delta.get(energy, 0.0) * f, L.beta.get(energy, 0.0) * f   # a missing energy leaves 0 (Sample.py:303-319)
            if L.map is None:
                uniform.append(bl)
                bias += bl * L.uniform
            else:
                maps.append(L.map)
                d.append(dl)
                b.append(bl)
        if not maps and not uniform:
            raise NotImplementedError("the sample has no layer")
        d_star = max((abs(v) for v in d), default=0.0) or 1.0
        b_star = max((abs(v) for v in b + uniform), default=0.0) or 1.0
        w_p, w_b, bias_b = [v / d_star for v in d], [v / b_star for v in b], bias / b_star
        source = tuple(t.data_ptr() for t in maps)
        if source != self._mixed_of:
            self._mixed.clear()
            self._mixed_of = source
        key = (tuple(w_p), tuple(w_b), bias_b)
        if key not in self._mixed:
            try:
                p_map = torch.empty((self.nx, self.ny), device=self.device, dtype=torch.float32)
                b_map = torch.empty_like(p_map)
            except torch.cuda.OutOfMemoryError as exc:
                raise MemoryError("a sample of %d materials needs %d bytes of device memory per energy for its mixed "
                                  "phase and attenuation maps (2 x %d x %d float32); %d energies are held already"
                                  % (len(layers), 8 * self.nx * self.ny, self.nx, self.ny, len(self._mixed))) from exc
            if maps:
                abi.mix_maps(maps, [w_p, w_b], [0.0, bias_b], [p_map, b_map])
            else:
                abi.fill(p_map, 0.0)
                abi.fill(b_map, bias_b)
            # the material maps are held with their mix: their addresses identify it
            self._mixed[key] = (p_map, b_map, tuple(maps))
        p_map, b_map, _ = self._mixed[key]
        return [(p_map, d_star, 0.0), (b_map, 0.0, b_star)]

    def _sample_layers(self, scene, energy, fits, fractions=None):
        """-> [(map, delta, beta)] the hops take for the sample at ``energy``; ``fractions``: see mixed_sample."""
        if not fits:
            return self.mixed_sample(scene.sample, energy, fractions)
        maps = self._split(scene.sample, energy)[0]
        if fractions is None:
            return maps
        return [(t, d * f, b * f) for (t, d, b), f in zip(maps, fractions)]

    @staticmethod
    def scatters(scene):
        """Whether a material of the sample has a dark-field model (Layer.scatter)."""
        return any(L.scatter is not None for L in scene.sample)

    @staticmethod
    def _rt_fractions(scene):
        """Per sample layer: the volume fraction of a scattering material, 1 otherwise (Sample.py:333, :344); None when
        nothing scatters."""
        if not ImageFormation.scatters(scene):
            return None
        return [L.scatter[1] if L.scatter is not None else 1.0 for L in scene.sample]

    def _new_outputs(self, nbins, first):
        """Detector images of one position, stacked [image][bin][x][y] in ONE device buffer
        (sample, reference; + propag, white at position 0) so they cross PCIe as one copy."""
        count = 4 if first else 2
        stack = torch.empty((count, nbins, self.det_x, self.det_y), device=self.device, dtype=torch.float32)
        out = {k: stack[i] for i, k in enumerate(IMAGES[:count])}
        out["_stack"] = stack
        return out

    def _mean_energy(self, energies, sums):
        """Experiment.py:485-486, :523 (Fresnel :351-358).  ``sums`` = per-energy sums of the reference beam, formed
        while it is deposited (ray tracing) or propagated (Fresnel)."""
        per = np.asarray(sums, dtype=np.float64) / float(self.nx * self.ny)
        return float(np.dot(per, energies)), float(per.sum())

    # ------------------------------------------------------------------ ray tracing
    def bins(self, scene):
        """Spectrum indices of each detector bin (closing rule of Experiment.py:501)."""
        out, cur, ibin = [], [], 0
        for ie, (energy, _) in enumerate(scene.spectrum):
            cur.append(ie)
            if energy > scene.thresholds[ibin] - scene.energy_sampling / 2:
                out.append(cur)
                cur, ibin = [], ibin + 1
        if cur:
            out.append(cur)     # energies after the last threshold never reach the detector (as upstream)
        return out

    def _rt_energies(self, scene, indices, closing):
        """ctypes array of per-energy hop scalars for the spectrum entries ``indices``; ``closing`` =
        set of spectrum indices after which the detector runs."""
        s = scene
        g2 = hm.refraction_gradient_scale(s.d2, s.magnification, s.study_pixel_um)
        g3 = hm.refraction_gradient_scale(s.d3, s.magnification, s.study_pixel_um)
        energies = (abi.RtEnergy * len(indices))()
        keep = []
        fits = self.sample_fits(s, with_membrane=True)
        fractions = self._rt_fractions(s)
        for slot, ie in enumerate(indices):
            energy, flux = s.spectrum[ie]
            k = hm.wavenumber(energy * 1000)
            i0 = s.mean_shot_count / s.os ** 2 * flux * s.common_factor(energy)      # :438, :451-459
            plate = s.plate_factor(energy)
            mem_maps, mem_ub, _ = self._split(s.membrane, energy)
            smp_maps = self._sample_layers(s, energy, fits, fractions)
            if not mem_maps or not smp_maps or len(mem_maps) + len(smp_maps) > abi.MAX_LAYERS:
                raise NotImplementedError("scene needs 1+ membrane maps and a sample, at most %d maps per hop"
                                          % abi.MAX_LAYERS)
            en = energies[slot]
            # uniform layers and the plate only scale the beam (:463, :478-480)
            en.intensity_membrane = i0 * np.exp(-2 * k * mem_ub) * plate
            en.intensity_propag = i0 * plate
            hop1 = [(t, d * g2, 0.0, 2 * k * b) for t, d, b in mem_maps]
            hop2 = [(t, d * g3, d * g3, 0.0) for t, d, b in mem_maps] + [(t, d * g3, 0.0, 2 * k * b) for t, d, b in smp_maps]
            prop = [(t, d * g3, 0.0, 2 * k * b) for t, d, b in smp_maps]
            for dst, src in ((en.hop1, hop1), (en.hop2, hop2), (en.propag, prop)):
                for m, (t, go, gr, at) in enumerate(src):
                    # a NULL map = the membrane of the position at hand (paresis_rt_run_positions)
                    dst[m].thickness = None if t is PER_POSITION else t.data_ptr()
                    dst[m].grad_obj, dst[m].grad_ref, dst[m].atten = go, gr, at
                    keep.append(t)
            en.n_hop1, en.n_hop2, en.n_propag = len(hop1), len(hop2), len(prop)
            en.close_bin = 1 if ie in closing else 0
        return energies, keep

    def _detector_fields(self, job, scene, sequence):
        """The fields paresis_rt_job and paresis_fresnel_job share: detector geometry and kernels, noise, the per-energy
        sums (self.means, grown to ``job.n_energies``) and the detector work.  Returns the kernels the job points to."""
        fwhm = scene.effective_source_fwhm()
        src = self._gauss(fwhm / 2.355) if fwhm != 0 else None
        psf = self._gauss(scene.psf_sigma) if scene.psf_sigma != 0 else None
        if job.n_energies > self.means.numel():
            self.means = torch.zeros(job.n_energies, device=self.device, dtype=torch.float64)
        job.oversampling, job.det_x, job.det_y = self.os, self.det_x, self.det_y
        job.means, job.detect_work = self.means.data_ptr(), self.work.data_ptr()
        job.src_kernel, job.src_half = (src.data_ptr(), (src.numel() - 1) // 2) if src is not None else (None, 0)
        job.psf_kernel, job.psf_half = (psf.data_ptr(), (psf.numel() - 1) // 2) if psf is not None else (None, 0)
        job.noise, job.seed, job.sequence = int(self.poisson), self.seed, sequence
        return src, psf

    def _rt_job(self, scene, energies, first, sequence, group=True):
        job = abi.RtJob()
        job.nx, job.ny = self.nx, self.ny
        job.first_point, job.n_energies, job.energies_host = int(first), len(energies), energies
        kernels = self._detector_fields(job, scene, sequence)
        job.i_bs = self.i_bs.data_ptr()
        job.i_bs_dirty = 1 if self._i_bs_dirty else 0
        for k, t in enumerate(self._group_buffers(scene) if group else ()):
            job.i_bs_group[k] = t.data_ptr()
        job.acc_sample, job.acc_ref = self.acc["sample"].data_ptr(), self.acc["reference"].data_ptr()
        job.acc_propag, job.acc_white = self.acc["propag"].data_ptr(), self.acc["white"].data_ptr()
        job.flag = self.flag.data_ptr()
        return job, kernels

    def _group_buffers(self, scene, owner=None):
        """Extra object-plane buffers so that up to MAX_GROUP energies of a detector bin share one object hop."""
        want = min(abi.MAX_GROUP, max((len(b) for b in self.bins(scene)), default=1)) - 1
        store = self.i_bs_group if owner is None else owner.setdefault("i_bs_group", [])
        while len(store) < want:
            store.append(torch.zeros((self.nx, self.ny), device=self.device, dtype=torch.float32))
        return store[:want]

    # ------------------------------------------------------------------ scattering samples (dark field)
    def _df_energies(self, scene, indices):
        """ctypes array of paresis_df_energy for the spectrum entries ``indices``: the angle map comes from the last
        scattering material's own thickness map (Sample.py:322-343 overwrites newDf), also when the hops see mixed maps."""
        s = scene
        to_px = s.d3 / (s.study_pixel_um * 1e-6 * s.magnification)           # refractionFileNumba2.py:114
        last = [L for L in s.sample if L.scatter is not None][-1]
        if last.map is None or last.map is PER_POSITION:
            raise NotImplementedError("a scattering material needs a thickness map of its own")
        out = (abi.DfEnergy * len(indices))()
        for slot, ie in enumerate(indices):
            energy, flux = s.spectrum[ie]
            out[slot].scatter_map = last.map.data_ptr()
            out[slot].angle_coeff = hm.angle_coefficient(last.delta.get(energy, 0.0), last.scatter) * to_px
            out[slot].dark_field_weight = flux / to_px                          # Experiment.py:491, in radians
        return out, last.map

    def _df_scratch(self):
        """The scratch images of paresis_df_run: angle, plain, scattered, clean, moved (any content between jobs)."""
        if self._df is None:
            self._df = self._new_df_scratch()
        return self._df

    def _new_df_scratch(self):
        return {k: torch.empty((self.nx, self.ny), device=self.device, dtype=torch.float32) for k in DF_SCRATCH}

    def _df_job(self, scene, job, indices, dark_field=None):
        """Wrap a paresis_rt_job (``job``) into a paresis_df_job for the spectrum entries ``indices``."""
        df_energies, keep = self._df_energies(scene, indices)
        scratch = self._df_scratch()
        dj = abi.DfJob()
        dj.rt = job
        dj.energies_df_host = df_energies
        for k in DF_SCRATCH:
            setattr(dj, k, scratch[k].data_ptr())
        dj.dark_field = dark_field.data_ptr() if dark_field is not None else None
        return dj, (df_energies, keep)

    @staticmethod
    def _rt_launches(n_energies, n_bins, first):
        # per energy: membrane hop, object hop (+ the sample-only hop at position 0); per bin: the detector (+ the white
        # fill)
        return n_energies * (3 if first else 2) + n_bins * (2 if first else 1)

    @staticmethod
    def _df_launches(n_energies, n_bins, first):
        # per energy: angle, membrane hop, split, 2 object hops, scatter (+ split, 2 hops, scatter, dark-field axpy at
        # position 0); per bin: the detector (+ the white fill)
        return n_energies * (11 if first else 6) + n_bins * (2 if first else 1)

    def _df_displacement(self, scene):
        """Dx, Dy of the sample-only beam at the last energy into self.dx_pad / self.dy_pad, zero-padded by
        margin2 = ceil(6 max(angle)) as fastRefractionDF returns them (refractionFileNumba2.py:115-117, Experiment.py:492);
        the angle map is the one paresis_df_run left in its scratch."""
        s = scene
        scratch = self._df_scratch()
        margin2 = int(np.ceil(float(scratch["angle"].max().item()) * 6))
        shape = (self.nx + 2 * margin2, self.ny + 2 * margin2)
        self.dx_pad = torch.zeros(shape, device=self.device, dtype=torch.float32)
        self.dy_pad = torch.zeros_like(self.dx_pad)
        g3 = hm.refraction_gradient_scale(s.d3, s.magnification, s.study_pixel_um)
        layers = self._sample_layers(s, s.spectrum[-1][0], self.sample_fits(s, with_membrane=True), self._rt_fractions(s))
        # the image goes to scratch: only the maps are wanted (paresis_df_run clears `moved` before it reads it)
        abi.refract_layers(None, 1.0, [(t, d * g3, 0.0, 0.0) for t, d, b in layers], scratch["moved"], margin=margin2,
                           dx_pad=self.dx_pad, dy_pad=self.dy_pad)

    @staticmethod
    def sequence(point_num, sequence_base=0):
        """Poisson stream id of a position; image k of bin b draws from sequence + 4b + k."""
        return (sequence_base + point_num) << 16

    @_on_own_device
    def compute_rt(self, scene, point_num, want_displacement=False, sequence_base=0, probe=None, want_mean=True,
                   defer=False):
        """Experiment.computeSampleAndReferenceImages_RT (Experiment.py:407-526) as one library
        call (paresis_rt_run; paresis_df_run when a sample material scatters, Layer.scatter).

        Returns a dict of device tensors [nbins, det_x, det_y]: sample, reference (+ propag, white
        at position 0; absent keys are all-zero images), plus ``mean_energy`` = (sum E*mean,
        sum mean) of Experiment.py:485-486.  A scattering sample adds ``dark_field`` at position 0: the
        [nx, ny] float32 map of Experiment.py:491 (radians, summed over the spectrum).  ``want_displacement``
        leaves the Dx, Dy maps of the sample-only beam at the last energy in self.dx_pad / self.dy_pad."""
        s = scene
        first = point_num == 0
        bins = self.bins(s)
        nbins, n_e = len(s.thresholds), len(s.spectrum)
        out = self._new_outputs(nbins, first)
        scatters = self.scatters(s)
        wd = first and want_displacement
        if wd and not scatters and (self.dx_pad is None or self.dx_pad.shape != (self.nx + 30, self.ny + 30)):
            self.dx_pad = torch.empty((self.nx + 30, self.ny + 30), device=self.device, dtype=torch.float32)
            self.dy_pad = torch.empty_like(self.dx_pad)
        closing = {b[-1] for b in bins[:nbins]}
        energies, keep = self._rt_energies(s, list(range(n_e)), closing)
        job, keep2 = self._rt_job(s, energies, first, self.sequence(point_num, sequence_base), group=not scatters)
        job.out_sample, job.out_ref = out["sample"].data_ptr(), out["reference"].data_ptr()
        if first:
            job.out_propag, job.out_white = out["propag"].data_ptr(), out["white"].data_ptr()
        if scatters:
            if first:
                out["dark_field"] = torch.zeros((self.nx, self.ny), device=self.device, dtype=torch.float32)
            dj, keep3 = self._df_job(s, job, list(range(n_e)), out.get("dark_field"))
            self._run_df(dj, self._df_launches(n_e, len(closing), first))
            if wd:
                self._df_displacement(s)
        else:
            if wd:
                job.dx_pad, job.dy_pad = self.dx_pad.data_ptr(), self.dy_pad.data_ptr()
            self._run(job, self._rt_launches(n_e, len(closing), first), probe)
        if want_mean and defer:
            # no host synchronisation here: the per-energy sums and the status flag travel with the images
            # (one small device buffer); the caller finishes with finish_deferred() once they are on the host
            out["aux"] = torch.cat((self.means[:n_e], self.flag.to(torch.float64)))
            self.flag.zero_()
        elif want_mean:
            out["mean_energy"] = self._mean_energy([e for e, _ in s.spectrum], sums=self.means[:n_e].cpu().numpy())
            self.check_flag()
        return out

    def finish_deferred(self, scene, aux_host):
        """``aux_host`` = host copy of ``out["aux"]`` of a deferred compute_rt: -> mean_energy, raising the
        reference's 'insane values' error if the status flag was set."""
        aux = np.asarray(aux_host, dtype=np.float64)
        if int(aux[-1]) & abi.FLAG_NONFINITE:
            raise InsaneValues("The calculated intensity refractive includes some nans or insane values")
        return self._mean_energy([e for e, _ in scene.spectrum], sums=aux[:-1])

    def _run(self, job, launches, probe=None):
        """paresis_rt_run keeps I_bs all-zero between jobs; a failed call may leave it dirty."""
        self._i_bs_dirty = True
        abi.rt_run(job, launches, probe)
        self._i_bs_dirty = False

    def _run_df(self, dj, launches):
        """paresis_df_run keeps the same I_bs contract."""
        self._i_bs_dirty = True
        abi.df_run(dj, launches)
        self._i_bs_dirty = False

    # ------------------------------------------------------------------ many positions, one call
    def _slots(self, n_slots, raster_bytes, fresnel=False, darkfield=False):
        """Scratch sets of paresis_rt_run_positions / paresis_fresnel_run_positions / paresis_df_run_positions: slot 0 is
        this engine's own buffers.  Each slot has detector work of its own (slots run concurrently).  ``fresnel``: each
        slot also gets a Fresnel plan and two waves of its own; ``darkfield``: the five scratch images of paresis_df_run."""
        f32 = dict(device=self.device, dtype=torch.float32)
        cache = self.__dict__.setdefault("_slot_cache", [])
        while len(cache) < n_slots:
            k = len(cache)
            cache.append(dict(
                i_bs=self.i_bs if k == 0 else torch.zeros((self.nx, self.ny), **f32),
                acc={name: (self.acc[name] if k == 0 else torch.empty((self.nx, self.ny), **f32)) for name in IMAGES},
                detect_work=self.work if k == 0 else torch.empty_like(self.work),
                work=None, stream=torch.cuda.Stream(device=self.device), dirty=False))
        for c in cache[:n_slots]:
            if c["work"] is None or c["work"].numel() < raster_bytes:
                c["work"] = torch.empty(raster_bytes, device=self.device, dtype=torch.uint8)
        if fresnel:
            self._fresnel_setup()
            for k, c in enumerate(cache[:n_slots]):
                if "plan" not in c:
                    c["plan"] = self._plan if k == 0 else abi.FresnelPlan(self.nx, self.ny, 15)
                    c["waves"] = self._waves if k == 0 else [torch.empty_like(w) for w in self._waves]
        if darkfield:
            for k, c in enumerate(cache[:n_slots]):
                if "df" not in c:
                    c["df"] = self._df_scratch() if k == 0 else self._new_df_scratch()
        return cache[:n_slots]

    def _positions_buffers(self, n_pos, n_firsts, nbins, n_e):
        """Outputs of a many-positions call: thickness maps, images [P, 2, nbins, dx, dy], the extra images of position 0,
        the per-energy sums."""
        f32 = dict(device=self.device, dtype=torch.float32)
        return dict(thickness=torch.empty((n_pos, self.nx, self.ny), **f32),
                    images=torch.empty((n_pos, 2, nbins, self.det_x, self.det_y), **f32),
                    extra=torch.empty((max(n_firsts, 1), 2, nbins, self.det_x, self.det_y), **f32),
                    sums=torch.zeros((n_pos, n_e), device=self.device, dtype=torch.float64))

    @staticmethod
    def _membrane(plan):
        """paresis_membrane of a geometry.MembranePlan (its sphere field when it has one) -> (struct, field or None)."""
        field = plan.field()
        membrane = abi.Membrane(plan.table.data_ptr(), plan.table.shape[0], plan.pix, plan.layers, plan.margin,
                                field.data_ptr() if field is not None else None,
                                field.shape[0] if field is not None else 0, field.shape[1] if field is not None else 0)
        return membrane, field

    def _c_positions(self, buffers, offsets, points, firsts, layers, sequence_base, want_means):
        """ctypes array of paresis_rt_position, with the offsets array it points to."""
        n_pos = len(offsets)
        offs = np.ascontiguousarray(np.asarray(offsets, dtype=np.int64).reshape(n_pos, layers, 2))
        c_pos = (abi.RtPosition * n_pos)()
        for p in range(n_pos):
            cp = c_pos[p]
            cp.offsets_host = offs[p].ctypes.data_as(abi.ctypes.POINTER(abi.ctypes.c_int64))
            cp.thickness = buffers["thickness"][p].data_ptr()
            cp.out_sample, cp.out_ref = buffers["images"][p, 0].data_ptr(), buffers["images"][p, 1].data_ptr()
            first = points[p] == 0
            if first:
                k = firsts.index(p)
                cp.out_propag, cp.out_white = buffers["extra"][k, 0].data_ptr(), buffers["extra"][k, 1].data_ptr()
            cp.means = buffers["sums"][p].data_ptr() if want_means else None
            cp.sequence = self.sequence(points[p], sequence_base)
            cp.first_point = 1 if first else 0
        return c_pos, offs

    @staticmethod
    def _positions_result(buffers, firsts):
        return dict(thickness=buffers["thickness"], sample=buffers["images"][:, 0], reference=buffers["images"][:, 1],
                    propag=buffers["extra"][:len(firsts), 0], white=buffers["extra"][:len(firsts), 1], sums=buffers["sums"],
                    firsts=firsts, buffers=buffers)

    def _positions_call(self, scene, plan, offsets, points, n_slots, buffers, sequence_base, want_means, slot_type, **kind):
        """What compute_rt_positions, compute_df_positions and compute_fresnel_positions set up alike: the energies that
        close a detector bin, the output buffers, the membrane, a ctypes array of ``slot_type`` with the fields every slot
        struct has (``kind``: see _slots), the positions, and the launches of one position's membrane (``cut``)."""
        n_pos = len(offsets)
        nbins, n_e = len(scene.thresholds), len(scene.spectrum)
        closing = {b[-1] for b in self.bins(scene)[:nbins]}
        firsts = [p for p in range(n_pos) if points[p] == 0]
        if buffers is None:
            buffers = self._positions_buffers(n_pos, len(firsts), nbins, n_e)
        membrane, field = self._membrane(plan)
        raster_bytes = abi.lib.paresis_raster_work_bytes(plan.table.shape[0], plan.layers, self.nx, self.ny)
        slots = self._slots(n_slots, raster_bytes, **kind)
        c_slots = (slot_type * n_slots)()
        for k, (sl, c) in enumerate(zip(c_slots, slots)):
            sl.acc_sample, sl.acc_ref = c["acc"]["sample"].data_ptr(), c["acc"]["reference"].data_ptr()
            sl.acc_propag, sl.acc_white = c["acc"]["propag"].data_ptr(), c["acc"]["white"].data_ptr()
            sl.raster_work, sl.raster_work_bytes = c["work"].data_ptr(), c["work"].numel()
            sl.stream = c["stream"].cuda_stream
            sl.detect_work = c["detect_work"].data_ptr()
            if hasattr(sl, "i_bs"):
                sl.i_bs = c["i_bs"].data_ptr()
                sl.i_bs_dirty = 1 if (c["dirty"] or (k == 0 and self._i_bs_dirty)) else 0
        c_pos, offs = self._c_positions(buffers, offsets, points, firsts, plan.layers, sequence_base, want_means)
        return SimpleNamespace(n_e=n_e, closing=closing, firsts=firsts, buffers=buffers, membrane=membrane, field=field,
                               cut=1 if field is not None else 2, slots=slots, c_slots=c_slots, c_pos=c_pos, offs=offs)

    @_on_own_device
    def compute_rt_positions(self, scene, plan, offsets, points, sequence_base=0, n_slots=2, probe_label=None,
                             probe_events=None, want_means=True, buffers=None, per_launch=0):
        """``len(offsets)`` membrane positions in one library call (paresis_rt_run_positions): per
        position the membrane is rasterised from ``plan`` (geometry.MembranePlan) at ``offsets[p]`` and
        the whole per-energy pipeline runs, positions alternating between ``n_slots`` streams.

        ``per_launch`` > 1: up to that many positions (<= n_slots, <= 8) share ONE launch of the membrane cut, of each
        hop and of the detector (blockIdx.z = position; paresis_rt_job.positions_per_launch) instead of running on
        ``n_slots`` streams -- for grids where one position does not fill the GPU.  Detector bins of one energy only.

        ``scene.membrane`` must hold one ``Layer(PER_POSITION, ...)`` for the rasterised map.
        Returns a dict of device tensors: thickness [P, N, N], sample / reference [P, nbins, dx, dy],
        propag / white [P0, nbins, dx, dy] for the positions with ``points[p] == 0`` (in order),
        sums [P, n_energies] (float64 sums of the reference beam, see paresis_rt_job.means)."""
        s = scene
        if self.scatters(s):
            raise NotImplementedError("scattering (dark-field) samples run many positions per call through "
                                      "compute_df_positions")
        call = self._positions_call(s, plan, offsets, points, n_slots, buffers, sequence_base, want_means, abi.RtSlot)
        energies, keep = self._rt_energies(s, list(range(call.n_e)), call.closing)
        job, keep2 = self._rt_job(s, energies, False, 0)
        job.positions_per_launch = int(per_launch)
        for k, (sl, c) in enumerate(zip(call.c_slots, call.slots)):
            for kk, t in enumerate(self._group_buffers(s, owner=None if k == 0 else c)):
                sl.i_bs_group[kk] = t.data_ptr()
            c["dirty"] = True
        self._i_bs_dirty = True
        launches = 0
        for p in range(len(offsets)):
            if probe_events is not None and probe_events[p] is not None:
                e0, e1 = probe_events[p]
                for e in (e0, e1):
                    if not e.cuda_event:
                        e.record()
                call.c_pos[p].probe_start, call.c_pos[p].probe_end = e0.cuda_event, e1.cuda_event
            launches += call.cut + self._rt_launches(call.n_e, len(call.closing), points[p] == 0)
        abi.rt_run_positions(job, call.membrane, call.c_pos, call.c_slots, launches,
                             probe_label if probe_events is not None else None)
        for c in call.slots:
            c["dirty"] = False
        self._i_bs_dirty = False
        return self._positions_result(call.buffers, call.firsts)

    @_on_own_device
    def compute_df_positions(self, scene, plan, offsets, points, sequence_base=0, n_slots=2, want_means=True, buffers=None):
        """``len(offsets)`` membrane positions of a scattering sample in one library call (paresis_df_run_positions): per
        position the membrane is cut from ``plan`` (geometry.MembranePlan) at ``offsets[p]`` and the dark-field chain of
        compute_rt runs, positions alternating between ``n_slots`` streams, each with buffers of its own.  No host
        synchronisation.

        ``scene.membrane`` must hold one ``Layer(PER_POSITION, ...)`` for the position's map, and a sample material must
        scatter (Layer.scatter).  Arguments and result as compute_rt_positions, plus dark_field [P0, nx, ny] (radians, as
        compute_rt's) for the positions with ``points[p] == 0`` (in order)."""
        s = scene
        if not self.scatters(s):
            raise NotImplementedError("no material of the sample scatters: compute_rt_positions runs such a scene")
        n_pos = len(offsets)
        call = self._positions_call(s, plan, offsets, points, n_slots, buffers, sequence_base, want_means, abi.DfSlot,
                                    darkfield=True)
        energies, keep = self._rt_energies(s, list(range(call.n_e)), call.closing)
        job, keep2 = self._rt_job(s, energies, False, 0, group=False)
        dj, keep3 = self._df_job(s, job, list(range(call.n_e)))
        buffers, firsts = call.buffers, call.firsts
        if "dark_field" not in buffers:
            buffers["dark_field"] = torch.empty((max(len(firsts), 1), self.nx, self.ny), device=self.device, dtype=torch.float32)
        buffers["dark_field"].zero_()         # paresis_df_run_positions adds to it
        for sl, c in zip(call.c_slots, call.slots):
            for name in DF_SCRATCH:
                setattr(sl, name, c["df"][name].data_ptr())
            c["dirty"] = True
        self._i_bs_dirty = True
        c_pos = (abi.DfPosition * n_pos)()
        for p in range(n_pos):
            c_pos[p].rt = call.c_pos[p]
            if points[p] == 0:
                c_pos[p].dark_field = buffers["dark_field"][firsts.index(p)].data_ptr()
        launches = sum(call.cut + self._df_launches(call.n_e, len(call.closing), points[p] == 0) for p in range(n_pos))
        abi.df_run_positions(dj, call.membrane, c_pos, call.c_slots, launches)
        for c in call.slots:
            c["dirty"] = False
        self._i_bs_dirty = False
        res = self._positions_result(buffers, firsts)
        res["dark_field"] = buffers["dark_field"][:len(firsts)]
        return res

    @_on_own_device
    def accumulate_rt(self, scene, point_num, indices, dark_field=None):
        """The energies ``indices`` (all of ONE detector bin) of a position, without the detector:
        leaves the partial sums in ``self.acc`` and returns the per-energy means of the reference
        beam (device float64 tensor, len(indices)).  Used when a bin's energies are spread over
        several GPUs (shard.py).  ``dark_field``: [nx, ny] float32 tensor that a scattering sample at
        position 0 adds these energies' share of compute_rt's ``dark_field`` to."""
        first = point_num == 0
        scatters = self.scatters(scene)
        energies, keep = self._rt_energies(scene, list(indices), closing=set())
        # no detector outputs: the library accumulates only
        job, keep2 = self._rt_job(scene, energies, first, 0, group=not scatters)
        if scatters:
            dj, keep3 = self._df_job(scene, job, list(indices), dark_field if first else None)
            self._run_df(dj, self._df_launches(len(indices), 0, first))
        else:
            self._run(job, self._rt_launches(len(indices), 0, first))
        return self.means[:len(indices)] / float(self.nx * self.ny)

    # ------------------------------------------------------------------ Fresnel
    def _fresnel_setup(self):
        if self._plan is None:
            self._plan = abi.FresnelPlan(self.nx, self.ny, 15)
            c64 = dict(device=self.device, dtype=torch.complex64)
            self._waves = [torch.empty((self.nx, self.ny), **c64) for _ in range(2)]

    def _transfer(self, scene, distance, energy, magnification):
        # everything the transfer function depends on (Experiment.py:243-250): the cache outlives a scene
        key = (distance, energy, magnification, tuple(int(v) for v in scene.study_dims), float(scene.study_pixel_um))
        if key not in self._vectors:
            hx, hy, phase = hm.fresnel_vectors(self.nx, self.ny, 15, scene.study_dims, scene.study_pixel_um,
                                               distance, energy, magnification)
            hx, hy = torch.as_tensor(hx, device=self.device), torch.as_tensor(hy, device=self.device)
            # the convolution kernels of this transfer function, prepared once for every position of the scan
            self._vectors[key] = (self._plan.kernel(hx, hy), phase)
        return self._vectors[key]

    @_on_own_device
    def propagate(self, scene, wave_in, distance, energy, magnification, wave_out=None, intensity_acc=None):
        """Experiment.wavePropagation (Experiment.py:219-252) on device fields."""
        self._fresnel_setup()
        kern, phase = self._transfer(scene, distance, energy, magnification)
        # |.|^2 ignores the global phase; a returned field carries it (formed in fp64 on the host)
        self._plan.convolve(wave_in, kern, phase if wave_out is not None else 1.0, wave_out, intensity_acc)

    @staticmethod
    def fresnel_amplitude(scene, energy, flux):
        """Amplitude of the incident wave at one energy (Experiment.py:308, :320-333); the plate scales every intensity
        linearly (:352-356).  Its square is that energy's share of the white field (:372-375)."""
        i0 = scene.mean_shot_count / scene.os ** 2 * flux * scene.common_factor(energy)
        return float(np.sqrt(i0 * scene.plate_factor(energy)))

    def _fresnel_energies(self, scene, indices, closing):
        """ctypes array of paresis_fresnel_energy for the spectrum entries ``indices``; ``closing`` = set of spectrum
        indices after which the detector runs.  Returns it with what it points to."""
        self._fresnel_setup()
        s = scene
        mag_mem_obj = (s.d1 + s.d2) / s.d1                                            # :340
        energies = (abi.FresnelEnergy * len(indices))()
        keep = []
        fits = self.sample_fits(s, with_membrane=False)
        for slot, ie in enumerate(indices):
            energy, flux = s.spectrum[ie]
            k = hm.wavenumber(energy * 1000)
            amp = self.fresnel_amplitude(s, energy, flux)
            mem_maps, mem_ub, _ = self._split(s.membrane, energy)
            smp_maps = self._sample_layers(s, energy, fits)
            if not mem_maps or not smp_maps:
                raise NotImplementedError("scene needs 1+ membrane maps and a sample")
            en = energies[slot]
            # after the membrane (:338); uniform layers: attenuation folded in, constant phase dropped
            en.amplitude_membrane = amp * np.exp(-k * mem_ub)
            en.amplitude_propag = amp
            en.white = amp * amp
            membrane = (abi.WaveLayer * len(mem_maps))()
            for dst, (t, d, b) in zip(membrane, mem_maps):
                # a NULL map = the membrane of the position at hand (paresis_fresnel_run_positions)
                dst.thickness = None if t is PER_POSITION else t.data_ptr()
                dst.atten, dst.phase = k * b, k * d
            en.membrane_host, en.n_membrane = membrane, len(mem_maps)
            for dst, (t, d, b) in zip(en.sample, smp_maps):
                dst.thickness, dst.atten, dst.phase = t.data_ptr(), k * b, k * d
            en.n_sample = len(smp_maps)
            hops = (("reference", s.d3 + s.d2, s.magnification),                      # :349
                    ("to_object", s.d2, mag_mem_obj),                                 # :340-341
                    ("to_detector", s.d3, s.magnification))                           # :348, :365
            for name, distance, magnification in hops:
                kern, phase = self._transfer(s, distance, energy, magnification)
                setattr(en, name, kern._h)
                setattr(en, "phase_" + name, abi.C32(float(np.real(phase)), float(np.imag(phase))))
            en.close_bin = 1 if ie in closing else 0
            keep += [membrane] + [t for t, _, _ in mem_maps + smp_maps if t is not PER_POSITION]
        return energies, keep

    def _fresnel_job(self, scene, energies, first, sequence):
        job = abi.FresnelJob()
        job.plan = self._plan._h
        job.first_point, job.n_energies, job.energies_host = int(first), len(energies), energies
        kernels = self._detector_fields(job, scene, sequence)
        job.wave_a, job.wave_b = self._waves[0].data_ptr(), self._waves[1].data_ptr()
        job.acc_sample, job.acc_ref = self.acc["sample"].data_ptr(), self.acc["reference"].data_ptr()
        job.acc_propag, job.acc_white = self.acc["propag"].data_ptr(), self.acc["white"].data_ptr()
        return job, kernels

    @staticmethod
    def _fresnel_launches(n_energies, n_bins, first):
        # per energy: 2 transmissions + 3 propagations (+ 1 + 1 at position 0), counted as _cabi does; per bin: the
        # detector (+ the white fill)
        return n_energies * (20 if not first else 27) + n_bins * (2 if first else 1)

    @_on_own_device
    def compute_fresnel(self, scene, point_num, sequence_base=0):
        """Experiment.computeSampleAndReferenceImages_Fresnel (Experiment.py:279-405) as one library call
        (paresis_fresnel_run).  Returns what compute_rt returns."""
        s = scene
        first = point_num == 0
        bins = self.bins(s)
        nbins, n_e = len(s.thresholds), len(s.spectrum)
        out = self._new_outputs(nbins, first)
        closing = {b[-1] for b in bins[:nbins]}
        energies, keep = self._fresnel_energies(s, list(range(n_e)), closing)
        job, keep2 = self._fresnel_job(s, energies, first, self.sequence(point_num, sequence_base))
        job.out_sample, job.out_ref = out["sample"].data_ptr(), out["reference"].data_ptr()
        if first:
            job.out_propag, job.out_white = out["propag"].data_ptr(), out["white"].data_ptr()
        abi.fresnel_run(job, self._fresnel_launches(n_e, len(closing), first))
        out["mean_energy"] = self._mean_energy([e for e, _ in s.spectrum], sums=self.means[:n_e].cpu().numpy())
        return out

    @_on_own_device
    def compute_fresnel_positions(self, scene, plan, offsets, points, sequence_base=0, n_slots=2, want_means=True,
                                  buffers=None):
        """``len(offsets)`` membrane positions of the Fresnel model in one library call (paresis_fresnel_run_positions): per
        position the membrane is cut from ``plan`` (geometry.MembranePlan) at ``offsets[p]`` and the Fresnel chain of
        compute_fresnel runs, positions alternating between ``n_slots`` streams, each with a plan and buffers of its own.
        No host synchronisation.

        ``scene.membrane`` must hold one ``Layer(PER_POSITION, ...)`` for the position's map.  Arguments and result as
        compute_rt_positions: thickness [P, N, N], sample / reference [P, nbins, dx, dy], propag / white
        [P0, nbins, dx, dy] for the positions with ``points[p] == 0`` (in order), sums [P, n_energies] (float64 sums of
        the reference beam, see paresis_fresnel_job.means), firsts, buffers."""
        s = scene
        call = self._positions_call(s, plan, offsets, points, n_slots, buffers, sequence_base, want_means, abi.FresnelSlot,
                                    fresnel=True)
        energies, keep = self._fresnel_energies(s, list(range(call.n_e)), call.closing)
        job, keep2 = self._fresnel_job(s, energies, False, 0)
        for sl, c in zip(call.c_slots, call.slots):
            sl.plan = c["plan"]._h
            sl.wave_a, sl.wave_b = c["waves"][0].data_ptr(), c["waves"][1].data_ptr()
        launches = sum(call.cut + self._fresnel_launches(call.n_e, len(call.closing), points[p] == 0)
                       for p in range(len(offsets)))
        abi.fresnel_run_positions(job, call.membrane, call.c_pos, call.c_slots, launches)
        return self._positions_result(call.buffers, call.firsts)

    @_on_own_device
    def accumulate_fresnel(self, scene, point_num, indices):
        """The energies ``indices`` (all of ONE detector bin) of a position, without the detector: leaves the partial
        sums in ``self.acc`` and returns the per-energy means of the reference beam (device float64 tensor,
        len(indices)).  The Fresnel counterpart of accumulate_rt (shard.py)."""
        first = point_num == 0
        energies, keep = self._fresnel_energies(scene, list(indices), closing=set())
        job, keep2 = self._fresnel_job(scene, energies, first, 0)
        abi.fresnel_run(job, self._fresnel_launches(len(indices), 0, first))
        return self.means[:len(indices)] / float(self.nx * self.ny)
