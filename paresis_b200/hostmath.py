"""Host-side fp64 scalar/vector preparation for the CUDA kernels.

Everything here is O(N) or O(1) per call: constants with the reference's digits, the 1-D
factors of its Gaussian kernels, the per-axis Fresnel transfer vectors and the per-energy
layer coefficients.  The per-pixel work is in ``csrc/``.
"""
import numpy as np

PLANCK = 6.626e-34   # getk.py:16
LIGHT = 2.998e8      # getk.py:17
CHARGE = 1.6e-19     # getk.py:18


def wavenumber(energy_ev):
    """getk.getk (getk.py:12-20); identical expression at Sample.py:265, :300."""
    return 2 * np.pi * energy_ev * CHARGE / (PLANCK * LIGHT)


def gaussian_half_width(sigma):
    """create_gaussian_shape's ``round(sigma*3)`` (Detector.py:212) -- Python round-half-even."""
    return int(round(sigma * 3))


def gaussian_1d(sigma):
    """1-D factor of create_gaussian_shape (Detector.py:201-220): the 2-D kernel
    exp(-(x^2+y^2)/2s^2)/sum is the outer product of this vector with itself."""
    half = gaussian_half_width(sigma)
    ax = np.arange(-half, half + 1, dtype=np.float64)
    g = np.exp(-(ax ** 2) / 2.0 / sigma ** 2)
    return g / g.sum()


def gaussian_2d(sigma):
    """create_gaussian_shape / gaussian_shape as the reference returns it (host array)."""
    half = gaussian_half_width(sigma)
    ax = np.arange(-half, half + 1, dtype=np.float64)
    g = np.exp(-(ax[None, :] ** 2 / 2.0 / sigma ** 2 + ax[:, None] ** 2 / 2.0 / sigma ** 2))
    return g / np.sum(g)


def fresnel_vectors(nx, ny, margin, study_dims, pixel_um, distance, energy_kev, magnification):
    """Per-axis transfer vectors for Experiment.wavePropagation (Experiment.py:239-250) in FFT
    (unshifted) order, with the inverse-FFT normalisation folded in.  The frequency step is
    2*pi / (N0 * pix) with N0 the UNPADDED study dimension (:246-247)."""
    k = wavenumber(energy_kev * 1000)
    out = []
    for n, n0 in ((nx + 2 * margin, study_dims[0]), (ny + 2 * margin, study_dims[1])):
        a = np.arange(n)
        shifted = (a + n // 2) % n - n // 2          # fftshift index -> signed frequency index
        u = shifted * 2 * np.pi / (n0 * pixel_um * 1e-6)
        out.append(np.exp(-1j * distance * u ** 2 / (2 * k * magnification)) / n)
    phase = np.exp(1j * k * distance / magnification)
    return out[0].astype(np.complex64), out[1].astype(np.complex64), complex(phase)


def refraction_gradient_scale(distance, magnification, pixel_um):
    """Pixels of displacement per unit of (delta * 2-pixel thickness difference):
    D = d(phi)/dx * z / k / (h M), phi = -k delta t, d/dx = (t[+1]-t[-1])/(2h)
    (Sample.py:348, refractionFileNumba2.py:54-56); k cancels."""
    h = pixel_um * 1e-6
    return -distance / (h * magnification) / (2.0 * h)


# dark-field models: sphere radius (um), volume fraction (Sample.py:325-326, :336-337)
MODELS = {"Lung": (47.0, 0.5), "cylinder_beeds": (15.0, 0.6)}


def angle_coefficient(delta, scatter):
    """newDf = coeff * sqrt(thickness[m]) in radians (Sample.py:328-332, :339-343) for a material of refractive decrement
    ``delta`` and ``scatter`` = (sphere radius um, volume fraction), a value of MODELS."""
    radius, fraction = scatter
    n_vol = fraction * 3 / 4 / np.pi / (radius ** 3)
    return 2 * delta * np.sqrt(n_vol ** (1 / 3) * 1e6) * np.sqrt(np.log(2 / delta) + 1)
