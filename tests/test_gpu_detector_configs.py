"""Every detector kernel configuration against the fp64 detection oracle (po.detection, Detector.py:79-119).

paresis_detect_counts picks one of three GPU paths from the oversampling factor os and the half-widths
HS = round(3 sigma_src), HP = round(3 sigma_psf):
  * detect_tile_kernel<OS, HS, HP> (csrc/detector_tile.cuh), one template instance per (OS, HS, HP) of
    PARESIS_DT_DISPATCH -- each with its own window sizes, unroll counts and phase-2 vector width;
  * detect_fused_kernel (csrc/detector.cu) for any other size;
  * the separable global-memory passes plus an in-place paresis_poisson when the fused kernel would need more than
    200 KB of shared memory.
Every tile instance runs at three detector shapes chosen so that its three phase-1 branches are all taken (checked on
the host by replaying the kernel's branch condition), on an input with sharp structure next to every edge, where the
reflect padding and the zero extension beyond the padded frame decide the result.  Noise: a draw is a pure function
of (seed, sequence, pixel) (csrc/poisson.cuh), so counts must equal paresis_poisson of the expectation bit for bit.
"""
import glob
import os
import re

import numpy as np
import pytest

import paresis_oracle as po
from conftest import ROOT, rel_l2

torch = pytest.importorskip("torch")

CSRC = os.path.join(ROOT, "paresis_b200", "csrc")

# sigmas without a rounding tie at 3 sigma -> half-width
SRC_SIGMA = {0: 0.1, 1: 0.4, 2: 0.7}                  # HS
PSF_SIGMA = {0: 0.0, 2: 0.6, 3: 1.0, 4: 1.2, 6: 2.0}    # HP
TILE_INSTANCES = [(o, hs, hp) for o in (1, 2, 3, 4) for hs in SRC_SIGMA for hp in PSF_SIGMA]
# (16, 16): the smallest detector the argument check admits (15 os <= 16 os - 1): the reflect padding reaches the far
# edge; (45, 77): partial tiles both ways, odd det_y (unpaired Philox words), ny % 4 != 0 for odd os;
# (70, 200): ny % 4 == 0, so a middle column tile loads aligned quads, and its last row tile clamps rows
TILE_SHAPES = [(16, 16), (45, 77), (70, 200)]

# the fused kernel: (os, source FWHM in oversampled pixels, PSF sigma in detector pixels), none of them a tile instance
FUSED = [
    (1, 2.355 * 0.4, 0.3),     # HS 1, HP 1
    (3, 2.355 * 0.7, 1.7),     # HS 2, HP 5
    (2, 2.5, 1.2),             # HS 3 (sigma 1.06), HP 4
    (5, 2.355 * 0.4, 1.2),     # HS 1, HP 4, os >= 5
    (4, 2.355 * 0.4, 5.5),     # HS 1, HP 16: 3 x 5.5 = 16.5 rounds half to even, as in the oracle; > 48 KB shared memory
]
FUSED_SHAPES = [(16, 16), (45, 77)]
# the global-memory passes: source sigma 30 (HS 90), PSF sigma 13.4 (HP 40) reach far past the padded frame
WIDE = (4, 2.355 * 30.0, 13.4)
WIDE_DET = (40, 50)

DET_PAD, DT_TX, DT_TY = 15, 32, 64          # csrc/detector_common.cuh, csrc/detector_tile.cuh
FUSED_TB, SMEM_DEFAULT, SMEM_FUSED_MAX = 32, 48 * 1024, 200 * 1024


def half_widths(os_, fwhm, psf_sigma):
    from paresis_b200 import hostmath as hm
    return hm.gaussian_half_width(fwhm / 2.355), (hm.gaussian_half_width(psf_sigma) if psf_sigma else 0)


def fused_smem_bytes(os_, hs, hp):
    """fused_smem_bytes() of csrc/detector.cu."""
    bw = FUSED_TB + 2 * hp
    sw = bw * os_ + 2 * hs
    return 4 * (sw * bw + bw * bw + (os_ + 2 * hs) + (2 * hp + 1) + sw + 2 * FUSED_TB * FUSED_TB)


def phase1_branches(os_, hs, hp, det, image_aligned=True):
    """Which phase-1 branches of detect_tile_kernel<os_, hs, hp> the tiles of one launch take: 'aligned' (128-bit loads,
    every row of the window inside the padded frame), 'clamped' (128-bit loads, rows beyond the frame read as zeros),
    'reflect' (per-column reflect indices).  A restatement of the kernel's `fast` test and the branch on x0."""
    det_x, det_y = det
    nx, ny = det_x * os_, det_y * os_
    npx = nx + 2 * DET_PAD * os_
    swx = (DT_TX + 2 * hp) * os_ + 2 * hs
    swy = (DT_TY + 2 * hp) * os_ + 2 * hs
    r1w = (swy + 6) // 4 * 4
    seen = set()
    for a0 in range(0, det_x, DT_TX):
        x0 = (a0 + DET_PAD - hp) * os_ - hs
        for b0 in range(0, det_y, DT_TY):
            yi0 = (b0 - hp) * os_ - hs
            ya = yi0 - yi0 % 4
            fast = image_aligned and ya >= 0 and ya + r1w <= ny and ny % 4 == 0
            if not fast:
                seen.add("reflect")
            elif x0 >= 0 and x0 + swx <= npx:
                seen.add("aligned")
            else:
                seen.add("clamped")
    return seen


def _macro(text, name):
    """Body of `#define name(...)`, continuation lines joined."""
    m = re.search(r"#define %s\(([^)]*)\)((?:[^\n]*\\\n)*[^\n]*)" % name, text)
    assert m, name
    return m.group(2).replace("\\\n", " ")


def tile_instances_in_sources():
    """(OS, HS, HP) of every detect_tile_kernel the library dispatches to, read from the sources."""
    with open(os.path.join(CSRC, "detector_tile.cuh")) as fh:
        tile = fh.read()
    hps = [int(v) for v in re.findall(r"PARESIS_DT_CASE\(OS_, HS_, (\d+)\)", _macro(tile, "PARESIS_DT_ROW"))]
    hss = [int(v) for v in re.findall(r"PARESIS_DT_ROW\(OS_, (\d+)\)", _macro(tile, "PARESIS_DT_DISPATCH"))]
    assert "launch_detect_tile<OS_, HS_, HP_>" in _macro(tile, "PARESIS_DT_CASE")
    with open(os.path.join(CSRC, "detector.cu")) as fh:
        det = fh.read()
    switch = re.search(r"static int dispatch_detect_tile\(.*?\n\}", det, re.S)
    assert switch
    cases = re.findall(r"case (\d+): return dispatch_detect_tile_os(\d+)\(", switch.group(0))
    assert cases and all(a == b for a, b in cases), cases
    oss = [int(a) for a, _ in cases]
    compiled = []
    for path in glob.glob(os.path.join(CSRC, "detector_tile_os*.cu")):
        with open(path) as fh:
            compiled += [int(v) for v in re.findall(r"^PARESIS_DT_DISPATCH\((\d+)\)", fh.read(), re.M)]
    assert sorted(compiled) == sorted(oss), (compiled, oss)
    out = [(o, hs, hp) for o in oss for hs in hss for hp in hps]
    assert len(set(out)) == len(out)
    return set(out)


# ---------------------------------------------------------------------------------------------------------------------
# host-only checks of the test matrix itself

def test_tile_instance_table_is_the_test_matrix():
    """The parametrisation covers exactly the compiled tile instances, with sigmas that give those half-widths."""
    assert tile_instances_in_sources() == set(TILE_INSTANCES)
    assert len(TILE_INSTANCES) == len(set(TILE_INSTANCES))
    for hs, s in SRC_SIGMA.items():
        assert half_widths(1, 2.355 * s, 0)[0] == hs
        assert abs(3 * s - round(3 * s)) < 0.45          # no tie: the oracle's round() agrees with any rounding
    for hp, s in PSF_SIGMA.items():
        assert half_widths(1, 2.355 * 0.1, s)[1] == hp
        assert abs(3 * s - round(3 * s)) < 0.45
    for os_, fwhm, psf in FUSED:
        hs, hp = half_widths(os_, fwhm, psf)
        assert (os_, hs, hp) not in TILE_INSTANCES
        assert fused_smem_bytes(os_, hs, hp) <= SMEM_FUSED_MAX
    assert max(fused_smem_bytes(o, *half_widths(o, f, p)) for o, f, p in FUSED) > SMEM_DEFAULT   # the attribute path
    assert half_widths(*WIDE) == (90, 40) and fused_smem_bytes(WIDE[0], 90, 40) > SMEM_FUSED_MAX


@pytest.mark.parametrize("os_,hs,hp", TILE_INSTANCES)
def test_tile_shapes_reach_every_phase1_branch(os_, hs, hp):
    seen = set()
    for det in TILE_SHAPES:
        seen |= phase1_branches(os_, hs, hp, det)
    assert seen == {"aligned", "clamped", "reflect"}, seen
    # a misaligned image takes the per-column branch everywhere
    assert phase1_branches(os_, hs, hp, (70, 200), image_aligned=False) == {"reflect"}


# ---------------------------------------------------------------------------------------------------------------------
# GPU

@pytest.fixture(scope="module")
def abi():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from paresis_b200 import _cabi
    return _cabi


def dev(a, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a)).to("cuda", dtype=dtype).contiguous()


def misaligned(shape, fill=0.0):
    """A contiguous float32 view that starts 4 bytes into its allocation (neither 8- nor 16-byte aligned)."""
    buf = torch.full((int(np.prod(shape)) + 1,), fill, device="cuda", dtype=torch.float32)
    return buf[1:].view(shape)


def edge_image(shape, seed):
    """Smooth + random + sharp steps right next to every edge, positive, ~1e3; fp32 values."""
    rng = np.random.default_rng(seed)
    nx, ny = shape
    x = np.linspace(0.0, 1.0, nx)[:, None]
    y = np.linspace(0.0, 1.0, ny)[None, :]
    img = 1000.0 + 250.0 * np.sin(9.0 * x + 4.0 * y) * np.cos(6.0 * y) + rng.uniform(-100.0, 100.0, shape)
    img[0, :] += 300.0
    img[2:5, :] += 600.0
    img[-4:-1, :] -= 400.0
    img[:, 1] += 800.0
    img[:, 3:6] -= 350.0
    img[:, -2] += 500.0
    img[nx // 3:, -6:-3] += 700.0
    return img.astype(np.float32)


def noise_image(shape, os_, seed):
    """Detector expectations from ~0.3 to ~3e4 (inversion below 10, PTRS above), fp32 values."""
    rng = np.random.default_rng(seed)
    nx, ny = shape
    x = np.linspace(0.0, 1.0, nx)[:, None]
    y = np.linspace(0.0, 1.0, ny)[None, :]
    e = -0.5 + 5.0 * (0.5 * x + 0.5 * y) + 0.1 * np.sin(20.0 * x * y)
    return (10.0 ** e / os_ ** 2 * rng.uniform(0.9, 1.1, shape)).astype(np.float32)


def kernels(fwhm, psf_sigma):
    """The 1-D source and PSF factors the engine uploads (None = no blur)."""
    from paresis_b200 import hostmath as hm
    src = dev(hm.gaussian_1d(fwhm / 2.355)) if fwhm != 0 else None
    psf = dev(hm.gaussian_1d(psf_sigma)) if psf_sigma != 0 else None
    return src, psf


def oracle(img32, os_, det, fwhm, psf_sigma):
    return po.detection(img32.astype(np.float64), fwhm, os_, det, psf_sigma)


def ring(a, w):
    m = np.ones(a.shape, dtype=bool)
    m[w:-w, w:-w] = False
    return a[m]


def counts(abi, img, os_, det, src, psf, noise=False, seed=0, seq=0, work=None, out=None):
    if out is None:
        out = torch.full(det, -7.0, device="cuda")
    abi.detect_counts(img, os_, det[0], det[1], src, psf, work, out, noise, seed, seq)
    return out


def poisson_of(abi, expect, seed, seq):
    c = torch.full(expect.shape, -7.0, device="cuda")
    abi.poisson(expect.contiguous(), c, seed, seq)
    return c


def check_against_oracle(got, want, hp):
    assert np.isfinite(got).all()
    assert rel_l2(got, want) < 1e-6
    # the border ring, where the reflect padding and the zero extension live (the global norm dilutes it)
    assert rel_l2(ring(got, hp + 2), ring(want, hp + 2)) < 2e-6


def check_moments(c, lam):
    c = c.double()
    lam = lam.double()
    ok = lam > 0
    z = ((c - lam) / lam.clamp_min(1e-30).sqrt())[ok]
    assert torch.equal(c, c.round()) and c.min().item() >= 0
    assert abs(z.mean().item()) < 0.08 and abs(z.std().item() - 1) < 0.08, (z.mean().item(), z.std().item())


@pytest.mark.gpu
@pytest.mark.parametrize("os_,hs,hp", TILE_INSTANCES)
def test_tile_instance_vs_oracle(abi, os_, hs, hp):
    fwhm, psf_sigma = 2.355 * SRC_SIGMA[hs], PSF_SIGMA[hp]
    src, psf = kernels(fwhm, psf_sigma)
    for k, det in enumerate(TILE_SHAPES):
        img = edge_image((det[0] * os_, det[1] * os_), seed=100 * os_ + 10 * hs + hp + k)
        got = counts(abi, dev(img), os_, det, src, psf).cpu().numpy()
        check_against_oracle(got, oracle(img, os_, det, fwhm, psf_sigma), hp)


@pytest.mark.gpu
@pytest.mark.parametrize("os_,hs,hp", TILE_INSTANCES)
def test_tile_instance_noise_is_poisson_of_expectation(abi, os_, hs, hp):
    """Pair path (even pixel), unpaired path (odd rows of det_y = 77), quick test, step 0 and block queues."""
    det = (45, 77)
    src, psf = kernels(2.355 * SRC_SIGMA[hs], PSF_SIGMA[hp])
    img = dev(noise_image((det[0] * os_, det[1] * os_), os_, seed=os_ + hs + hp))
    lam = counts(abi, img, os_, det, src, psf)
    assert lam.min().item() < 1.0 and lam.max().item() > 1e4
    assert (lam < 10).sum().item() > 200 and (lam >= 10).sum().item() > 200
    for seed, seq in ((5, 0), (2 ** 40 + 3, 2 ** 33 + 17)):
        c = counts(abi, img, os_, det, src, psf, noise=True, seed=seed, seq=seq)
        assert torch.equal(c, poisson_of(abi, lam, seed, seq))
    check_moments(c, lam)


@pytest.mark.gpu
@pytest.mark.parametrize("os_,hs,hp", [(2, 1, 3), (3, 2, 4)])
@pytest.mark.parametrize("det", [(70, 200), (45, 77)])
def test_tile_kernel_unaligned_views(abi, os_, hs, hp, det):
    """An image view 4 bytes into its allocation takes the per-column branch of phase 1, which adds the same taps in
    the same order as the 128-bit branches; an output view 4 bytes in makes the float2 stores step aside."""
    src, psf = kernels(2.355 * SRC_SIGMA[hs], PSF_SIGMA[hp])
    shape = (det[0] * os_, det[1] * os_)
    img = dev(noise_image(shape, os_, seed=3) * 1e-3 + edge_image(shape, seed=4))
    img_off = misaligned(shape)
    img_off.copy_(img)
    assert img_off.data_ptr() % 16 == 4
    for noise in (False, True):
        ref = counts(abi, img, os_, det, src, psf, noise=noise, seed=9, seq=4)
        assert torch.equal(counts(abi, img_off, os_, det, src, psf, noise=noise, seed=9, seq=4), ref), noise
        out_off = misaligned(det, -7.0)
        counts(abi, img, os_, det, src, psf, noise=noise, seed=9, seq=4, out=out_off)
        assert torch.equal(out_off, ref), noise
        assert out_off._base[0].item() == -7.0          # nothing written in front of the view


@pytest.mark.gpu
@pytest.mark.parametrize("os_,fwhm,psf_sigma", FUSED)
def test_fused_kernel_vs_oracle(abi, os_, fwhm, psf_sigma):
    hs, hp = half_widths(os_, fwhm, psf_sigma)
    src, psf = kernels(fwhm, psf_sigma)
    for k, det in enumerate(FUSED_SHAPES):
        shape = (det[0] * os_, det[1] * os_)
        img = edge_image(shape, seed=7 * os_ + hp + k)
        got = counts(abi, dev(img), os_, det, src, psf).cpu().numpy()
        check_against_oracle(got, oracle(img, os_, det, fwhm, psf_sigma), hp)
    nimg = dev(noise_image(shape, os_, seed=hs + hp))
    lam = counts(abi, nimg, os_, det, src, psf)
    c = counts(abi, nimg, os_, det, src, psf, noise=True, seed=21, seq=2 ** 35 + 1)
    assert torch.equal(c, poisson_of(abi, lam, 21, 2 ** 35 + 1))
    check_moments(c, lam)


@pytest.mark.gpu
def test_wide_kernels_take_global_memory_passes(abi):
    """More than 200 KB of shared memory for the fused kernel: blur, bin and PSF as separable passes through the work
    buffer, then the draw in place.  The kernels reach far past the padded frame: the oracle's zero extension."""
    os_, fwhm, psf_sigma = WIDE
    det = WIDE_DET
    shape = (det[0] * os_, det[1] * os_)
    src, psf = kernels(fwhm, psf_sigma)
    assert (src.numel(), psf.numel()) == (181, 81)
    img = edge_image(shape, seed=31)
    work = torch.empty(abi.detect_work_floats(shape[0], shape[1], os_, det[0], det[1]), device="cuda")
    lam = counts(abi, dev(img), os_, det, src, psf, work=work)
    want = oracle(img, os_, det, fwhm, psf_sigma)
    got = lam.cpu().numpy()
    assert np.isfinite(got).all()
    # (hundreds of fp32 taps per output in four passes)
    assert rel_l2(got, want) < 1e-6
    assert rel_l2(ring(got, 8), ring(want, 8)) < 2e-6
    c = counts(abi, dev(img), os_, det, src, psf, noise=True, seed=77, seq=5, work=work)
    assert torch.equal(c, poisson_of(abi, lam, 77, 5))
    with pytest.raises(abi.ParesisError, match="needs the work buffer"):
        counts(abi, dev(img), os_, det, src, psf)


MULTI_CONFIGS = [(2, 2.355 * 0.4, 1.0), (3, 2.355 * 0.7, 1.7)]    # tile instance (2, 1, 3); fused (HS 2, HP 5)


@pytest.mark.gpu
@pytest.mark.parametrize("os_,fwhm,psf_sigma", MULTI_CONFIGS)
def test_images_in_one_launch_match_one_by_one(abi, os_, fwhm, psf_sigma):
    det = (45, 77)
    shape = (det[0] * os_, det[1] * os_)
    src, psf = kernels(fwhm, psf_sigma)
    imgs = [dev(noise_image(shape, os_, seed=50 + k) * (1.0 + 0.25 * k) + 0.01 * edge_image(shape, seed=k))
            for k in range(8)]
    seqs = [1000 + 37 * k for k in range(8)]
    for n in (1, 2, 4, 8):
        for noise in (False, True):
            single = [counts(abi, imgs[k], os_, det, src, psf, noise=noise, seed=13, seq=seqs[k]) for k in range(n)]
            multi = [torch.full(det, -7.0, device="cuda") for _ in range(n)]
            abi.detect_counts_multi(imgs[:n], os_, det[0], det[1], src, psf, None, multi, noise, 13, seqs[:n])
            for k in range(n):
                assert torch.equal(multi[k], single[k]), (n, noise, k)
            if noise and n > 1:
                assert not torch.equal(multi[0], multi[1])
    out9 = [torch.empty(det, device="cuda") for _ in range(9)]
    with pytest.raises(abi.ParesisError, match=r"1\.\.8 images"):
        abi.detect_counts_multi(imgs + imgs[:1], os_, det[0], det[1], src, psf, None, out9, True, 13, list(range(9)))
    with pytest.raises(ValueError):
        abi.detect_counts_multi(imgs[:3], os_, det[0], det[1], src, psf, None, out9[:2], True, 13, seqs[:3])
    with pytest.raises(ValueError):
        abi.detect_counts_multi(imgs[:3], os_, det[0], det[1], src, psf, None, out9[:3], True, 13, seqs[:4])
    # a one-tap source kernel (sigma 0.1, HS 0) is no source blur
    one_tap, _ = kernels(2.355 * 0.1, 0.0)
    assert one_tap.numel() == 1
    for noise in (False, True):
        a = counts(abi, imgs[0], os_, det, None, psf, noise=noise, seed=1, seq=2)
        b = counts(abi, imgs[0], os_, det, one_tap, psf, noise=noise, seed=1, seq=2)
        assert torch.equal(a, b)
        m = [torch.empty(det, device="cuda") for _ in range(2)]
        abi.detect_counts_multi(imgs[:2], os_, det[0], det[1], one_tap, psf, None, m, noise, 1, [2, 3])
        assert torch.equal(m[0], a)


@pytest.mark.gpu
def test_fused_kernel_above_48k_on_every_device(abi):
    """The dynamic shared-memory attribute is set per device: a fused launch above 48 KB runs on each of them."""
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs two CUDA devices")
    os_, fwhm, psf_sigma = FUSED[-1]
    assert fused_smem_bytes(os_, *half_widths(os_, fwhm, psf_sigma)) > SMEM_DEFAULT
    det = (45, 77)
    img = edge_image((det[0] * os_, det[1] * os_), seed=8)
    want = oracle(img, os_, det, fwhm, psf_sigma)
    results = []
    for d in range(n):
        with torch.cuda.device(d):
            src, psf = kernels(fwhm, psf_sigma)
            got = counts(abi, dev(img), os_, det, src, psf)
            torch.cuda.synchronize()
            results.append(got.cpu())
        assert rel_l2(results[-1].numpy(), want) < 1e-6, d
    for r in results[1:]:
        assert torch.equal(r, results[0])
