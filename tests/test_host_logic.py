"""CPU tests of the host-side logic and of the C-ABI surface (no kernel is launched)."""
import ctypes
import os
import re

import numpy as np
import pytest

import paresis_oracle as po
from conftest import ROOT, rel_l2


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "paresis_b200.h")).read()
    declared = set(re.findall(r"\b(paresis_[a-z0-9_]+)\s*\(", header))
    declared -= {"paresis_layer", "paresis_c32", "paresis_stream"}
    from paresis_b200 import _cabi
    assert declared == set(_cabi.EXPORTS)
    lib = ctypes.CDLL(_cabi.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), name
    assert lib.paresis_version() >= 100
    # argument validation happens before any CUDA call
    assert _cabi.lib.paresis_splat(None, None, None, None, 4, 4, 0, 2, None, None) == 2
    assert b"null pointer" in _cabi.lib.paresis_last_error()
    assert _cabi.detect_work_floats(2048, 2048, 2, 1024, 1024) == (2048 + 60) * 1054 + 1054 * 1054 + 1054 * 1024


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    import importlib
    from paresis_b200 import _cabi
    monkeypatch.setattr(_cabi, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(ImportError, match="no CPU or PyTorch fallback"):
        _cabi._load()


def test_hostmath_matches_oracle(golden):
    from paresis_b200 import hostmath as hm
    assert hm.wavenumber(25000) == po.wavenumber(25000)
    g = golden("detector")
    for k, s in enumerate(g["sigmas"]):
        ref = g["g%d" % k]
        assert np.allclose(hm.gaussian_2d(float(s)), ref, rtol=1e-14, atol=0)
        one = hm.gaussian_1d(float(s))
        assert np.allclose(np.outer(one, one), ref, rtol=1e-13, atol=1e-300)   # separability used by the kernels
        assert hm.gaussian_half_width(float(s)) == (ref.shape[0] - 1) // 2
    # Fresnel vectors reproduce the reference's shifted transfer function
    nx, ny, m, pix, z, E, M = 20, 26, 15, 2.9, 1.6, 52.0, 1.0114
    hx, hy, phase = hm.fresnel_vectors(nx, ny, m, (nx, ny), pix, z, E, M)
    k = po.wavenumber(E * 1000)
    u = (np.arange(nx + 2 * m) - (nx + 2 * m) // 2) * 2 * np.pi / (nx * pix * 1e-6)
    v = (np.arange(ny + 2 * m) - (ny + 2 * m) // 2) * 2 * np.pi / (ny * pix * 1e-6)
    kern = np.exp(-1j * z * (u[:, None] ** 2 + v[None, :] ** 2) / (2 * k * M))
    want = np.fft.ifftshift(kern) / ((nx + 2 * m) * (ny + 2 * m))
    assert np.abs(np.outer(hx, hy) - want).max() < 1e-9
    assert abs(phase - np.exp(1j * k * z / M)) < 1e-9


def test_delta_beta_tables_match_reference_values(golden):
    """The shipped export + interpolation reproduce what the reference derived from its xls."""
    from paresis_b200.hostio import tables
    g = golden("e2e_rt_poly3")
    energies = [float(r[0]) for r in g["membrane_db"]]
    cusn = tables.interpolate("CuSn", energies)
    pmma = tables.interpolate("PMMA", energies)
    for row, (d0, b0), (d1, b1) in zip(g["membrane_db"], cusn, pmma):
        assert np.allclose([d0, d1, b0, b1], row[1:], rtol=1e-12)
    assert tables.interpolate("Unobtainium", [52.0]) is None
    assert tables.interpolate("CuSn", [1.0]) == [(0, 1)]      # below the table: Sample.py:124-128


def test_image_io_round_trip(tmp_path):
    from paresis_b200.hostio import imageio
    a = np.random.default_rng(0).random((37, 53)).astype(np.float32)
    for ext, w, r in ((".tif", imageio.write_tiff, imageio.read_tiff), (".edf", imageio.write_edf, imageio.read_edf)):
        p = str(tmp_path / ("img" + ext))
        w(p, a)
        assert np.array_equal(r(p), a) and np.array_equal(imageio.open_image(p), a)
    cv2 = pytest.importorskip("cv2")
    assert np.array_equal(cv2.imread(str(tmp_path / "img.tif"), cv2.IMREAD_UNCHANGED), a)


def test_workspace_and_xml(tmp_path):
    from paresis_b200 import workspace
    from paresis_b200.hostio import xmlparams
    ws = workspace.make_workspace(str(tmp_path / "ws"), sphere_count=50)
    assert os.path.exists(os.path.join(ws, "xmlFiles", "Experiment.xml"))
    assert os.path.exists(os.path.join(ws, "Samples", "DeltaBeta", "delta_beta_tables.npz"))
    import json
    assert len(json.load(open(os.path.join(ws, "Samples", "Membranes", "CuSn.txt")))) == 50
    e = xmlparams.find_entry(os.path.join(ws, "xmlFiles", "Experiment.xml"), "experiment", "Fil_Nylon_ID17")
    assert e.get("distSourceToMembrane", float) == 140 and e.get("inVacuum") == "True" and not e.has("plateName")
    assert xmlparams.find_entry(os.path.join(ws, "xmlFiles", "Experiment.xml"), "experiment", "nope") is None
    rows = workspace.synthetic_sphere_rows(0, 60000)
    from ref_harness import synthetic_sphere_rows
    assert np.array_equal(rows, synthetic_sphere_rows(0, 60000))


def test_source_spectra(tmp_path, monkeypatch):
    from paresis_b200 import workspace
    ws = workspace.make_workspace(str(tmp_path / "ws"), sphere_count=10)
    monkeypatch.chdir(ws)
    monkeypatch.syspath_prepend(workspace.SHIM_DIR)
    import importlib
    Source = importlib.import_module("Source").Source
    s = Source(); s.myName = "id17"; s.defineCorrectValuesSource(); s.setMySpectrum()
    assert s.mySpectrum == [(52.0, 1)] and s.source_dict["myEnergySampling"] == 1
    s = Source(); s.myName = "synthetic_poly64"; s.defineCorrectValuesSource(); s.setMySpectrum()
    assert len(s.mySpectrum) == 64 and abs(sum(w for _, w in s.mySpectrum) - 1) < 1e-12
    assert s.mySpectrum[0][0] == 20.0 and s.mySpectrum[-1][0] == 83.0
    s = Source(); s.myName = "missing"
    with pytest.raises(ValueError, match="Source not found"):
        s.defineCorrectValuesSource()
    s = Source(); s.myName = "tube_W_50kVp"; s.defineCorrectValuesSource()
    with pytest.raises(ImportError, match="spekpy"):
        s.setMySpectrum()


def test_xls_spectrum_matches_reference(tmp_path, golden):
    """Source.setMySpectrum on PARESIS's Sources/W_50kVp.xls (Source.py:131-240: read the Energy / Flux columns with the
    in-repo BIFF8 reader, re-bin to myEnergySampling, keep bins above 1e-3 of the flux) against the unmodified reference."""
    import importlib
    import os
    import sys
    from paresis_b200 import workspace
    g = golden("spectrum_xls")
    ws = workspace.make_workspace(str(tmp_path / "ws"), sphere_count=10)
    old = os.getcwd()
    os.chdir(ws)
    sys.path.insert(0, workspace.SHIM_DIR)
    try:
        Source = importlib.import_module("Source").Source
        for sampling in (4.0, 2.0, 1.0):
            s = Source()
            s.myName = "xls_W_50kVp"
            s.defineCorrectValuesSource()
            assert s.spectrumFromXls and s.source_dict["myEnergySampling"] == 4.0
            s.source_dict["myEnergySampling"] = sampling
            s.setMySpectrum()
            want = g["spectrum_%g" % sampling]
            got = np.array(s.mySpectrum, dtype=float)
            assert got.shape == want.shape
            assert np.allclose(got, want, rtol=1e-12, atol=0)
            assert abs(got[:, 1].sum() - 1) < 0.05          # weights are fractions of the flux (tail bin excluded, as upstream)
    finally:
        os.chdir(old)


def test_async_writer_and_geometry_from_images(tmp_path):
    """save_image hands files to a writer thread (main.py:98-110 overlaps the next position); loadSampleGeometryFromImages
    (createSampGeom.py:263-293) reads one thickness image per material, sorted by path, .tif / .tiff / .edf."""
    import importlib
    import os
    import sys
    from paresis_b200 import workspace
    sys.path.insert(0, workspace.SHIM_DIR)
    io = importlib.import_module("InputOutput.pagailleIO")
    geom = importlib.import_module("Samples.createSampGeom")
    rng = np.random.default_rng(3)
    maps = {"b_second.tiff": rng.random((40, 56)) * 1e-3, "a_first.tif": rng.random((40, 56)) * 2e-3, "c_third.edf": rng.random((40, 56))}
    folder = tmp_path / "geom" / "nested"
    for name, arr in maps.items():
        io.save_image(arr, str(folder / name))                 # creates the folders, returns before the file is complete
    big = rng.random((1500, 1500))
    for k in range(6):
        io.save_image(big, str(tmp_path / ("big_%d.tif" % k)))
    got, params = geom.loadSampleGeometryFromImages(str(folder), 40, 56, 1.0)      # openImage waits for the writer
    assert params == {"myGeometryFolder": (str(folder), "")}
    assert len(got) == 3
    for arr, name in zip(got, ("a_first.tif", "b_second.tiff", "c_third.edf")):
        assert arr.dtype == np.float32 and np.array_equal(arr, maps[name].astype(np.float32))
    io.wait_for_writes()
    assert all(os.path.getsize(tmp_path / ("big_%d.tif" % k)) > 1500 * 1500 * 4 for k in range(6))
    with pytest.raises(Exception, match="does not exist or is incorrectly named"):
        geom.loadSampleGeometryFromImages(str(tmp_path / "nothing_here"), 40, 56, 1.0)
    # a failing write surfaces at the next hand-over
    (tmp_path / "is_a_directory.tif").mkdir()
    io.save_image(big, str(tmp_path / "is_a_directory.tif"))
    with pytest.raises(OSError):
        io.wait_for_writes()
    io.wait_for_writes()                                      # the error was delivered once; the writer keeps working
    io.save_image(big, str(tmp_path / "after.tif"))
    io.wait_for_writes()
    assert os.path.getsize(tmp_path / "after.tif") > 1500 * 1500 * 4
