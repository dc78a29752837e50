"""Projected-thickness maps generated and kept on the GPU.

Host logic of Samples/getMembraneFromFile.py:60-171 and Samples/createSampGeom.py:15-107
(file parsing, rescaling, stitching, the ``np.random.randint`` draws in the reference's
order); the per-pixel work is in csrc/geometry.cu.
"""
import json
import os

import numpy as np
import torch

from . import _cabi as abi
from . import transfer
from .host_api import device


class DeviceGeometry:
    """Per-material thickness maps (metres) in HBM; uniform layers are kept as scalars.

    Quacks like the ``[n_mat, N, N]`` ndarray PARESIS stores in ``Sample.myGeometry`` for the
    accesses it makes: ``len``, ``.ndim``, ``.shape``, ``geom[m]`` (float32 host copy of one
    map, what main.py:99 saves) and ``np.asarray(geom)`` (float64 stack)."""

    ndim = 3

    def __init__(self, entries, shape):
        self.entries = list(entries)          # torch.Tensor [N, N] float32 | float (uniform thickness)
        self.map_shape = (int(shape[0]), int(shape[1]))
        self._pending = {}
        self._host = {}
        self._full = {}       # materialised uniform entries: the same tensor every call (engine.mixed_sample keys on it)

    def prefetch(self, m=0):
        """Start copying map ``m`` to pinned host memory; overlaps whatever the GPU does next."""
        if m not in self._host and m not in self._pending and isinstance(self.entries[m], torch.Tensor):
            self._pending[m] = transfer.Pending(self.entries[m])

    @property
    def shape(self):
        return (len(self.entries),) + self.map_shape

    def __len__(self):
        return len(self.entries)

    def __getitem__(self, m):
        e = self.entries[m]
        if not isinstance(e, torch.Tensor):
            return np.full(self.map_shape, e, dtype=np.float32)
        if m not in self._host:
            self.prefetch(m)
            self._host[m] = self._pending.pop(m).wait()
        return self._host[m]

    def __array__(self, dtype=None, copy=None):
        stack = np.stack([np.asarray(self[m], dtype=np.float64) for m in range(len(self.entries))])
        return stack.astype(dtype) if dtype is not None else stack

    def device_entries(self, materialise=False):
        out = []
        for m, e in enumerate(self.entries):
            if materialise and not isinstance(e, torch.Tensor):
                key = (m, str(device()))
                if key not in self._full:
                    self._full[key] = torch.full(self.map_shape, float(e), device=device(), dtype=torch.float32)
                e = self._full[key]
            out.append(e)
        return out


def from_host(array):
    """Upload a user-supplied [n_mat, N, N] array; flat maps become uniform scalars."""
    arr = np.asarray(array)
    if arr.ndim != 3:
        raise Exception("Sample Geometry has the wrong nb of dim [material, x, y]")   # Sample.py:264
    entries = []
    for m in range(arr.shape[0]):
        lo, hi = float(arr[m].min()), float(arr[m].max())
        if lo == hi:
            entries.append(lo)
        else:
            entries.append(transfer.upload(arr[m], torch.float32, device()))
    return DeviceGeometry(entries, arr.shape[1:])


# ---------------------------------------------------------------------------- membrane
_MEMBRANE_FILE = "Samples/Membranes/CuSn.txt"
_host_tables = {}     # parsed + rescaled + tiled sphere lists, keyed by file identity and geometry
_device_tables = {}   # their device copies
_device_fields = {}   # sphere fields rasterised from them (paresis_raster_field)
FIELD_BYTES_LIMIT = 16 << 30   # beyond this the membrane is rasterised per position instead


def drop_device_tables():
    """Forget the device copies (the next position uploads the sphere list again)."""
    global _speculated
    _speculated = None
    _device_tables.clear()
    _device_fields.clear()


def _sphere_table(path, mean_radius, dim_x, dim_y, pix):
    """getMembraneFromFile.py:84-124: load, rescale to the wanted mean radius, move the origin to
    the top-left corner, tile along x then y until the list covers the field of view.
    The reference re-reads the file at every membrane position; here the parsed list is cached on
    the host (keyed by the file's identity) and on the device."""
    st = os.stat(path)
    key = (os.path.abspath(path), st.st_mtime_ns, st.st_size, mean_radius, dim_x, dim_y, pix)
    if key not in _host_tables:
        if path.split('/')[-1] != 'CuSn.txt':
            raise Exception("Enter segmented membrane size ")                           # :90
        corr = mean_radius / 12.8
        ext_x = int(np.floor(8102)) * corr + mean_radius
        ext_y = int(np.floor(9740)) * corr + mean_radius
        with open(path) as fh:
            tab = np.asarray(json.load(fh), dtype=np.float64) * corr
        tab[:, 1] += ext_x / 2
        tab[:, 0] += ext_y / 2
        base, step = tab.copy(), ext_x
        while ext_x / pix - dim_x < 0:
            print("segmented membrane too small: proceeding with stitching along x")
            shifted = base.copy()
            shifted[:, 1] += ext_x
            tab = np.concatenate((tab, shifted), axis=0)
            ext_x += step
        base, step = tab.copy(), ext_y
        while ext_y / pix - dim_y < 0:
            print("segmented membrane too small: proceeding with stitching along y")
            shifted = base.copy()
            shifted[:, 0] += ext_y
            tab = np.concatenate((tab, shifted), axis=0)
            ext_y += step
        _host_tables.clear()
        _device_tables.clear()
        _device_fields.clear()
        _host_tables[key] = (np.ascontiguousarray(tab), ext_x, ext_y)
    tab, ext_x, ext_y = _host_tables[key]
    dkey = key + (torch.cuda.current_device(),)
    if dkey not in _device_tables:
        _device_tables[dkey] = transfer.upload(tab, torch.float64, device())
    return _device_tables[dkey], ext_x, ext_y


class MembranePlan:
    """Everything about a segmented membrane that does not change from one position to the next
    (getMembraneFromFile.py:84-124, :130-133): the device sphere table and the draw ranges."""

    def __init__(self, sample, dim_x, dim_y, pix):
        self.dim_x, self.dim_y, self.pix = int(dim_x), int(dim_y), float(pix)
        self.layers = int(sample.myNbOfLayers)
        self.margin = int(np.ceil(10 * sample.myMeanSphereRadius / pix))
        self.margin2 = int(np.floor(self.margin / 2))
        self.table, self.ext_x, self.ext_y = _sphere_table(_MEMBRANE_FILE, sample.myMeanSphereRadius, self.dim_x, self.dim_y, pix)
        self._field_key = (self.table.data_ptr(), self.pix, self.margin, torch.cuda.current_device())

    def field(self):
        """The sphere field of this membrane (device tensor), or None when positions must be rasterised one by
        one: a grain reaching further than margin/2 pixels would be clipped by the reference's acceptance window
        (getMembraneFromFile.py:151), which a shifted window of the field cannot reproduce."""
        if self._field_key not in _device_fields:
            fx = int(np.ceil(self.ext_x / self.pix)) + self.margin + 1
            fy = int(np.ceil(self.ext_y / self.pix)) + self.margin + 1
            reach = int(np.floor(float(self.table[:, 2].max().item()) / self.pix)) + 1 if self.table.shape[0] else 0
            if reach > self.margin2 or fx * fy * 4 > FIELD_BYTES_LIMIT:
                _device_fields[self._field_key] = None
            else:
                field = torch.empty((fx, fy), device=self.table.device, dtype=torch.float32)
                abi.raster_field(self.table, self.pix, field)
                _device_fields[self._field_key] = field
        return _device_fields[self._field_key]

    def draw_offsets(self):
        """Two ``np.random.randint`` draws per layer, x first, from numpy's global stream (:139-140), so
        ``np.random.seed`` reproduces the reference's membrane positions."""
        offsets = []
        for _ in range(self.layers):
            ox = np.random.randint(self.margin2, self.ext_x / self.pix - self.dim_x - self.margin2)
            oy = np.random.randint(self.margin2, self.ext_y / self.pix - self.dim_y - self.margin2)
            offsets.append((int(ox), int(oy)))
        return offsets


_plans = {}


def _plan(sample, dim_x, dim_y, pix):
    """MembranePlan of this membrane, rebuilt when the sphere file or the geometry changes."""
    st = os.stat(_MEMBRANE_FILE)
    key = (sample.myMeanSphereRadius, sample.myNbOfLayers, int(dim_x), int(dim_y), float(pix), st.st_mtime_ns, st.st_size,
           torch.cuda.current_device())
    plan = _plans.get(key)
    if plan is None or plan._field_key[0] != plan.table.data_ptr() or not _device_tables:
        _plans.clear()
        plan = _plans[key] = MembranePlan(sample, dim_x, dim_y, pix)
    return plan


_speculated = None     # the next position's map, cut ahead of time: dict(plan, offsets, geom)


def _cut_membrane(plan, offsets, pix, grains):
    field = plan.field()
    if field is not None:
        abi.membrane_from_field(field, offsets, plan.margin, plan.dim_x, plan.dim_y, grains)
    else:
        abi.raster_spheres(plan.table, pix, offsets, plan.dim_x, plan.dim_y, plan.margin, grains)


def speculate_next_membrane(sample, dim_x, dim_y, pix, support_um):
    """Cut the membrane map the NEXT getMembraneSegmentedFromFile call will ask for, and start its copy to the host, now.

    The per-position flow of main.py (:63-110) is strictly serial: the next position's map is only requested once this
    position's images are on the host, so the device->host link idles through the host's turn-around and the cut
    kernel.  The next offsets are the next ``np.random.randint`` draws (getMembraneFromFile.py:139-140): they are drawn
    here from a COPY of numpy's global state (the caller's stream is left untouched); when the real call draws the
    same numbers -- nobody re-seeded or drew in between -- the map and its copy are already under way; otherwise the
    speculation is dropped and the map is cut as usual.  Results are identical either way."""
    global _speculated
    plan = _plan(sample, dim_x, dim_y, pix)
    state = np.random.get_state()
    offsets = plan.draw_offsets()
    np.random.set_state(state)
    grains = torch.empty((plan.dim_x, plan.dim_y), device=device(), dtype=torch.float32)
    _cut_membrane(plan, offsets, pix, grains)
    geom = DeviceGeometry([grains, support_um * 1e-6], (plan.dim_x, plan.dim_y))
    geom.prefetch(0)
    _speculated = dict(plan=plan, offsets=offsets, geom=geom, support=support_um)


def membrane_segmented(sample, dim_x, dim_y, pix, point_num, support_um, out=None, prefetch=False):
    """getMembraneSegmentedFromFile (Samples/getMembraneFromFile.py:60-171)."""
    global _speculated
    plan = _plan(sample, dim_x, dim_y, pix)
    offsets = plan.draw_offsets()
    dim_x, dim_y = plan.dim_x, plan.dim_y
    params = {'Average sphere radius': (sample.myMeanSphereRadius, 'um'),
              'Number of layers': (sample.myNbOfLayers, ''),
              'Support total thickness': (support_um, 'um')}
    ahead, _speculated = _speculated, None
    if (ahead is not None and out is None and prefetch and ahead["plan"] is plan and ahead["offsets"] == offsets
            and ahead["support"] == support_um):
        return ahead["geom"], params
    grains = out if out is not None else torch.empty((dim_x, dim_y), device=device(), dtype=torch.float32)
    _cut_membrane(plan, offsets, pix, grains)
    geom = DeviceGeometry([grains, support_um * 1e-6], (dim_x, dim_y))
    if prefetch:
        geom.prefetch(0)      # main.py:99 saves this map: start the copy now, it overlaps the image formation
    return geom, params


# ---------------------------------------------------------------------------- samples
def sample_sphere(radius_um, dim_x, dim_y, pix):
    """CreateSampleSphere arithmetic (createSampGeom.py:41-53)."""
    out = torch.empty((int(dim_x), int(dim_y)), device=device(), dtype=torch.float32)
    abi.sphere_map(radius_um, int(dim_x), int(dim_y), pix, out)
    return DeviceGeometry([out], (dim_x, dim_y))


def sample_cylinder(radius_um, orientation_deg, dim_x, dim_y, pix):
    """CreateSampleCylindre arithmetic (createSampGeom.py:87-106), rotation included."""
    if 2 * radius_um / pix > 2 * dim_x or 2 * radius_um / pix > 2 * dim_y:
        raise Exception('The sample is too big for the detector field of view (increase dimX, dimY)')
    out = torch.empty((int(dim_x), int(dim_y)), device=device(), dtype=torch.float32)
    abi.cylinder_map(radius_um, orientation_deg, int(dim_x), int(dim_y), pix, out)
    return DeviceGeometry([out], (dim_x, dim_y))


def sample_two_spheres(kind, dim_x, dim_y, pix):
    """CreateSampleSpheresInCylinder (kind 0) / CreateSampleSpheresInParallelepiped (kind 1), createSampGeom.py:110-260."""
    out = torch.empty((3, int(dim_x), int(dim_y)), device=device(), dtype=torch.float32)
    try:
        abi.two_sphere_phantom(kind, int(dim_x), int(dim_y), pix, out)
    except abi.ParesisError as exc:
        if "too big" in str(exc):
            raise Exception('The sample is too big for the detector field of view (increase dimX, dimY)')
        raise
    return DeviceGeometry([out[0], out[1], out[2]], (dim_x, dim_y))
