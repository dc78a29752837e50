"""Sharding the (energy x membrane position) units of a simulation over GPUs.

Positions are independent (each has its own membrane map and output files, main.py:63-110):
``positions_of`` just deals them out, no communication.  Energies of one detector bin share an
accumulator (Experiment.py:482-483): each rank forms its partial sums, applies the LINEAR part
of the detector (blur + bin-down, noise off) and the ranks add those detector-resolution images
with one NCCL reduction per bin; the Poisson draw follows the sum, on the owner rank, with the
same counter-based stream a single GPU would use, so the shard layout does not change the
statistics.  One process per GPU, ``torch.distributed`` (NCCL over NVLink; gloo for CPU tests).
"""
import numpy as np
import torch
import torch.distributed as dist

from . import _cabi as abi
from .engine import IMAGES


def positions_of(n_positions, rank, world):
    """Round-robin membrane positions of a rank (rank 0 gets position 0 and its extra images)."""
    return list(range(rank, n_positions, world))


def energies_of(indices, rank, world):
    """Round-robin share of one detector bin's spectrum indices."""
    return list(indices[rank::world])


def reduce_images(stack, owner=0, group=None):
    """Sum per-rank partial images onto ``owner`` (in place).  ``stack`` is any float tensor."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        # `owner` is a rank OF THE GROUP; dist.reduce wants the global rank
        dst = dist.get_global_rank(group, owner) if group is not None else owner
        dist.reduce(stack, dst=dst, op=dist.ReduceOp.SUM, group=group)
    return stack


def combine_means(values, indices, n_total, group=None):
    """Per-energy reference means computed by different ranks -> one vector on every rank."""
    full = torch.zeros(n_total, dtype=torch.float64, device=values.device)
    if len(indices):
        full[torch.as_tensor(list(indices), device=values.device)] = values
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(full, op=dist.ReduceOp.SUM, group=group)
    return full


class ShardedPosition:
    """What ``compute_rt_energy_sharded(..., defer=True)`` and ``compute_fresnel_energy_sharded(..., defer=True)`` return on
    every rank: the device work of the position is queued, its host-side tail is not done yet.  ``finish()`` waits for the per-energy means and the status flags (one
    all_reduce, already queued), raises ``InsaneValues`` on every rank if any rank saw a non-finite value, and returns what
    the immediate call returns (the result dict on the owner, None elsewhere).  The images must not be used before it."""

    def __init__(self, out, tail_host, ready, work, spectrum, is_owner):
        self._out, self._tail, self._ready, self._work = out, tail_host, ready, work
        self._spectrum, self._is_owner, self._done = spectrum, is_owner, False

    def finish(self):
        if not self._done:
            self._ready.synchronize()
            self._done = True
            tail = self._tail.numpy()
            if tail[-1] != 0:
                from .engine import InsaneValues
                raise InsaneValues("The calculated intensity refractive includes some nans or insane values")
            if self._is_owner:
                m = tail[:-1]
                energies = np.array([e for e, _ in self._spectrum])
                self._out["mean_energy"] = (float(np.dot(m, energies)), float(m.sum()))
        return self._out if self._is_owner else None


def compute_rt_energy_sharded(engine, scene, point_num, owner=0, group=None, sequence_base=0, reduce_events=None, defer=False):
    """One membrane position with the spectrum spread over the ranks of ``group``.

    Every rank calls this with the same scene.  Returns, on ``owner``, the dict that
    ``ImageFormation.compute_rt`` returns (device tensors + mean_energy); None elsewhere.
    ``reduce_events``: a list that receives one (start, end) CUDA event pair per NCCL reduction (bench.py).
    ``defer=True``: return a ``ShardedPosition`` instead, without waiting for the device: the caller queues the next
    position first and calls ``finish()`` on this one afterwards (every rank, same order), so the host's turn-around and
    the device->host read of the means overlap the next position's kernels.
    A scattering sample at position 0 also gives ``dark_field`` on the owner: each rank adds its energies' share and
    the shares are summed with one more reduction."""
    def white(energy, flux):   # Experiment.py:490-497
        return scene.mean_shot_count / scene.os ** 2 * flux * scene.common_factor(energy) * scene.plate_factor(energy)
    dark = None
    if point_num == 0 and engine.scatters(scene):
        dark = torch.zeros((engine.nx, engine.ny), device=engine.device, dtype=torch.float32)

    def accumulate(sc, point, indices):
        return engine.accumulate_rt(sc, point, indices, dark_field=dark)
    return _energy_sharded(accumulate, white, engine, scene, point_num, owner, group, sequence_base, reduce_events,
                           defer, dark)


def compute_fresnel_energy_sharded(engine, scene, point_num, owner=0, group=None, sequence_base=0, reduce_events=None,
                                   defer=False):
    """The Fresnel model (``ImageFormation.compute_fresnel``) with the spectrum spread over the ranks of ``group``: same
    arguments and results as ``compute_rt_energy_sharded``."""
    def white(energy, flux):   # Experiment.py:372-375
        return engine.fresnel_amplitude(scene, energy, flux) ** 2
    return _energy_sharded(engine.accumulate_fresnel, white, engine, scene, point_num, owner, group, sequence_base,
                           reduce_events, defer)


def _energy_sharded(accumulate, white_of, engine, scene, point_num, owner, group, sequence_base, reduce_events, defer,
                    dark_field=None):
    """Body of the energy-sharded calls.  ``accumulate(scene, point_num, indices)``: the model's partial sums of some
    energies of one bin into ``engine.acc``, returning their per-energy reference means; ``white_of(energy, flux)``: one
    energy's share of the white field.  ``dark_field``: this rank's share of the dark-field map, which ``accumulate``
    adds to; it is summed onto the owner and returned there."""
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    first = point_num == 0
    bins = engine.bins(scene)[:len(scene.thresholds)]
    n_e = len(scene.spectrum)
    count = 4 if first else 2
    out = engine._new_outputs(len(bins), first) if rank == owner else None
    means = torch.zeros(n_e, dtype=torch.float64, device=engine.device)
    fwhm = scene.effective_source_fwhm()
    src = engine._gauss(fwhm / 2.355) if fwhm != 0 else None
    psf = engine._gauss(scene.psf_sigma) if scene.psf_sigma != 0 else None
    partial = torch.zeros((count, engine.det_x, engine.det_y), device=engine.device, dtype=torch.float32)
    for b, indices in enumerate(bins):
        mine = energies_of(indices, rank, world)
        partial.zero_()
        if mine:
            means[torch.as_tensor(mine, device=engine.device)] = accumulate(scene, point_num, mine)
            if first:   # the white field is the incident beam itself: fill it with this rank's share
                abi.fill(engine.acc["white"], sum(white_of(*scene.spectrum[i]) for i in mine))
            for k, name in enumerate(IMAGES[:count]):
                # the linear part of the detector before the exchange: detector-resolution images travel
                abi.detect_counts(engine.acc[name], engine.os, engine.det_x, engine.det_y, src, psf, engine.work,
                                  partial[k], False)
        if reduce_events is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            reduce_images(partial, owner, group)
            e1.record()
            reduce_events.append((e0, e1))
        else:
            reduce_images(partial, owner, group)
        if rank == owner:
            seq = engine.sequence(point_num, sequence_base) + 4 * b
            for k, name in enumerate(IMAGES[:count]):
                if engine.poisson:
                    abi.poisson(partial[k], out[name][b], engine.seed, seq + k)
                else:
                    out[name][b].copy_(partial[k])
    if dark_field is not None:
        reduce_images(dark_field, owner, group)
        if rank == owner:
            out["dark_field"] = dark_field
    # the reference's NaN / "insane values" guard (refractionFileNumba2.py:81-82) must fire whichever rank saw the bad
    # value: the status flags travel with the means (one all_reduce), every rank clears its own and every rank raises
    tail = torch.cat((means, engine.flag.to(torch.float64)))
    engine.flag.zero_()
    if defer:
        work = dist.all_reduce(tail, op=dist.ReduceOp.SUM, group=group, async_op=True) if world > 1 else None
        if work is not None:
            work.wait()                         # orders the copy below after the collective on this stream; the host goes on
        host = torch.empty(tail.shape, dtype=tail.dtype, pin_memory=True)
        host.copy_(tail, non_blocking=True)
        ready = torch.cuda.Event()
        ready.record()
        return ShardedPosition(out, host, ready, work, scene.spectrum, rank == owner)
    if world > 1:
        dist.all_reduce(tail, op=dist.ReduceOp.SUM, group=group)
    tail = tail.cpu().numpy()
    if tail[-1] != 0:
        from .engine import InsaneValues
        raise InsaneValues("The calculated intensity refractive includes some nans or insane values")
    if rank != owner:
        return None
    m = tail[:-1]
    energies = np.array([e for e, _ in scene.spectrum])
    out["mean_energy"] = (float(np.dot(m, energies)), float(m.sum()))
    return out
