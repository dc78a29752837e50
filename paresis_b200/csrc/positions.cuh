// What the run entries (paresis_rt_run, paresis_fresnel_run, paresis_df_run and their _positions forms) share: the
// detector-bin close of one position, the slot driver of the many-positions entries with the membrane map and the layer
// maps of one position, the checks of a ray-tracing job, and the argument checks of the many-positions entries.
#pragma once
#include <vector>

#include "common.cuh"

namespace paresis {

// All images of detector bin `ibin` in one launch (Experiment.py:501-521): sample and reference, at position 0 also the
// sample-only image and the white field, which is filled with `white` first.  `probe_start` / `probe_end` (both or
// neither, cudaEvent_t): recorded around the detector launch.  Job: paresis_rt_job or paresis_fresnel_job.
template <class Job>
int close_bin(const Job& job, int nx, int ny, int ibin, float white, paresis_stream stream, void* probe_start = nullptr,
              void* probe_end = nullptr) {
    const size_t n = (size_t)nx * ny, nd = (size_t)job.det_x * job.det_y;
    const int count = job.first_point ? 4 : 2;
    if (job.first_point) {
        const int rc = paresis_fill(job.acc_white, white, n, stream);
        if (rc) return rc;
    }
    const uint64_t seq = job.sequence + (uint64_t)ibin * 4;
    const float* in_k[4] = {job.acc_sample, job.acc_ref, job.acc_propag, job.acc_white};
    float* out_k[4] = {job.out_sample + (size_t)ibin * nd, job.out_ref + (size_t)ibin * nd,
                       job.first_point ? job.out_propag + (size_t)ibin * nd : nullptr,
                       job.first_point ? job.out_white + (size_t)ibin * nd : nullptr};
    const uint64_t seq_k[4] = {seq, seq + 1, seq + 2, seq + 3};
    if (probe_start) cudaEventRecord((cudaEvent_t)probe_start, (cudaStream_t)stream);
    const int rc = paresis_detect_counts_multi(in_k, out_k, seq_k, count, nx, ny, job.oversampling, job.det_x, job.det_y,
                                               job.src_kernel, job.src_half, job.psf_kernel, job.psf_half, job.detect_work,
                                               job.noise, job.seed, stream);
    if (probe_end) cudaEventRecord((cudaEvent_t)probe_end, (cudaStream_t)stream);
    return rc;
}

// fork / join events of the slot streams, created once per process and device
struct SlotEvents {
    cudaEvent_t fork = nullptr;
    std::vector<cudaEvent_t> join;
    int ensure(int n);
};

// the events of the current device, with at least n join events
int slot_events(int n, SlotEvents** out);

// The positions of a scan on the slot streams: position p runs as run(p, slots[p mod n_slots]) on that slot's stream.
// Every slot stream first waits for `stream`, and `stream` waits for every slot stream at the end.  alone(p): position p
// runs alone on the GPU -- the other slots drain first and wait for it.  n_positions >= 1.
template <class Slot, class Run, class Alone>
int run_on_slots(Slot* slots, int n_slots, int n_positions, paresis_stream stream, Run&& run, Alone&& alone) {
    SlotEvents* events = nullptr;
    int rc = slot_events(n_slots, &events);
    if (rc) return rc;
    SlotEvents& ev = *events;
    cudaStream_t main_stream = (cudaStream_t)stream;
    const int used = n_slots < n_positions ? n_slots : n_positions;
    PARESIS_CUDA(cudaEventRecord(ev.fork, main_stream));
    for (int k = 0; k < used; ++k) PARESIS_CUDA(cudaStreamWaitEvent((cudaStream_t)slots[k].stream, ev.fork, 0));
    for (int p = 0; p < n_positions; ++p) {
        Slot& slot = slots[p % n_slots];
        const bool solo = alone(p);
        if (solo) {
            for (int k = 0; k < used; ++k) {
                if (&slots[k] == &slot) continue;
                PARESIS_CUDA(cudaEventRecord(ev.join[k], (cudaStream_t)slots[k].stream));
                PARESIS_CUDA(cudaStreamWaitEvent((cudaStream_t)slot.stream, ev.join[k], 0));
            }
        }
        rc = run(p, slot);
        if (rc) return rc;
        if (solo) {
            PARESIS_CUDA(cudaEventRecord(ev.fork, (cudaStream_t)slot.stream));
            for (int k = 0; k < used; ++k)
                if (&slots[k] != &slot) PARESIS_CUDA(cudaStreamWaitEvent((cudaStream_t)slots[k].stream, ev.fork, 0));
        }
    }
    for (int k = 0; k < used; ++k) {
        PARESIS_CUDA(cudaEventRecord(ev.join[k], (cudaStream_t)slots[k].stream));
        PARESIS_CUDA(cudaStreamWaitEvent(main_stream, ev.join[k], 0));
    }
    return PARESIS_OK;
}

// ... with every position running alongside the others
template <class Slot, class Run>
int run_on_slots(Slot* slots, int n_slots, int n_positions, paresis_stream stream, Run&& run) {
    return run_on_slots(slots, n_slots, n_positions, stream, run, [](int) { return false; });
}

// The membrane map of the position at `offsets_host` into thickness[nx][ny]: cut from the sphere field
// (paresis_membrane_from_field), or rasterised (paresis_raster_spheres, with `raster_work`) when the membrane has none.
int membrane_of_position(const paresis_membrane* mem, const int64_t* offsets_host, int nx, int ny, float* thickness,
                         void* raster_work, size_t raster_work_bytes, paresis_stream stream);

// The fields of a job that come from the position: first_point, means, detector outputs and sequence.
template <class Job>
void bind_position(Job& j, const paresis_rt_position& pos) {
    j.first_point = pos.first_point;
    j.means = pos.means;
    j.out_sample = pos.out_sample; j.out_ref = pos.out_ref; j.out_propag = pos.out_propag; j.out_white = pos.out_white;
    j.sequence = pos.sequence;
}

// out[e] = energies[e] for e < n_energies, except that a NULL hop1 / hop2 map stands for `thickness`, the membrane map
// of the position at hand.  Only the layers below n_hop1 / n_hop2 are read or written.
void bind_position_maps(const paresis_rt_energy* energies, int n_energies, const float* thickness, paresis_rt_energy* out);

// The argument checks of the run entries (host memory only); `who` prefixes the message.
// A ray-tracing job (paresis_rt_run, paresis_df_run's job->rt): energies and a frame of at least 3 x 3 ...
int check_rt_frame(const char* who, const paresis_rt_job& r);
// ... and everything of a single-position job: the frame, i_bs and the accumulators, the detector outputs (all of them,
// or none to accumulate only), acc_white and the detector geometry with outputs, and the energies (check_rt_energies):
int check_rt_job(const char* who, const paresis_rt_job& r);
// per energy, 1 .. PARESIS_MAX_LAYERS layers in each hop (the sample-only hop when `first`) and no NULL map; with
// `position_maps`, a NULL hop1 / hop2 map stands for the position's membrane map (a NULL propag map never does):
int check_rt_energies(const char* who, const paresis_rt_job& r, bool first, bool position_maps);
// The pointers and counts of a many-positions call:
int check_call(const char* who, const void* job, const paresis_membrane* mem, const void* positions, const void* slots,
               int n_positions, int n_slots);
// the membrane has a sphere field or spheres, and the detector geometry:
int check_membrane_detector(const char* who, const paresis_membrane* mem, int oversampling, int det_x, int det_y);
// position p has offsets, a thickness buffer and all its detector outputs:
int check_position(const char* who, const paresis_rt_position& pos, int p);
// position p has no probe events (an entry that records none):
int check_no_probe(const char* who, const paresis_rt_position& pos, int p);
// Slots run concurrently, so no image may belong to two of them.  images(slot): a std::array of the slot's image
// pointers, NULL for none.
template <class Slot, class Images>
int check_slots_apart(const char* who, const Slot* slots, int n_slots, Images&& images) {
    for (int k = 1; k < n_slots; ++k) {
        const auto mine = images(slots[k]);
        for (int j = 0; j < k; ++j) {
            const auto theirs = images(slots[j]);
            for (const void* a : mine)
                for (const void* b : theirs)
                    if (a && a == b) {
                        set_last_error("%s: slot %d shares an image buffer with another slot (slots run concurrently)", who, k);
                        return PARESIS_ERR_ARG;
                    }
        }
    }
    return PARESIS_OK;
}
// without a sphere field, every slot has raster work of at least paresis_raster_work_bytes:
template <class Slot>
int check_raster_work(const char* who, const paresis_membrane* mem, int nx, int ny, const Slot* slots, int n_slots) {
    if (mem->field) return PARESIS_OK;
    const size_t need = paresis_raster_work_bytes(mem->n_spheres, mem->n_layers, nx, ny);
    for (int k = 0; k < n_slots; ++k)
        if (!slots[k].raster_work || slots[k].raster_work_bytes < need) {
            set_last_error("%s: slot %d: the membrane has no sphere field and the raster work is smaller than "
                           "paresis_raster_work_bytes", who, k);
            return PARESIS_ERR_ARG;
        }
    return PARESIS_OK;
}

}  // namespace paresis
