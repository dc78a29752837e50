// What the many-positions entries (paresis_rt_run_positions, paresis_fresnel_run_positions, paresis_df_run_positions)
// share: the fork / join of their slot streams and the membrane map of one position.
#pragma once
#include <vector>

#include "common.cuh"

namespace paresis {

// fork / join events of the slot streams, created once per process and device
struct SlotEvents {
    cudaEvent_t fork = nullptr;
    std::vector<cudaEvent_t> join;
    int ensure(int n);
};

// the events of the current device, with at least n join events
int slot_events(int n, SlotEvents** out);

// every slot stream of slots[0 .. used) waits for `main`
template <class Slot>
int fork_slots(SlotEvents& ev, cudaStream_t main, const Slot* slots, int used) {
    PARESIS_CUDA(cudaEventRecord(ev.fork, main));
    for (int k = 0; k < used; ++k) PARESIS_CUDA(cudaStreamWaitEvent((cudaStream_t)slots[k].stream, ev.fork, 0));
    return PARESIS_OK;
}

// `main` waits for every slot stream of slots[0 .. used)
template <class Slot>
int join_slots(SlotEvents& ev, cudaStream_t main, const Slot* slots, int used) {
    for (int k = 0; k < used; ++k) {
        PARESIS_CUDA(cudaEventRecord(ev.join[k], (cudaStream_t)slots[k].stream));
        PARESIS_CUDA(cudaStreamWaitEvent(main, ev.join[k], 0));
    }
    return PARESIS_OK;
}

// The membrane map of the position at `offsets_host` into thickness[nx][ny]: cut from the sphere field
// (paresis_membrane_from_field), or rasterised (paresis_raster_spheres, with `raster_work`) when the membrane has none.
int membrane_of_position(const paresis_membrane* mem, const int64_t* offsets_host, int nx, int ny, float* thickness,
                         void* raster_work, size_t raster_work_bytes, paresis_stream stream);

}  // namespace paresis
