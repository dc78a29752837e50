// Shared parts of the many-positions entries (positions.cuh).
#include "positions.cuh"

namespace paresis {

int SlotEvents::ensure(int n) {
    if (!fork) PARESIS_CUDA(cudaEventCreateWithFlags(&fork, cudaEventDisableTiming));
    while ((int)join.size() < n) {
        cudaEvent_t e;
        PARESIS_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        join.push_back(e);
    }
    return PARESIS_OK;
}

namespace {
SlotEvents g_events_of[32];     // CUDA events belong to a device
}  // namespace

int slot_events(int n, SlotEvents** out) {
    int dev = 0;
    PARESIS_CUDA(cudaGetDevice(&dev));
    SlotEvents& ev = g_events_of[(dev < 0 || dev >= 32) ? 0 : dev];
    const int rc = ev.ensure(n);
    if (rc) return rc;
    *out = &ev;
    return PARESIS_OK;
}

int membrane_of_position(const paresis_membrane* mem, const int64_t* offsets_host, int nx, int ny, float* thickness,
                         void* raster_work, size_t raster_work_bytes, paresis_stream stream) {
    if (mem->field)
        return paresis_membrane_from_field(mem->field, mem->field_x, mem->field_y, offsets_host, mem->n_layers, mem->margin, nx,
                                           ny, thickness, stream);
    return paresis_raster_spheres(mem->spheres, mem->n_spheres, mem->pix_um, offsets_host, mem->n_layers, nx, ny, mem->margin,
                                  thickness, raster_work, raster_work_bytes, stream);
}

}  // namespace paresis
