// Shared parts of the run entries (positions.cuh).
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

int bad(const char* fmt, const char* who, int i = 0) {
    set_last_error(fmt, who, i);
    return PARESIS_ERR_ARG;
}
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

void bind_position_maps(const paresis_rt_energy* energies, int n_energies, const float* thickness, paresis_rt_energy* out) {
    auto bind = [&](const paresis_layer* src, int n, paresis_layer* dst) {
        for (int m = 0; m < n && m < PARESIS_MAX_LAYERS; ++m) dst[m].thickness = src[m].thickness ? src[m].thickness : thickness;
    };
    for (int e = 0; e < n_energies; ++e) {
        const paresis_rt_energy& src = energies[e];
        bind(src.hop1, src.n_hop1, out[e].hop1);
        bind(src.hop2, src.n_hop2, out[e].hop2);
    }
}

int check_rt_frame(const char* who, const paresis_rt_job& r) {
    if (!r.energies_host || r.n_energies < 1) return bad("%s: no energies", who);
    if (r.nx < 3 || r.ny < 3) {
        set_last_error("%s: bad frame %d x %d", who, r.nx, r.ny);
        return PARESIS_ERR_ARG;
    }
    return PARESIS_OK;
}

int check_rt_job(const char* who, const paresis_rt_job& r) {
    const int rc = check_rt_frame(who, r);
    if (rc) return rc;
    if (!r.i_bs || !r.acc_sample || !r.acc_ref || (r.first_point && !r.acc_propag))
        return bad("%s: null object-plane buffer or accumulator", who);
    const bool detect = r.out_sample || r.out_ref || r.out_propag || r.out_white;
    if (detect && (!r.out_sample || !r.out_ref || (r.first_point && (!r.out_propag || !r.out_white || !r.acc_white))))
        return bad("%s: incomplete detector outputs (all of them, or none to accumulate only)", who);
    if (detect && (r.oversampling < 1 || r.det_x < 1 || r.det_y < 1)) return bad("%s: bad detector geometry", who);
    return check_rt_energies(who, r, r.first_point != 0, false);
}

int check_rt_energies(const char* who, const paresis_rt_job& r, bool first, bool position_maps) {
    auto bad_energy = [&](const char* what, int e) {
        set_last_error("%s: energy %d: %s", who, e, what);
        return PARESIS_ERR_ARG;
    };
    for (int e = 0; e < r.n_energies; ++e) {
        const paresis_rt_energy& en = r.energies_host[e];
        if (en.n_hop1 < 1 || en.n_hop1 > PARESIS_MAX_LAYERS) return bad_energy("need 1 .. PARESIS_MAX_LAYERS membrane maps", e);
        if (en.n_hop2 < 1 || en.n_hop2 > PARESIS_MAX_LAYERS)
            return bad_energy("need 1 .. PARESIS_MAX_LAYERS membrane + sample maps in the object hop (mix the sample's maps)", e);
        if (first && (en.n_propag < 1 || en.n_propag > PARESIS_MAX_LAYERS))
            return bad_energy("need 1 .. PARESIS_MAX_LAYERS sample maps in the sample-only hop", e);
        for (int m = 0; m < en.n_hop1; ++m) if (!en.hop1[m].thickness && !position_maps) return bad_energy("null membrane map", e);
        for (int m = 0; m < en.n_hop2; ++m) if (!en.hop2[m].thickness && !position_maps) return bad_energy("null object-hop map", e);
        if (first)
            for (int m = 0; m < en.n_propag; ++m) if (!en.propag[m].thickness) return bad_energy("null sample map", e);
    }
    return PARESIS_OK;
}

int check_call(const char* who, const void* job, const paresis_membrane* mem, const void* positions, const void* slots,
               int n_positions, int n_slots) {
    if (!job || !mem || !positions || !slots) return bad("%s: null job, membrane, positions or slots", who);
    if (n_slots < 1 || n_positions < 0) return bad("%s: need n_slots >= 1 and n_positions >= 0", who);
    return PARESIS_OK;
}

int check_membrane_detector(const char* who, const paresis_membrane* mem, int oversampling, int det_x, int det_y) {
    if (!mem->field && !mem->spheres) return bad("%s: the membrane has neither a sphere field nor spheres", who);
    if (oversampling < 1 || det_x < 1 || det_y < 1) return bad("%s: bad detector geometry", who);
    return PARESIS_OK;
}

int check_position(const char* who, const paresis_rt_position& pos, int p) {
    if (!pos.offsets_host || !pos.thickness) return bad("%s: position %d lacks offsets or a thickness buffer", who, p);
    if (!pos.out_sample || !pos.out_ref || (pos.first_point && (!pos.out_propag || !pos.out_white)))
        return bad("%s: position %d has incomplete detector outputs", who, p);
    return PARESIS_OK;
}

int check_no_probe(const char* who, const paresis_rt_position& pos, int p) {
    if (pos.probe_start || pos.probe_end) return bad("%s: position %d has probe events (this entry has no probe)", who, p);
    return PARESIS_OK;
}

}  // namespace paresis
