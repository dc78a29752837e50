// Membrane positions of the Fresnel model as single library calls.
//
// Reference: Experiment.computeSampleAndReferenceImages_Fresnel, Experiment.py:279-405 -- the loop over the spectrum with
// its two transmissions and three propagations per energy (four at position 0), the mean of the reference image and the
// detector call at every bin close (:378-398).  The host shim prepares the per-energy coefficients in fp64 and the
// transfer kernels once per (distance, energy, magnification); everything below is kernel launches.
//
// The reference beam's propagation sums its own |.|^2 in fp64 while it adds it to the accumulator (post_lines_kernel),
// so every energy's share of the mean is known on its own: a rank of the energy-sharded path, which sees only some of a
// bin's energies, needs exactly that.
//
// paresis_fresnel_run_positions runs the same launch sequence for many membrane positions of a scan (main.py:63-110) in
// one call, the positions dealt over slots that each own a plan, waves and accumulators and run on their own stream, so
// that consecutive positions overlap on the GPU.
#include <cuda_runtime.h>

#include <vector>

#include "common.cuh"
#include "fresnel.cuh"
#include "positions.cuh"

using namespace paresis;

namespace {

int bad(const char* who, const char* what, int e) {
    set_last_error("%s: energy %d: %s", who, e, what);
    return PARESIS_ERR_ARG;
}

// The per-energy checks of a job (host memory only).  `position_maps`: a NULL membrane map stands for the membrane of the
// position at hand (paresis_fresnel_run_positions); a NULL sample map is always an error.
int check_energies(const char* who, const paresis_fresnel_job* job, bool position_maps) {
    for (int e = 0; e < job->n_energies; ++e) {
        const paresis_fresnel_energy& en = job->energies_host[e];
        if (en.n_membrane < 1 || !en.membrane_host) return bad(who, "no membrane layer", e);
        for (int m = 0; m < en.n_membrane; ++m)
            if (!en.membrane_host[m].thickness && !position_maps) return bad(who, "null membrane map", e);
        if (en.n_sample < 1 || en.n_sample > PARESIS_MAX_LAYERS) return bad(who, "need 1 .. PARESIS_MAX_LAYERS sample layers", e);
        for (int m = 0; m < en.n_sample; ++m)
            if (!en.sample[m].thickness) return bad(who, "null sample map", e);
        if (!en.reference || !en.to_object || !en.to_detector) return bad(who, "null transfer kernel", e);
    }
    return PARESIS_OK;
}

// the plan and kernels are host structures too: a kernel prepared for another grid would read past its arrays
int check_kernels(const char* who, const paresis_fresnel_job* job, const paresis_fresnel_plan* plan) {
    for (int e = 0; e < job->n_energies; ++e) {
        const paresis_fresnel_energy& en = job->energies_host[e];
        if (!fresnel_kernel_fits(plan, en.reference) || !fresnel_kernel_fits(plan, en.to_object) ||
            !fresnel_kernel_fits(plan, en.to_detector))
            return bad(who, "a transfer kernel was prepared for a plan of another size", e);
    }
    return PARESIS_OK;
}

// every check that reads host memory only: nothing is launched before the whole job is known to be well formed
int check_job(const paresis_fresnel_job* job) {
    const char* who = "paresis_fresnel_run";
    if (!job) { set_last_error("%s: null job", who); return PARESIS_ERR_ARG; }
    if (!job->plan) { set_last_error("%s: null plan", who); return PARESIS_ERR_ARG; }
    if (!job->energies_host || job->n_energies < 1) { set_last_error("%s: no energies", who); return PARESIS_ERR_ARG; }
    if (!job->wave_a || !job->wave_b || !job->acc_sample || !job->acc_ref || (job->first_point && !job->acc_propag)) {
        set_last_error("%s: null wave or accumulator", who);
        return PARESIS_ERR_ARG;
    }
    const bool detect = job->out_sample || job->out_ref || job->out_propag || job->out_white;
    if (detect && (!job->out_sample || !job->out_ref ||
                   (job->first_point && (!job->out_propag || !job->out_white || !job->acc_white)))) {
        set_last_error("%s: incomplete detector outputs (all of them, or none to accumulate only)", who);
        return PARESIS_ERR_ARG;
    }
    if (detect && (job->oversampling < 1 || job->det_x < 1 || job->det_y < 1)) {
        set_last_error("%s: bad detector geometry", who);
        return PARESIS_ERR_ARG;
    }
    const int rc = check_energies(who, job, false);
    if (rc) return rc;
    return check_kernels(who, job, job->plan);
}

// Sample.py:279 for any number of maps, PARESIS_MAX_LAYERS at a time (transmission is multiplicative): the first group
// starts from `w_in` (NULL: the uniform amplitude), the others work in place on `w_out`.
int transmit(const paresis_c32* w_in, float amplitude, const paresis_wave_layer* layers, int n, paresis_c32* w_out, size_t pixels,
             paresis_stream stream) {
    for (int g = 0; g < n; g += PARESIS_MAX_LAYERS) {
        const int k = n - g < PARESIS_MAX_LAYERS ? n - g : PARESIS_MAX_LAYERS;
        const float* t[PARESIS_MAX_LAYERS];
        double att[PARESIS_MAX_LAYERS], ph[PARESIS_MAX_LAYERS];
        for (int m = 0; m < k; ++m) { t[m] = layers[g + m].thickness; att[m] = layers[g + m].atten; ph[m] = layers[g + m].phase; }
        const int rc = paresis_transmit_wave(g == 0 ? w_in : w_out, amplitude, t, att, ph, k, w_out, pixels, stream);
        if (rc) return rc;
    }
    return PARESIS_OK;
}

inline float2 f2(paresis_c32 c) { return make_float2(c.re, c.im); }

// the launch sequence of a checked job
int run_job(const paresis_fresnel_job* job, paresis_stream stream) {
    int rc = PARESIS_OK;
    cudaStream_t s = (cudaStream_t)stream;
    int nx = 0, ny = 0;
    fresnel_plan_dims(job->plan, &nx, &ny);
    const size_t n = (size_t)nx * ny, nd = (size_t)job->det_x * job->det_y;
    const bool detect = job->out_sample != nullptr;
    float2* wa = reinterpret_cast<float2*>(job->wave_a);
    float2* wb = reinterpret_cast<float2*>(job->wave_b);
    if (job->means) PARESIS_CUDA(cudaMemsetAsync(job->means, 0, sizeof(double) * job->n_energies, s));
    bool fresh_bin = true;
    int ibin = 0;
    double white = 0.0;
    for (int e = 0; e < job->n_energies; ++e) {
        const paresis_fresnel_energy& en = job->energies_host[e];
        if (fresh_bin) {
            PARESIS_CUDA(cudaMemsetAsync(job->acc_sample, 0, sizeof(float) * n, s));
            PARESIS_CUDA(cudaMemsetAsync(job->acc_ref, 0, sizeof(float) * n, s));
            if (job->first_point) PARESIS_CUDA(cudaMemsetAsync(job->acc_propag, 0, sizeof(float) * n, s));
            white = 0.0;
            fresh_bin = false;
        }
        // after the membrane (:338); uniform layers: attenuation folded into the amplitude, constant phase dropped
        rc = transmit(nullptr, en.amplitude_membrane, en.membrane_host, en.n_membrane, job->wave_a, n, stream);
        if (rc) return rc;
        // reference beam: membrane -> detector in one hop (:349, :354), its sum on the way
        rc = fresnel_convolve(job->plan, wa, en.reference, f2(en.phase_reference), nullptr, job->acc_ref,
                              job->means ? job->means + e : nullptr, s);
        if (rc) return rc;
        // sample beam: membrane -> object (:340-341), through the sample (:344), -> detector (:348)
        rc = fresnel_convolve(job->plan, wa, en.to_object, f2(en.phase_to_object), wb, nullptr, nullptr, s);
        if (rc) return rc;
        rc = transmit(job->wave_b, 0.f, en.sample, en.n_sample, job->wave_b, n, stream);
        if (rc) return rc;
        rc = fresnel_convolve(job->plan, wb, en.to_detector, f2(en.phase_to_detector), nullptr, job->acc_sample, nullptr, s);
        if (rc) return rc;
        if (job->first_point) {
            // the sample alone (:365-370); the white field is the incident beam itself (:372-375)
            rc = transmit(nullptr, en.amplitude_propag, en.sample, en.n_sample, job->wave_b, n, stream);
            if (rc) return rc;
            rc = fresnel_convolve(job->plan, wb, en.to_detector, f2(en.phase_to_detector), nullptr, job->acc_propag, nullptr, s);
            if (rc) return rc;
            white += en.white;
        }
        if (detect && en.close_bin) {   // :378-398, all images of the bin in one launch
            const int count = job->first_point ? 4 : 2;
            if (job->first_point) {
                rc = paresis_fill(job->acc_white, (float)white, n, stream);
                if (rc) return rc;
            }
            const uint64_t seq = job->sequence + (uint64_t)ibin * 4;
            const float* in_k[4] = {job->acc_sample, job->acc_ref, job->acc_propag, job->acc_white};
            float* out_k[4] = {job->out_sample + (size_t)ibin * nd, job->out_ref + (size_t)ibin * nd,
                               job->first_point ? job->out_propag + (size_t)ibin * nd : nullptr,
                               job->first_point ? job->out_white + (size_t)ibin * nd : nullptr};
            const uint64_t seq_k[4] = {seq, seq + 1, seq + 2, seq + 3};
            rc = paresis_detect_counts_multi(in_k, out_k, seq_k, count, nx, ny, job->oversampling, job->det_x, job->det_y,
                                             job->src_kernel, job->src_half, job->psf_kernel, job->psf_half, job->detect_work,
                                             job->noise, job->seed, stream);
            if (rc) return rc;
            ++ibin;
            fresh_bin = true;
        }
    }
    return PARESIS_OK;
}

}  // namespace

extern "C" int paresis_fresnel_run(const paresis_fresnel_job* job, paresis_stream stream) {
    const int rc = check_job(job);
    if (rc) return rc;
    return run_job(job, stream);
}

namespace {

int bad_positions(const char* fmt, int i) {
    set_last_error(fmt, i);
    return PARESIS_ERR_ARG;
}

// every argument of paresis_fresnel_run_positions, host memory only
int check_positions(const paresis_fresnel_job* job, const paresis_membrane* mem, const paresis_rt_position* positions,
                    int n_positions, const paresis_fresnel_slot* slots, int n_slots) {
    const char* who = "paresis_fresnel_run_positions";
    if (!job || !mem || !positions || !slots) {
        set_last_error("%s: null job, membrane, positions or slots", who);
        return PARESIS_ERR_ARG;
    }
    if (n_slots < 1 || n_positions < 0) {
        set_last_error("%s: need n_slots >= 1 and n_positions >= 0", who);
        return PARESIS_ERR_ARG;
    }
    if (n_positions == 0) return PARESIS_OK;       // nothing to run, nothing else to check
    if (!job->energies_host || job->n_energies < 1) { set_last_error("%s: no energies", who); return PARESIS_ERR_ARG; }
    if (!mem->field && !mem->spheres) { set_last_error("%s: the membrane has neither a sphere field nor spheres", who); return PARESIS_ERR_ARG; }
    if (job->oversampling < 1 || job->det_x < 1 || job->det_y < 1) {
        set_last_error("%s: bad detector geometry", who);
        return PARESIS_ERR_ARG;
    }
    for (int p = 0; p < n_positions; ++p) {
        const paresis_rt_position& pos = positions[p];
        if (!pos.offsets_host || !pos.thickness)
            return bad_positions("paresis_fresnel_run_positions: position %d lacks offsets or a thickness buffer", p);
        if (!pos.out_sample || !pos.out_ref || (pos.first_point && (!pos.out_propag || !pos.out_white)))
            return bad_positions("paresis_fresnel_run_positions: position %d has incomplete detector outputs", p);
        if (pos.probe_start || pos.probe_end)
            return bad_positions("paresis_fresnel_run_positions: position %d has probe events (this entry has no probe)", p);
    }
    int nx = 0, ny = 0;
    for (int k = 0; k < n_slots; ++k) {
        const paresis_fresnel_slot& sl = slots[k];
        if (!sl.plan) return bad_positions("paresis_fresnel_run_positions: slot %d has no plan", k);
        if (!sl.wave_a || !sl.wave_b || !sl.acc_sample || !sl.acc_ref || !sl.acc_propag || !sl.acc_white)
            return bad_positions("paresis_fresnel_run_positions: slot %d lacks a wave or an accumulator", k);
        for (int j = 0; j < k; ++j)
            if (slots[j].plan == sl.plan)
                return bad_positions("paresis_fresnel_run_positions: slot %d shares its plan with another slot (a plan owns its "
                                     "work buffers)", k);
    }
    int rc = check_energies(who, job, true);
    if (rc) return rc;
    for (int k = 0; k < n_slots; ++k) {
        rc = check_kernels(who, job, slots[k].plan);
        if (rc) return rc;
    }
    fresnel_plan_dims(slots[0].plan, &nx, &ny);
    if (!mem->field) {
        const size_t need = paresis_raster_work_bytes(mem->n_spheres, mem->n_layers, nx, ny);
        for (int k = 0; k < n_slots; ++k)
            if (!slots[k].raster_work || slots[k].raster_work_bytes < need)
                return bad_positions("paresis_fresnel_run_positions: slot %d: the membrane has no sphere field and the raster "
                                     "work is smaller than paresis_raster_work_bytes", k);
    }
    return PARESIS_OK;
}

}  // namespace

// Each position: its membrane map (cut from the sphere field, or rasterised), then the launch sequence of
// paresis_fresnel_run on its slot's stream with the slot's plan and buffers.  Position p goes to slot p mod n_slots.
extern "C" int paresis_fresnel_run_positions(const paresis_fresnel_job* job, const paresis_membrane* mem,
                                             const paresis_rt_position* positions, int n_positions,
                                             paresis_fresnel_slot* slots, int n_slots, paresis_stream stream) {
    int rc = check_positions(job, mem, positions, n_positions, slots, n_slots);
    if (rc) return rc;
    if (n_positions == 0) return PARESIS_OK;
    int nx = 0, ny = 0;
    fresnel_plan_dims(slots[0].plan, &nx, &ny);
    SlotEvents* events = nullptr;
    rc = slot_events(n_slots, &events);
    if (rc) return rc;
    cudaStream_t main_stream = (cudaStream_t)stream;
    const int used = n_slots < n_positions ? n_slots : n_positions;
    rc = fork_slots(*events, main_stream, slots, used);
    if (rc) return rc;

    // the template's energies with a NULL membrane map replaced by the position's: membrane layers of energy e start at
    // first[e] of `layers`
    std::vector<paresis_fresnel_energy> energies(job->energies_host, job->energies_host + job->n_energies);
    std::vector<int> first(job->n_energies);
    int n_layers = 0;
    for (int e = 0; e < job->n_energies; ++e) { first[e] = n_layers; n_layers += job->energies_host[e].n_membrane; }
    std::vector<paresis_wave_layer> layers(n_layers);
    for (int e = 0; e < job->n_energies; ++e) energies[e].membrane_host = layers.data() + first[e];
    for (int p = 0; p < n_positions; ++p) {
        const paresis_rt_position& pos = positions[p];
        const paresis_fresnel_slot& slot = slots[p % n_slots];
        rc = membrane_of_position(mem, pos.offsets_host, nx, ny, pos.thickness, slot.raster_work, slot.raster_work_bytes, slot.stream);
        if (rc) return rc;
        for (int e = 0; e < job->n_energies; ++e) {
            const paresis_fresnel_energy& src = job->energies_host[e];
            for (int m = 0; m < src.n_membrane; ++m) {
                paresis_wave_layer& dst = layers[first[e] + m];
                dst = src.membrane_host[m];
                if (!dst.thickness) dst.thickness = pos.thickness;
            }
        }
        paresis_fresnel_job j = *job;
        j.plan = slot.plan;
        j.energies_host = energies.data();
        j.first_point = pos.first_point;
        j.wave_a = slot.wave_a; j.wave_b = slot.wave_b;
        j.acc_sample = slot.acc_sample; j.acc_ref = slot.acc_ref; j.acc_propag = slot.acc_propag; j.acc_white = slot.acc_white;
        j.detect_work = slot.detect_work;
        j.means = pos.means;
        j.out_sample = pos.out_sample; j.out_ref = pos.out_ref; j.out_propag = pos.out_propag; j.out_white = pos.out_white;
        j.sequence = pos.sequence;
        rc = run_job(&j, slot.stream);
        if (rc) return rc;
    }
    return join_slots(*events, main_stream, slots, used);
}
