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
#include <cuda_runtime.h>

#include "common.cuh"
#include "fresnel.cuh"

using namespace paresis;

namespace {

int bad(const char* what, int e) {
    set_last_error("paresis_fresnel_run: energy %d: %s", e, what);
    return PARESIS_ERR_ARG;
}

// every check that reads host memory only: nothing is launched before the whole job is known to be well formed
int check_job(const paresis_fresnel_job* job) {
    if (!job) { set_last_error("paresis_fresnel_run: null job"); return PARESIS_ERR_ARG; }
    if (!job->plan) { set_last_error("paresis_fresnel_run: null plan"); return PARESIS_ERR_ARG; }
    if (!job->energies_host || job->n_energies < 1) { set_last_error("paresis_fresnel_run: no energies"); return PARESIS_ERR_ARG; }
    if (!job->wave_a || !job->wave_b || !job->acc_sample || !job->acc_ref || (job->first_point && !job->acc_propag)) {
        set_last_error("paresis_fresnel_run: null wave or accumulator");
        return PARESIS_ERR_ARG;
    }
    const bool detect = job->out_sample || job->out_ref || job->out_propag || job->out_white;
    if (detect && (!job->out_sample || !job->out_ref ||
                   (job->first_point && (!job->out_propag || !job->out_white || !job->acc_white)))) {
        set_last_error("paresis_fresnel_run: incomplete detector outputs (all of them, or none to accumulate only)");
        return PARESIS_ERR_ARG;
    }
    if (detect && (job->oversampling < 1 || job->det_x < 1 || job->det_y < 1)) {
        set_last_error("paresis_fresnel_run: bad detector geometry");
        return PARESIS_ERR_ARG;
    }
    for (int e = 0; e < job->n_energies; ++e) {
        const paresis_fresnel_energy& en = job->energies_host[e];
        if (en.n_membrane < 1 || !en.membrane_host) return bad("no membrane layer", e);
        for (int m = 0; m < en.n_membrane; ++m)
            if (!en.membrane_host[m].thickness) return bad("null membrane map", e);
        if (en.n_sample < 1 || en.n_sample > PARESIS_MAX_LAYERS) return bad("need 1 .. PARESIS_MAX_LAYERS sample layers", e);
        for (int m = 0; m < en.n_sample; ++m)
            if (!en.sample[m].thickness) return bad("null sample map", e);
        if (!en.reference || !en.to_object || !en.to_detector) return bad("null transfer kernel", e);
    }
    // the plan and kernels are host structures too: a kernel prepared for another grid would read past its arrays
    for (int e = 0; e < job->n_energies; ++e) {
        const paresis_fresnel_energy& en = job->energies_host[e];
        if (!fresnel_kernel_fits(job->plan, en.reference) || !fresnel_kernel_fits(job->plan, en.to_object) ||
            !fresnel_kernel_fits(job->plan, en.to_detector))
            return bad("a transfer kernel was prepared for a plan of another size", e);
    }
    return PARESIS_OK;
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

}  // namespace

extern "C" int paresis_fresnel_run(const paresis_fresnel_job* job, paresis_stream stream) {
    int rc = check_job(job);
    if (rc) return rc;
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
