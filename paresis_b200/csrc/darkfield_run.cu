// Membrane positions of the ray-tracing model with a scattering sample as single library calls.
//
// Reference: Experiment.computeSampleAndReferenceImages_RT, Experiment.py:407-526, for a sample with the Lung /
// 'cylinder_beeds' dark-field model (Sample.py:322-343): the sample beam goes through fastRefractionDF
// (refractionFileNumba2.py:88-196) -- the rays with and without a scattering angle are refracted apart, then the
// scattered ones are spread over Gaussian patches of their angle.  The host prepares the per-energy scalars in fp64;
// everything below is kernel launches of csrc/darkfield.cu and the mode-0 refraction hop.
//
// The object hop runs as two dual-beam hops, one on the plain rays and one on the scattered rays.  The splat is linear
// in intensity, so their two reference deposits add up to the reference beam of the whole object-plane image, and each
// energy's reference sum comes out of the hops (sum_ref) with no reduction pass.
#include "common.cuh"

using namespace paresis;

namespace {

constexpr int kMargin = 15;   // refractionFileNumba2.py:50

int bad(const char* what, int e) {
    set_last_error("paresis_df_run: energy %d: %s", e, what);
    return PARESIS_ERR_ARG;
}

// every check that reads host memory only: nothing is launched before the whole job is known to be well formed
int check_job(const paresis_df_job* job) {
    if (!job) { set_last_error("paresis_df_run: null job"); return PARESIS_ERR_ARG; }
    const paresis_rt_job& r = job->rt;
    if (!r.energies_host || !job->energies_df_host || r.n_energies < 1) {
        set_last_error("paresis_df_run: no energies");
        return PARESIS_ERR_ARG;
    }
    if (r.nx < 3 || r.ny < 3) { set_last_error("paresis_df_run: bad frame %d x %d", r.nx, r.ny); return PARESIS_ERR_ARG; }
    if (!r.i_bs || !r.acc_sample || !r.acc_ref || (r.first_point && !r.acc_propag)) {
        set_last_error("paresis_df_run: null object-plane buffer or accumulator");
        return PARESIS_ERR_ARG;
    }
    if (!job->angle || !job->plain || !job->scattered || !job->clean || !job->moved) {
        set_last_error("paresis_df_run: null dark-field scratch buffer");
        return PARESIS_ERR_ARG;
    }
    const bool detect = r.out_sample || r.out_ref || r.out_propag || r.out_white;
    if (detect && (!r.out_sample || !r.out_ref || (r.first_point && (!r.out_propag || !r.out_white || !r.acc_white)))) {
        set_last_error("paresis_df_run: incomplete detector outputs (all of them, or none to accumulate only)");
        return PARESIS_ERR_ARG;
    }
    if (detect && (r.oversampling < 1 || r.det_x < 1 || r.det_y < 1)) {
        set_last_error("paresis_df_run: bad detector geometry");
        return PARESIS_ERR_ARG;
    }
    if (job->dark_field && !r.first_point) {
        set_last_error("paresis_df_run: the dark-field map belongs to position 0 (first_point)");
        return PARESIS_ERR_ARG;
    }
    for (int e = 0; e < r.n_energies; ++e) {
        const paresis_rt_energy& en = r.energies_host[e];
        const paresis_df_energy& df = job->energies_df_host[e];
        if (en.n_hop1 < 1 || en.n_hop1 > PARESIS_MAX_LAYERS) return bad("need 1 .. PARESIS_MAX_LAYERS membrane maps", e);
        if (en.n_hop2 < 1 || en.n_hop2 > PARESIS_MAX_LAYERS)
            return bad("need 1 .. PARESIS_MAX_LAYERS membrane + sample maps in the object hop (mix the sample's maps)", e);
        if (r.first_point && (en.n_propag < 1 || en.n_propag > PARESIS_MAX_LAYERS))
            return bad("need 1 .. PARESIS_MAX_LAYERS sample maps in the sample-only hop", e);
        for (int m = 0; m < en.n_hop1; ++m) if (!en.hop1[m].thickness) return bad("null membrane map", e);
        for (int m = 0; m < en.n_hop2; ++m) if (!en.hop2[m].thickness) return bad("null object-hop map", e);
        if (r.first_point)
            for (int m = 0; m < en.n_propag; ++m) if (!en.propag[m].thickness) return bad("null sample map", e);
        if (!df.scatter_map) return bad("no scattering map", e);
    }
    return PARESIS_OK;
}

}  // namespace

extern "C" int paresis_df_run(const paresis_df_job* job, paresis_stream stream) {
    int rc = check_job(job);
    if (rc) return rc;
    const paresis_rt_job& r = job->rt;
    cudaStream_t s = (cudaStream_t)stream;
    const int nx = r.nx, ny = r.ny;
    const size_t n = (size_t)nx * ny, nd = (size_t)r.det_x * r.det_y;
    const float limit = nx / 4.f;                         // refractionFileNumba2.py:130
    const bool detect = r.out_sample != nullptr;
    if (r.i_bs_dirty) PARESIS_CUDA(cudaMemsetAsync(r.i_bs, 0, sizeof(float) * n, s));
    // one hop of the mode-0 kernels; zero_fill: up to two buffers this hop does not touch, cleared for a later one
    auto hop = [&](const float* in, float uniform, const paresis_layer* layers, int n_layers, float* out_obj, float* out_ref,
                   float scale, float* z0, float* z1, float* z2, double* zero_scalar, double* sum_ref) {
        paresis_refract_extras x{};
        x.throughput = r.throughput;
        x.intensity_scale = scale;
        x.zero_fill[0] = z0; x.zero_fill[1] = z1; x.zero_fill[2] = z2;
        x.zero_scalar = zero_scalar;
        x.sum_ref = sum_ref;
        return paresis_refract_layers_ex(in, uniform, layers, n_layers, out_obj, out_ref, nullptr, nullptr, nx, ny, kMargin,
                                         r.flag, &x, stream);
    };
    bool fresh_bin = true;
    int ibin = 0;
    float white = 0.f;
    for (int e = 0; e < r.n_energies; ++e) {
        const paresis_rt_energy& en = r.energies_host[e];
        const paresis_df_energy& df = job->energies_df_host[e];
        double* mean_e = r.means ? r.means + e : nullptr;
        // the scattering angle in pixels at the detector (Sample.py:322-343, refractionFileNumba2.py:114)
        rc = paresis_df_angle(df.scatter_map, df.angle_coeff, job->angle, n, stream);
        if (rc) return rc;
        // membrane -> object plane (Experiment.py:463-466); a fresh detector bin starts from zero accumulators
        float* z[3] = {nullptr, nullptr, nullptr};
        if (fresh_bin) {
            z[0] = r.acc_sample; z[1] = r.acc_ref; z[2] = r.first_point ? r.acc_propag : nullptr;
            white = 0.f;
            fresh_bin = false;
        }
        rc = hop(nullptr, en.intensity_membrane, en.hop1, en.n_hop1, r.i_bs, nullptr, en.intensity_membrane, z[0], z[1], z[2],
                 mean_e, nullptr);
        if (rc) return rc;
        // the object-plane beam split by scattering angle (refractionFileNumba2.py:130, :143-146)
        rc = paresis_df_split(r.i_bs, 0.f, job->angle, limit, job->plain, job->scattered, job->clean, n, stream);
        if (rc) return rc;
        // object -> detector, sample and reference beams (:469-474): the plain rays, then the scattered rays.  The first
        // hop clears `moved` for the second; the second clears I_bs, which the split has consumed.
        rc = hop(job->plain, 0.f, en.hop2, en.n_hop2, r.acc_sample, r.acc_ref, en.intensity_membrane, job->moved, nullptr, nullptr,
                 nullptr, mean_e);
        if (rc) return rc;
        rc = hop(job->scattered, 0.f, en.hop2, en.n_hop2, job->moved, r.acc_ref, en.intensity_membrane, r.i_bs, nullptr, nullptr,
                 nullptr, mean_e);
        if (rc) return rc;
        // the refracted scattered rays spread over their Gaussian patches (refractionFileNumba2.py:171-186)
        rc = paresis_df_scatter(job->moved, job->clean, r.acc_sample, nx, ny, stream);
        if (rc) return rc;
        if (r.first_point) {
            // the sample alone (:490-498) through the same split; the white field is the incident beam itself
            rc = paresis_df_split(nullptr, en.intensity_propag, job->angle, limit, job->plain, job->scattered, job->clean, n, stream);
            if (rc) return rc;
            rc = hop(job->plain, 0.f, en.propag, en.n_propag, r.acc_propag, nullptr, en.intensity_propag, job->moved, nullptr,
                     nullptr, nullptr, nullptr);
            if (rc) return rc;
            rc = hop(job->scattered, 0.f, en.propag, en.n_propag, job->moved, nullptr, en.intensity_propag, nullptr, nullptr,
                     nullptr, nullptr, nullptr);
            if (rc) return rc;
            rc = paresis_df_scatter(job->moved, job->clean, r.acc_propag, nx, ny, stream);
            if (rc) return rc;
            if (job->dark_field) {   // self.darkFieldPropag += DarkFieldPropag * flux (:491), back in radians
                rc = paresis_axpy(job->dark_field, job->angle, (float)df.dark_field_weight, n, stream);
                if (rc) return rc;
            }
            white += en.intensity_propag;
        }
        if (detect && en.close_bin) {   // :501-521, all images of the bin in one launch
            const int count = r.first_point ? 4 : 2;
            if (r.first_point) {
                rc = paresis_fill(r.acc_white, white, n, stream);
                if (rc) return rc;
            }
            const uint64_t seq = r.sequence + (uint64_t)ibin * 4;
            const float* in_k[4] = {r.acc_sample, r.acc_ref, r.acc_propag, r.acc_white};
            float* out_k[4] = {r.out_sample + (size_t)ibin * nd, r.out_ref + (size_t)ibin * nd,
                               r.first_point ? r.out_propag + (size_t)ibin * nd : nullptr,
                               r.first_point ? r.out_white + (size_t)ibin * nd : nullptr};
            const uint64_t seq_k[4] = {seq, seq + 1, seq + 2, seq + 3};
            rc = paresis_detect_counts_multi(in_k, out_k, seq_k, count, nx, ny, r.oversampling, r.det_x, r.det_y, r.src_kernel,
                                             r.src_half, r.psf_kernel, r.psf_half, r.detect_work, r.noise, r.seed, stream);
            if (rc) return rc;
            ++ibin;
            fresh_bin = true;
        }
    }
    return PARESIS_OK;
}
