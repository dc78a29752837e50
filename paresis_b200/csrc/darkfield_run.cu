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
//
// paresis_df_run_positions runs the same launch sequence for many membrane positions of a scan (main.py:63-110) in one
// call, the positions dealt over slots that each own an object-plane buffer, accumulators and dark-field scratch and run
// on their own stream, so that consecutive positions overlap on the GPU.
#include <cuda_runtime.h>

#include <array>
#include <vector>

#include "common.cuh"
#include "positions.cuh"

using namespace paresis;

namespace {

constexpr int kMargin = 15;   // refractionFileNumba2.py:50

// every energy has a scattering map (host memory only)
int check_scatter_maps(const char* who, const paresis_df_job* job) {
    for (int e = 0; e < job->rt.n_energies; ++e)
        if (!job->energies_df_host[e].scatter_map) {
            set_last_error("%s: energy %d: no scattering map", who, e);
            return PARESIS_ERR_ARG;
        }
    return PARESIS_OK;
}

// every check that reads host memory only: nothing is launched before the whole job is known to be well formed
int check_job(const paresis_df_job* job) {
    const char* who = "paresis_df_run";
    if (!job) { set_last_error("%s: null job", who); return PARESIS_ERR_ARG; }
    if (!job->energies_df_host) { set_last_error("%s: no energies", who); return PARESIS_ERR_ARG; }
    const paresis_rt_job& r = job->rt;
    int rc = check_rt_job(who, r);
    if (rc) return rc;
    if (!job->angle || !job->plain || !job->scattered || !job->clean || !job->moved) {
        set_last_error("%s: null dark-field scratch buffer", who);
        return PARESIS_ERR_ARG;
    }
    if (job->dark_field && !r.first_point) {
        set_last_error("%s: the dark-field map belongs to position 0 (first_point)", who);
        return PARESIS_ERR_ARG;
    }
    return check_scatter_maps(who, job);
}

// the launch sequence of a checked job
int run_job(const paresis_df_job* job, paresis_stream stream) {
    int rc = PARESIS_OK;
    const paresis_rt_job& r = job->rt;
    cudaStream_t s = (cudaStream_t)stream;
    const int nx = r.nx, ny = r.ny;
    const size_t n = (size_t)nx * ny;
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
            rc = close_bin(r, nx, ny, ibin, white, stream);
            if (rc) return rc;
            ++ibin;
            fresh_bin = true;
        }
    }
    return PARESIS_OK;
}

}  // namespace

extern "C" int paresis_df_run(const paresis_df_job* job, paresis_stream stream) {
    const int rc = check_job(job);
    if (rc) return rc;
    return run_job(job, stream);
}

namespace {

int bad_positions(const char* fmt, int i) {
    set_last_error(fmt, i);
    return PARESIS_ERR_ARG;
}

// every argument of paresis_df_run_positions, host memory only
int check_positions(const paresis_df_job* job, const paresis_membrane* mem, const paresis_df_position* positions,
                    int n_positions, const paresis_df_slot* slots, int n_slots) {
    const char* who = "paresis_df_run_positions";
    int rc = check_call(who, job, mem, positions, slots, n_positions, n_slots);
    if (rc || n_positions == 0) return rc;       // nothing to run, nothing else to check
    const paresis_rt_job& r = job->rt;
    if (!job->energies_df_host) { set_last_error("%s: no energies", who); return PARESIS_ERR_ARG; }
    rc = check_rt_frame(who, r);
    if (rc) return rc;
    rc = check_membrane_detector(who, mem, r.oversampling, r.det_x, r.det_y);
    if (rc) return rc;
    bool any_first = false;
    for (int p = 0; p < n_positions; ++p) {
        const paresis_rt_position& pos = positions[p].rt;
        rc = check_position(who, pos, p);
        if (rc) return rc;
        rc = check_no_probe(who, pos, p);
        if (rc) return rc;
        if (positions[p].dark_field && !pos.first_point)
            return bad_positions("paresis_df_run_positions: position %d: the dark-field map belongs to position 0 (first_point)", p);
        any_first |= pos.first_point != 0;
    }
    for (int k = 0; k < n_slots; ++k) {
        const paresis_df_slot& sl = slots[k];
        if (!sl.i_bs || !sl.acc_sample || !sl.acc_ref || !sl.acc_propag || !sl.acc_white)
            return bad_positions("paresis_df_run_positions: slot %d lacks an object-plane buffer or an accumulator", k);
        if (!sl.angle || !sl.plain || !sl.scattered || !sl.clean || !sl.moved)
            return bad_positions("paresis_df_run_positions: slot %d lacks a dark-field scratch image", k);
    }
    rc = check_slots_apart(who, slots, n_slots, [](const paresis_df_slot& sl) {
        return std::array<const void*, 11>{sl.i_bs, sl.acc_sample, sl.acc_ref, sl.acc_propag, sl.acc_white, sl.angle,
                                           sl.plain, sl.scattered, sl.clean, sl.moved, sl.detect_work};
    });
    if (rc) return rc;
    rc = check_rt_energies(who, r, any_first, true);
    if (rc) return rc;
    rc = check_scatter_maps(who, job);
    if (rc) return rc;
    return check_raster_work(who, mem, r.nx, r.ny, slots, n_slots);
}

}  // namespace

// Each position: its membrane map (cut from the sphere field, or rasterised), then the launch sequence of paresis_df_run
// on its slot's stream with the slot's buffers.  Position p goes to slot p mod n_slots.
extern "C" int paresis_df_run_positions(const paresis_df_job* job, const paresis_membrane* mem,
                                        const paresis_df_position* positions, int n_positions, paresis_df_slot* slots,
                                        int n_slots, paresis_stream stream) {
    int rc = check_positions(job, mem, positions, n_positions, slots, n_slots);
    if (rc) return rc;
    if (n_positions == 0) return PARESIS_OK;
    const paresis_rt_job& r = job->rt;
    std::vector<paresis_rt_energy> energies(r.energies_host, r.energies_host + r.n_energies);
    return run_on_slots(slots, n_slots, n_positions, stream, [&](int p, paresis_df_slot& slot) -> int {
        const paresis_rt_position& pos = positions[p].rt;
        int rc = membrane_of_position(mem, pos.offsets_host, r.nx, r.ny, pos.thickness, slot.raster_work, slot.raster_work_bytes,
                                      slot.stream);
        if (rc) return rc;
        bind_position_maps(r.energies_host, r.n_energies, pos.thickness, energies.data());
        paresis_df_job j = *job;
        paresis_rt_job& jr = j.rt;
        jr.energies_host = energies.data();
        bind_position(jr, pos);
        jr.i_bs = slot.i_bs; jr.acc_sample = slot.acc_sample; jr.acc_ref = slot.acc_ref;
        jr.acc_propag = slot.acc_propag; jr.acc_white = slot.acc_white;
        jr.i_bs_dirty = slot.i_bs_dirty;
        jr.detect_work = slot.detect_work;
        if (n_positions > 1) jr.throughput = 1;       // launches of neighbouring positions overlap: least work per pixel wins
        j.angle = slot.angle; j.plain = slot.plain; j.scattered = slot.scattered; j.clean = slot.clean; j.moved = slot.moved;
        j.dark_field = positions[p].dark_field;
        rc = run_job(&j, slot.stream);
        if (rc) return rc;
        slot.i_bs_dirty = 0;
        return PARESIS_OK;
    });
}
