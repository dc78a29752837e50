// Membrane positions of the ray-tracing model as single library calls.
//
// Reference: Experiment.computeSampleAndReferenceImages_RT, Experiment.py:407-526 -- the loop over
// the spectrum (:448) with its three or four refraction hops per energy (:463-498), the mean of the
// reference image (:485-486) and the detector call at every bin close (:501-521); main.py:63-110 for
// the loop over membrane positions around it.  The host shim prepares the per-energy scalars in fp64;
// everything below is kernel launches.
//
// Launch sequence of one steady-state position (mono): raster bin + gather, membrane hop, sample +
// reference hop, detector = 5 kernels and one 16 KB memset.  There are no zero-fill or reduction
// passes: each hop zero-fills what the next one scatters into, the object hop clears I_bs behind
// itself and sums the reference beam while it deposits it (paresis_refract_extras).
#include <array>
#include <vector>

#include "common.cuh"
#include "positions.cuh"

using namespace paresis;

namespace {

// i_bs_group is a list that ends at its first NULL entry: no entry may follow a NULL one
bool group_list_ok(float* const* group) {
    for (int k = 1; k < PARESIS_MAX_GROUP - 1; ++k)
        if (group[k] && !group[k - 1]) return false;
    return true;
}

// every check that reads host memory only: nothing is launched before the whole job is known to be well formed
int check_job(const paresis_rt_job* job) {
    const char* who = "paresis_rt_run";
    if (!job) { set_last_error("%s: null job", who); return PARESIS_ERR_ARG; }
    const int rc = check_rt_job(who, *job);
    if (rc) return rc;
    if ((job->dx_pad == nullptr) != (job->dy_pad == nullptr)) {
        set_last_error("%s: dx_pad and dy_pad come together", who);
        return PARESIS_ERR_ARG;
    }
    if (!group_list_ok(job->i_bs_group)) {
        set_last_error("%s: an i_bs_group entry follows a NULL one (the list ends at its first NULL)", who);
        return PARESIS_ERR_ARG;
    }
    return PARESIS_OK;
}

// the launch sequence of a checked job
int run_job(const paresis_rt_job* job, paresis_stream stream) {
    cudaStream_t s = (cudaStream_t)stream;
    const size_t n = (size_t)job->nx * job->ny;
    const int margin = 15;   // refractionFileNumba2.py:50
    const bool detect = job->out_sample != nullptr;
    // object-plane intensity buffers: one per energy of a group (all zero between jobs)
    float* ibs[PARESIS_MAX_GROUP] = {job->i_bs};
    int n_ibs = 1;
    for (int k = 0; k < PARESIS_MAX_GROUP - 1 && job->i_bs_group[k]; ++k) ibs[n_ibs++] = job->i_bs_group[k];
    if (job->i_bs_dirty)
        for (int k = 0; k < n_ibs; ++k) PARESIS_CUDA(cudaMemsetAsync(ibs[k], 0, sizeof(float) * n, s));
    bool fresh_bin = true;
    int ibin = 0;
    float white = 0.f;
    auto probe = [&](int kind, bool start) {
        if (job->probe == kind && job->probe_start && job->probe_end)
            cudaEventRecord((cudaEvent_t)(start ? job->probe_start : job->probe_end), s);
    };
    // membrane -> object plane (Experiment.py:463-466); a fresh detector bin starts from zero accumulators
    auto membrane_hop = [&](int e, float* dst) -> int {
        const paresis_rt_energy& en = job->energies_host[e];
        paresis_refract_extras x1{};
        x1.throughput = job->throughput;
        if (fresh_bin) {
            x1.zero_fill[0] = job->acc_sample;
            x1.zero_fill[1] = job->acc_ref;
            x1.zero_fill[2] = job->first_point ? job->acc_propag : nullptr;
            white = 0.f;
            fresh_bin = false;
        }
        x1.zero_scalar = job->means ? job->means + e : nullptr;
        x1.intensity_scale = en.intensity_membrane;
        if (e == 0) probe(1, true);
        const int rc = paresis_refract_layers_ex(nullptr, en.intensity_membrane, en.hop1, en.n_hop1, dst, nullptr, nullptr, nullptr,
                                                 job->nx, job->ny, margin, job->flag, &x1, stream);
        if (e == 0) probe(1, false);
        return rc;
    };
    // the sample alone (:490-498); the white field is the incident beam itself
    auto propagation_hop = [&](int e) -> int {
        const paresis_rt_energy& en = job->energies_host[e];
        const bool want_d = job->dx_pad && job->dy_pad && e == job->n_energies - 1;
        if (want_d) {
            const size_t np = (size_t)(job->nx + 2 * margin) * (job->ny + 2 * margin);
            PARESIS_CUDA(cudaMemsetAsync(job->dx_pad, 0, sizeof(float) * np, s));
            PARESIS_CUDA(cudaMemsetAsync(job->dy_pad, 0, sizeof(float) * np, s));
        }
        paresis_refract_extras x3{};
        x3.throughput = job->throughput;
        x3.intensity_scale = en.intensity_propag;
        const int rc = paresis_refract_layers_ex(nullptr, en.intensity_propag, en.propag, en.n_propag, job->acc_propag, nullptr,
                                                 want_d ? job->dx_pad : nullptr, want_d ? job->dy_pad : nullptr, job->nx, job->ny,
                                                 margin, job->flag, &x3, stream);
        white += en.intensity_propag;
        return rc;
    };
    auto same_maps = [&](const paresis_rt_energy& p, const paresis_rt_energy& q) {
        if (p.n_hop2 != q.n_hop2) return false;
        for (int m = 0; m < p.n_hop2; ++m)
            if (p.hop2[m].thickness != q.hop2[m].thickness) return false;
        return true;
    };
    for (int e = 0; e < job->n_energies;) {
        const paresis_rt_energy& en = job->energies_host[e];
        // energies of the same detector bin that share their maps go through the object hop together
        int group = 1;
        while (group < n_ibs && e + group < job->n_energies && !job->energies_host[e + group - 1].close_bin &&
               same_maps(en, job->energies_host[e + group]))
            ++group;
        int rc;
        if (group == 1) {
            rc = membrane_hop(e, job->i_bs);
            if (rc) return rc;
            // object -> detector: sample beam and reference beam in one pass over I_bs (:469-474), which is
            // cleared behind the pass; the reference beam is summed on the way (:485-486)
            paresis_refract_extras x2{};
            x2.throughput = job->throughput;
            x2.clear_input = 1;
            x2.sum_ref = job->means ? job->means + e : nullptr;
            x2.intensity_scale = en.intensity_membrane;
            if (e == 0) probe(2, true);
            rc = paresis_refract_layers_ex(job->i_bs, 0.f, en.hop2, en.n_hop2, job->acc_sample, job->acc_ref, nullptr, nullptr,
                                           job->nx, job->ny, margin, job->flag, &x2, stream);
            if (e == 0) probe(2, false);
            if (rc) return rc;
        } else {
            paresis_group_energy ge[PARESIS_MAX_GROUP];
            for (int g = 0; g < group; ++g) {
                rc = membrane_hop(e + g, ibs[g]);
                if (rc) return rc;
                const paresis_rt_energy& eg = job->energies_host[e + g];
                for (int m = 0; m < eg.n_hop2; ++m) ge[g].layers[m] = eg.hop2[m];
                ge[g].n_layers = eg.n_hop2;
                ge[g].intensity_in = ibs[g];
                ge[g].intensity_scale = eg.intensity_membrane;
                ge[g].sum_ref = job->means ? job->means + e + g : nullptr;
            }
            if (e == 0) probe(2, true);
            rc = paresis_refract_group(ge, group, job->acc_sample, job->acc_ref, job->nx, job->ny, job->flag, stream);
            if (e == 0) probe(2, false);
            if (rc) return rc;
        }
        for (int g = 0; g < group; ++g) {
            if (job->first_point) {
                rc = propagation_hop(e + g);
                if (rc) return rc;
            }
        }
        if (detect && job->energies_host[e + group - 1].close_bin) {   // :501-521
            const bool probed = ibin == 0 && job->probe == 3 && job->probe_start && job->probe_end;
            rc = close_bin(*job, job->nx, job->ny, ibin, white, stream, probed ? job->probe_start : nullptr,
                           probed ? job->probe_end : nullptr);
            if (rc) return rc;
            ++ibin;
            fresh_bin = true;
        }
        e += group;
    }
    return PARESIS_OK;
}

}  // namespace

extern "C" int paresis_rt_run(const paresis_rt_job* job, paresis_stream stream) {
    const int rc = check_job(job);
    if (rc) return rc;
    return run_job(job, stream);
}

// ---------------------------------------------------------------------------------------------------------------
// Several positions per launch.  A position at 2048^2 is 18 pixels per resident thread: ramp, tail and per-block set-up
// of its kernels cannot be amortised inside one position (DESIGN.md, "What bounds the hops").  Here the membrane cut,
// each hop and the detector of up to `positions_per_launch` positions are ONE launch each (blockIdx.z = position, slot
// z's scratch), all on the caller's stream.  Position 0 (propagation + white images, Experiment.py:488-498) runs alone.
// ---------------------------------------------------------------------------------------------------------------
static bool single_energy_bins(const paresis_rt_job* job) {
    for (int e = 0; e < job->n_energies; ++e)
        if (!job->energies_host[e].close_bin) return false;
    return true;
}

static int run_positions_batched(const paresis_rt_job* job, const paresis_membrane* mem, const paresis_rt_position* positions,
                                 int n_positions, paresis_rt_slot* slots, int n_slots, paresis_stream stream) {
    cudaStream_t s = (cudaStream_t)stream;
    const size_t n = (size_t)job->nx * job->ny, nd = (size_t)job->det_x * job->det_y;
    int per = job->positions_per_launch;
    if (per > n_slots) per = n_slots;
    if (per > PARESIS_MAX_HOP_BATCH) per = PARESIS_MAX_HOP_BATCH;
    for (int k = 0; k < n_slots; ++k)
        if (slots[k].i_bs_dirty) { PARESIS_CUDA(cudaMemsetAsync(slots[k].i_bs, 0, sizeof(float) * n, s)); slots[k].i_bs_dirty = 0; }

    auto run_group = [&](const int* idx, int g) -> int {
        const paresis_rt_position* pos[PARESIS_MAX_HOP_BATCH];
        const int64_t* offs[PARESIS_MAX_HOP_BATCH];
        float* thick[PARESIS_MAX_HOP_BATCH];
        void *ev0 = nullptr, *ev1 = nullptr;              // probe events of the first probed position of the group
        for (int z = 0; z < g; ++z) {
            pos[z] = &positions[idx[z]];
            offs[z] = pos[z]->offsets_host; thick[z] = pos[z]->thickness;
            if (!ev0 && pos[z]->probe_start && pos[z]->probe_end) { ev0 = pos[z]->probe_start; ev1 = pos[z]->probe_end; }
        }
        auto probe = [&](int kind, bool start) {
            if (job->probe == kind && ev0) cudaEventRecord((cudaEvent_t)(start ? ev0 : ev1), s);
        };
        probe(4, true);
        int rc = paresis_membrane_from_field_batch(mem->field, mem->field_x, mem->field_y, offs, thick, g, mem->n_layers, mem->margin,
                                                   job->nx, job->ny, stream);
        probe(4, false);
        if (rc) return rc;
        int ibin = 0;
        for (int e = 0; e < job->n_energies; ++e) {
            const paresis_rt_energy& en = job->energies_host[e];
            paresis_tile_hop_item h1[PARESIS_MAX_HOP_BATCH] = {}, h2[PARESIS_MAX_HOP_BATCH] = {};
            for (int z = 0; z < g; ++z) {
                const paresis_rt_slot& sl = slots[z];
                for (int m = 0; m < en.n_hop1; ++m) h1[z].thickness[m] = en.hop1[m].thickness ? en.hop1[m].thickness : thick[z];
                h1[z].out_obj = sl.i_bs;
                h1[z].zero_fill[0] = sl.acc_sample;          // every energy closes its bin here: fresh accumulators each time
                h1[z].zero_fill[1] = sl.acc_ref;
                h1[z].zero_scalar = pos[z]->means ? pos[z]->means + e : nullptr;
                for (int m = 0; m < en.n_hop2; ++m) h2[z].thickness[m] = en.hop2[m].thickness ? en.hop2[m].thickness : thick[z];
                h2[z].intensity_in = sl.i_bs;
                h2[z].out_obj = sl.acc_sample;
                h2[z].out_ref = sl.acc_ref;
                h2[z].sum_ref = pos[z]->means ? pos[z]->means + e : nullptr;
            }
            if (e == 0) probe(1, true);
            rc = paresis_refract_tile_batch(h1, g, en.hop1, en.n_hop1, en.intensity_membrane, en.intensity_membrane, 0, job->nx, job->ny,
                                            job->flag, stream);
            if (e == 0) probe(1, false);
            if (rc) return rc;
            if (e == 0) probe(2, true);
            rc = paresis_refract_tile_batch(h2, g, en.hop2, en.n_hop2, 0.f, en.intensity_membrane, 1, job->nx, job->ny, job->flag, stream);
            if (e == 0) probe(2, false);
            if (rc) return rc;
            // the detector: sample + reference image of up to four positions per launch (Experiment.py:501-521)
            for (int z0 = 0; z0 < g; z0 += 4) {
                const int gz = g - z0 < 4 ? g - z0 : 4;
                const float* in_k[8]; float* out_k[8]; uint64_t seq_k[8];
                for (int z = 0; z < gz; ++z) {
                    const uint64_t seq = pos[z0 + z]->sequence + (uint64_t)ibin * 4;
                    in_k[2 * z] = slots[z0 + z].acc_sample; out_k[2 * z] = pos[z0 + z]->out_sample + (size_t)ibin * nd; seq_k[2 * z] = seq;
                    in_k[2 * z + 1] = slots[z0 + z].acc_ref; out_k[2 * z + 1] = pos[z0 + z]->out_ref + (size_t)ibin * nd; seq_k[2 * z + 1] = seq + 1;
                }
                if (ibin == 0 && z0 == 0) probe(3, true);
                rc = paresis_detect_counts_multi(in_k, out_k, seq_k, 2 * gz, job->nx, job->ny, job->oversampling, job->det_x, job->det_y,
                                                 job->src_kernel, job->src_half, job->psf_kernel, job->psf_half, job->detect_work,
                                                 job->noise, job->seed, stream);
                if (ibin == 0 && z0 == 0) probe(3, false);
                if (rc) return rc;
            }
            ++ibin;
        }
        return PARESIS_OK;
    };

    std::vector<paresis_rt_energy> energies(job->energies_host, job->energies_host + job->n_energies);
    int group[PARESIS_MAX_HOP_BATCH], g = 0;
    for (int p = 0; p < n_positions; ++p) {
        const paresis_rt_position& pos = positions[p];
        if (!pos.first_point) {
            group[g++] = p;
            if (g == per) { int rc = run_group(group, g); if (rc) return rc; g = 0; }
            continue;
        }
        // position 0: on its own, through the per-position pipeline, after what is pending (it shares slot 0)
        if (g) { int rc = run_group(group, g); if (rc) return rc; g = 0; }
        int rc = paresis_membrane_from_field(mem->field, mem->field_x, mem->field_y, pos.offsets_host, mem->n_layers, mem->margin,
                                             job->nx, job->ny, pos.thickness, stream);
        if (rc) return rc;
        bind_position_maps(job->energies_host, job->n_energies, pos.thickness, energies.data());
        paresis_rt_job j = *job;
        j.energies_host = energies.data();
        j.first_point = 1;
        j.i_bs = slots[0].i_bs; j.acc_sample = slots[0].acc_sample; j.acc_ref = slots[0].acc_ref;
        j.acc_propag = slots[0].acc_propag; j.acc_white = slots[0].acc_white;
        j.i_bs_dirty = 0;
        j.means = pos.means;
        j.out_sample = pos.out_sample; j.out_ref = pos.out_ref; j.out_propag = pos.out_propag; j.out_white = pos.out_white;
        j.sequence = pos.sequence;
        j.probe = 0;
        j.dx_pad = j.dy_pad = nullptr;
        rc = run_job(&j, stream);
        if (rc) return rc;
    }
    if (g) { int rc = run_group(group, g); if (rc) return rc; }
    return PARESIS_OK;
}

// every argument of paresis_rt_run_positions, host memory only
static int check_positions(const paresis_rt_job* job, const paresis_membrane* mem, const paresis_rt_position* positions,
                           int n_positions, const paresis_rt_slot* slots, int n_slots) {
    const char* who = "paresis_rt_run_positions";
    int rc = check_call(who, job, mem, positions, slots, n_positions, n_slots);
    if (rc || n_positions == 0) return rc;       // nothing to run, nothing else to check
    rc = check_rt_frame(who, *job);
    if (rc) return rc;
    rc = check_membrane_detector(who, mem, job->oversampling, job->det_x, job->det_y);
    if (rc) return rc;
    bool any_first = false;
    for (int p = 0; p < n_positions; ++p) {
        rc = check_position(who, positions[p], p);
        if (rc) return rc;
        any_first |= positions[p].first_point != 0;
    }
    for (int k = 0; k < n_slots; ++k) {
        const paresis_rt_slot& sl = slots[k];
        if (!sl.i_bs || !sl.acc_sample || !sl.acc_ref || !sl.acc_propag || !sl.acc_white) {
            set_last_error("%s: slot %d lacks an object-plane buffer or an accumulator", who, k);
            return PARESIS_ERR_ARG;
        }
        if (!group_list_ok(sl.i_bs_group)) {
            set_last_error("%s: slot %d: an i_bs_group entry follows a NULL one (the list ends at its first NULL)", who, k);
            return PARESIS_ERR_ARG;
        }
    }
    rc = check_slots_apart(who, slots, n_slots, [](const paresis_rt_slot& sl) {
        std::array<const void*, 6 + PARESIS_MAX_GROUP - 1> images{sl.i_bs, sl.acc_sample, sl.acc_ref, sl.acc_propag,
                                                                  sl.acc_white, sl.detect_work};
        for (int k = 0; k < PARESIS_MAX_GROUP - 1; ++k) images[6 + k] = sl.i_bs_group[k];
        return images;
    });
    if (rc) return rc;
    rc = check_rt_energies(who, *job, any_first, true);
    if (rc) return rc;
    return check_raster_work(who, mem, job->nx, job->ny, slots, n_slots);
}

// Each position: its membrane map (cut from the sphere field, or rasterised), then the launch sequence of paresis_rt_run
// on its slot's stream with the slot's buffers -- or, with positions_per_launch, several positions per launch.
extern "C" int paresis_rt_run_positions(const paresis_rt_job* job, const paresis_membrane* mem,
                                        const paresis_rt_position* positions, int n_positions,
                                        paresis_rt_slot* slots, int n_slots, paresis_stream stream) {
    const int rc = check_positions(job, mem, positions, n_positions, slots, n_slots);
    if (rc) return rc;
    if (n_positions == 0) return PARESIS_OK;
    if (job->positions_per_launch > 1 && mem->field && !job->i_bs_group[0] && single_energy_bins(job))
        return run_positions_batched(job, mem, positions, n_positions, slots, n_slots, stream);
    std::vector<paresis_rt_energy> energies(job->energies_host, job->energies_host + job->n_energies);
    // A probed position runs alone on the GPU, so that the CUDA events around its kernel time that kernel and not its
    // neighbours on the other streams.
    auto probed = [&](int p) { return job->probe != 0 && positions[p].probe_start && positions[p].probe_end && n_slots > 1; };
    auto run = [&](int p, paresis_rt_slot& slot) -> int {
        const paresis_rt_position& pos = positions[p];
        const bool probe_raster = job->probe == 4 && pos.probe_start && pos.probe_end;
        if (probe_raster) cudaEventRecord((cudaEvent_t)pos.probe_start, (cudaStream_t)slot.stream);
        int rc = membrane_of_position(mem, pos.offsets_host, job->nx, job->ny, pos.thickness, slot.raster_work,
                                      slot.raster_work_bytes, slot.stream);
        if (probe_raster) cudaEventRecord((cudaEvent_t)pos.probe_end, (cudaStream_t)slot.stream);
        if (rc) return rc;
        bind_position_maps(job->energies_host, job->n_energies, pos.thickness, energies.data());
        paresis_rt_job j = *job;
        j.energies_host = energies.data();
        bind_position(j, pos);
        j.i_bs = slot.i_bs; j.acc_sample = slot.acc_sample; j.acc_ref = slot.acc_ref;
        for (int k = 0; k < PARESIS_MAX_GROUP - 1; ++k) j.i_bs_group[k] = slot.i_bs_group[k];
        j.acc_propag = slot.acc_propag; j.acc_white = slot.acc_white;
        j.i_bs_dirty = slot.i_bs_dirty;
        j.detect_work = slot.detect_work;
        j.probe_start = pos.probe_start; j.probe_end = pos.probe_end;
        if (!pos.probe_start || !pos.probe_end) j.probe = 0;
        j.dx_pad = j.dy_pad = nullptr;
        if (n_positions > 1) j.throughput = 1;        // launches of neighbouring positions overlap: least work per pixel wins
        rc = run_job(&j, slot.stream);
        if (rc) return rc;
        slot.i_bs_dirty = 0;
        return PARESIS_OK;
    };
    return run_on_slots(slots, n_slots, n_positions, stream, run, probed);
}
