/*
 * paresis_b200 -- C ABI of the B200 (sm_100a) image-formation library.
 *
 * This is the drop-in boundary for PARESIS's per-(energy, membrane position) hot path.
 * PARESIS has no FFI of its own: the functions below replace, one for one, the Python /
 * Numba callables its orchestration layer invokes (SURVEY.md section 8b).  Each entry cites
 * the reference interface it stands in for, as path:line under /root/reference/CodePython.
 *
 * Conventions
 *   - plain C: raw pointers, sizes, scalars by value; no torch / C++ types.
 *   - every array pointer is DEVICE memory unless the parameter name ends in `_host`.
 *   - images are row-major [nx][ny] (axis 0 = "x" = row, as in the reference), pitch = ny.
 *   - the caller owns all memory; the library owns only cuFFT plans (explicit create/destroy).
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on that stream.
 *   - return value: PARESIS_OK or an error code; paresis_last_error() gives the text.
 *   - `flag` (nullable) is a device int that kernels OR status bits into
 *     (PARESIS_FLAG_NONFINITE = the reference's "nans or insane values" guard,
 *     refractionFileNumba2.py:81-82); the host shim reads it lazily and raises.
 */
#ifndef PARESIS_B200_H
#define PARESIS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PARESIS_OK 0
#define PARESIS_ERR_CUDA 1
#define PARESIS_ERR_ARG 2
#define PARESIS_ERR_CUFFT 3

#define PARESIS_FLAG_NONFINITE 1

#define PARESIS_MAX_LAYERS 4
#define PARESIS_MAX_HOP_BATCH 8   /* membrane positions that can share one launch (blockIdx.z) */

typedef void* paresis_stream;
typedef struct { float re, im; } paresis_c32;

int paresis_version(void);
const char* paresis_last_error(void);
/* Performance knobs, results unaffected.  key 0: deposit mode of the fused refraction kernels
 * (0 = one REDG per deposit, 2 = warp/register aggregated, default); key 1: source rows per warp
 * (0 = automatic); key 2: -1 = direct-to-L2 hop kernels, 0 = tile kernels (default); key 3: source rows per block of the tile
 * hops (0 = chosen per launch to fill whole waves, the default). */
int paresis_set_tuning(int key, int value);
/* Frees the library's cached per-device scratch (the ray lists of the strip kernels: up to 16 bytes per study pixel and
 * beam, kept between calls so that a call allocates nothing).  Safe at any time; the next call allocates again. */
int paresis_trim(void);

/* ---------------------------------------------------------------------------------------
 * Refraction model (ray tracing)
 * ------------------------------------------------------------------------------------- */

/* fastloopNumba(Nx, Ny, I, I2, Dy, Dx, DxFloor, DyFloor) -- refractionFileNumba2.py:198-263
 * (same body: refractionFileNumba.py:70-135).  out += bilinear scatter of `intensity` by
 * (dx, dy) pixels.  `margin` is the virtual zero padding of the loop frame: 0 reproduces a
 * direct call (edge quirk of :238-262 included), 15 / 10 what fastRefraction v2 / v1 see
 * after pad + crop (refractionFileNumba2.py:65-78).  `variant`: 0 = plain REDs,
 * 1 = warp-aggregated rows, 2 = warp-aggregated rows + register-carried columns (default),
 * 3 = fixed-point shared-memory tiles with a dense flush (the one for torn displacement fields such as a
 * membrane's; deposits are quantised to 2^-19 ... 2^-18 of the mean ray of each 16 x 256 source tile, rays
 * brighter than twice that mean bypass the tiles). */
int paresis_splat(const float* intensity, const float* dx, const float* dy, float* out,
                  int nx, int ny, int margin, int variant, int* flag, paresis_stream stream);

/* fastRefraction(I, phi, z, E, M, pix) -- refractionFileNumba2.py:25-86 (v1:
 * refractionFileNumba.py:11-68), fused: gradient (np.gradient edge_order=2, :54) ->
 * displacement in pixels (:55-56) -> clean-up (:59-64) -> scatter (:77) in one kernel.
 * out[nx][ny] += result.  dx_pad / dy_pad (nullable) receive the cleaned displacement maps
 * at offset (margin, margin) of a pre-zeroed [(nx+2m)][(ny+2m)] array, which is what the
 * reference returns (:86).  phi is fp64 so that a phase of ~1e2-1e3 rad keeps its gradient.
 * clamp_px: rays displaced by more than this are dropped; <= 0 selects v2's rule |Dx| > nx,
 * |Dy| > ny (:61-64), 1e3 is v1's (refractionFileNumba.py:46-49). */
int paresis_refract_phi(const float* intensity, const double* phi, float* out,
                        float* dx_pad, float* dy_pad, int nx, int ny, int margin,
                        double distance_m, double energy_kev, double magnification, double pixel_um,
                        double clamp_px, int* flag, paresis_stream stream);

/* One projected-thickness map and its per-energy coefficients, formed in fp64 on the host:
 *   grad_obj / grad_ref : pixels of displacement per metre of 2-pixel thickness difference,
 *                         -delta * z / (h * M) / (2h)    (Sample.py:348 + refractionFileNumba2.py:54-56)
 *                         for the object beam / the reference beam (0 = map not in that beam)
 *   atten               : 2 k beta, 1/m (Sample.py:347); applied to the object beam only */
typedef struct {
    const float* thickness;
    float grad_obj;
    float grad_ref;
    float atten;
} paresis_layer;

/* AnalyticalSample.setWaveRT (Sample.py:285-351) + Experiment.refraction (Experiment.py:255-277)
 * fused for the per-energy loop of computeSampleAndReferenceImages_RT (Experiment.py:463-474):
 *   I_obj = I_in * exp(-sum atten_m t_m),  D_obj = sum grad_obj_m * d(t_m),  out_obj += scatter
 *   I_ref = I_in                          D_ref = sum grad_ref_m * d(t_m),  out_ref += scatter
 * intensity_in may be NULL (uniform `intensity_uniform`, e.g. I0 * flux).  out_ref may be NULL.
 * dx_pad / dy_pad (both or neither; only with out_ref == NULL) receive the cleaned object-beam
 * displacement at (margin, margin) of a pre-zeroed [(nx+2m)][(ny+2m)] array -- the Dx, Dy that
 * Experiment.refraction returns (Experiment.py:492, :526).
 * Thickness is differenced first and scaled after, so uniform layers cancel exactly. */
int paresis_refract_layers(const float* intensity_in, float intensity_uniform,
                           const paresis_layer* layers_host, int n_layers,
                           float* out_obj, float* out_ref, float* dx_pad, float* dy_pad,
                           int nx, int ny, int margin, int* flag, paresis_stream stream);

/* The same kernel with the bookkeeping the per-position pipeline hangs on it, so that a membrane
 * position needs no separate zero-fill or reduction launches:
 *   zero_fill[k]  : [nx][ny] buffers set to 0, pixel by pixel (the accumulators the NEXT hop scatters into);
 *   clear_input   : intensity_in is zeroed once read (it is the scatter target of the next energy);
 *   zero_scalar   : *zero_scalar = 0 (the sum slot a later launch adds to);
 *   sum_ref       : *sum_ref += everything the reference beam deposits inside the image
 *                   (= nx*ny * np.mean(intensityReferenceBeforeDetection), Experiment.py:485-486);
 *   intensity_scale: see below. */
typedef struct {
    float* zero_fill[3];
    int clear_input;
    double* zero_scalar;
    double* sum_ref;
    float intensity_scale;   /* > 0: the nominal beam intensity (e.g. I0 * flux).  Enables the shared-memory tile
                                kernels, which accumulate in 32-bit fixed point with a unit of intensity_scale / 2^19
                                (2^21 .. 2^22 in the strip kernels); rays brighter than 2 x intensity_scale, dimmer than
                                2^9 units, or negative, still take the fp32 path. */
    int mode;                /* 0: out += result, source-owner tiles + REDs (round-1 kernels; honours every field above);
                                1: out  = result  (fastRefraction's own contract: it scatters into fresh zeros,
                                   refractionFileNumba2.py:70,77) -- owner-computes rolling strips, plain stores;
                                2: out += result, owner-computes rolling strips (the owner adds its finished rows).
                                Modes 1 / 2 need intensity_scale and ignore zero_fill / clear_input / zero_scalar. */
    int reach;               /* modes 1 / 2, single beam: 8 or 12 = pixels a ray may move and still take the tiles */
    int throughput;          /* mode 0: 0 = rows per block chosen so that THIS launch fills whole waves (best for a kernel
                                running alone); 1 = full-height tiles, least work per pixel (best when the caller keeps
                                several launches in flight, as paresis_rt_run_positions does: +3.9 % on its job) */
} paresis_refract_extras;

int paresis_refract_layers_ex(const float* intensity_in, float intensity_uniform,
                              const paresis_layer* layers_host, int n_layers,
                              float* out_obj, float* out_ref, float* dx_pad, float* dy_pad,
                              int nx, int ny, int margin, int* flag,
                              const paresis_refract_extras* extras_host, paresis_stream stream);

/* The strip hop (modes 1 / 2 above) for up to PARESIS_MAX_HOP_BATCH membrane positions in ONE launch: the items share
 * the layer coefficients (layers_host[m].grad_obj / grad_ref / atten; its thickness pointers are ignored) and differ in
 * their images.  Experiment.py:463-474 for each item.  `work`: scratch of paresis_refract_hop_work_bytes() bytes for the
 * rays that cannot take the tiles (NULL: taken from the stream-ordered pool for the duration of the call). */
typedef struct {
    const float* intensity_in;                      /* NULL: uniform `intensity_uniform` */
    const float* thickness[PARESIS_MAX_LAYERS];
    float* out_obj;
    float* out_ref;                                 /* NULL: single beam */
    double* sum_ref;                                /* *sum_ref += what the reference beam deposits inside the image; may be NULL */
} paresis_hop_item;

/* The round-1 tile hop (mode 0: out += through dense REDs, with the pipeline bookkeeping of paresis_refract_extras) for up
 * to PARESIS_MAX_HOP_BATCH membrane positions in ONE launch -- at 2048^2 a single position does not fill the GPU (ramp,
 * tail and per-tile set-up are two thirds of the kernel time); a grid of several positions pays them once. */
typedef struct {
    const float* intensity_in;
    const float* thickness[PARESIS_MAX_LAYERS];
    float* out_obj;
    float* out_ref;
    float* zero_fill[3];
    double* zero_scalar;
    double* sum_ref;
} paresis_tile_hop_item;

int paresis_refract_tile_batch(const paresis_tile_hop_item* items_host, int n_items, const paresis_layer* layers_host, int n_layers,
                               float intensity_uniform, float intensity_scale, int clear_input, int nx, int ny, int* flag,
                               paresis_stream stream);

size_t paresis_refract_hop_work_bytes(int nx, int ny, int n_layers, int n_items, int dual, int has_intensity_map, int reach);
int paresis_refract_hop_batch(const paresis_hop_item* items_host, int n_items, const paresis_layer* layers_host, int n_layers,
                              float intensity_uniform, float intensity_scale, int accumulate, int reach, int nx, int ny,
                              void* work, size_t work_bytes, int* flag, paresis_stream stream);

/* The object hop (sample + reference beams, as paresis_refract_layers with out_ref) of up to
 * PARESIS_MAX_GROUP energies of ONE detector bin in a single pass: inside a bin every energy repeats the hop
 * on the same thickness maps and adds to the same accumulators (Experiment.py:448-498, :482-483), so the
 * gradients are formed once and each energy only brings its coefficients and its own object-plane intensity
 * image (which is cleared behind the pass, like paresis_refract_extras.clear_input).
 *   layers[m].thickness must be the same pointers for every energy of the group;
 *   intensity_scale   : nominal beam intensity of that energy (> 0), see paresis_refract_extras;
 *   sum_ref           : *sum_ref += what the reference beam of that energy deposits inside the image (may be NULL). */
#define PARESIS_MAX_GROUP 4
typedef struct {
    paresis_layer layers[PARESIS_MAX_LAYERS];
    int n_layers;
    float* intensity_in;
    float intensity_scale;
    double* sum_ref;
} paresis_group_energy;

int paresis_refract_group(const paresis_group_energy* energies_host, int n_energies,
                          float* out_obj, float* out_ref, int nx, int ny, int* flag, paresis_stream stream);

/* AnalyticalSample.setWaveRT as a stand-alone call (Sample.py:285-351, no dark-field branch):
 * I_out = I_in * exp(-sum atten_m t_m); phi_out = phi_in - sum phase_m t_m (phase_m = k delta_m).
 * phi_in may be NULL (0).  n = pixels. */
int paresis_transmit_rt(const float* intensity_in, const double* phi_in,
                        const float* const* thickness_host, const double* atten_host,
                        const double* phase_host, int n_layers,
                        float* intensity_out, double* phi_out, size_t n, paresis_stream stream);

/* out[k][p] = bias[k] + sum_m weights[k][m] * maps[m][p], k < n_out (1..2), m < n_maps (>= 1, no upper limit);
 * fp64 accumulation, one rounding to fp32.  The per-energy phase / attenuation maps of a sample with more
 * materials than a hop takes (Sample.py:279, :347-348).  weights_host is row-major [n_out][n_maps]; bias_host
 * may be NULL (0).  n = pixels of every map. */
int paresis_mix_maps(const float* const* maps_host, int n_maps, const double* weights_host, const double* bias_host,
                     int n_out, float* const* out_host, size_t n, paresis_stream stream);

/* Experiment.computeSampleAndReferenceImages_RT for one membrane position in ONE call
 * (Experiment.py:407-526).  The host prepares, per spectrum energy, the scalars of the three
 * refraction hops; the library runs the whole launch sequence on `stream`. */
typedef struct {
    float intensity_membrane;  /* I0*flux*air*efficiency*plate*exp(-2k sum(beta t)) of the uniform membrane layers (:451-463) */
    float intensity_propag;    /* I0*flux*air*efficiency*plate: sample-only beam and white field (:490-497) */
    paresis_layer hop1[PARESIS_MAX_LAYERS];    /* membrane -> object plane, distance d2 (:466) */
    int n_hop1;
    paresis_layer hop2[PARESIS_MAX_LAYERS];    /* object -> detector, sample + reference beams, d3 (:473-474) */
    int n_hop2;
    paresis_layer propag[PARESIS_MAX_LAYERS];  /* object -> detector without membrane, d3 (:492) */
    int n_propag;
    int close_bin;             /* run the detector after this energy (:501) */
} paresis_rt_energy;

typedef struct {
    int nx, ny, oversampling, det_x, det_y;
    int first_point;           /* membrane position 0: propagation and white images too (:488, :510-514) */
    int n_energies;
    const paresis_rt_energy* energies_host;
    float* i_bs;               /* [nx][ny] scratch: intensity in the object plane.  Must be ALL ZERO on entry unless
                                  i_bs_dirty is set; it is all zero again when the job has run. */
    float* acc_sample; float* acc_ref; float* acc_propag; float* acc_white;   /* [nx][ny] accumulators (any content) */
    double* means;             /* [n_energies]: SUM over the image of the reference beam of each energy; divide by
                                  nx*ny for np.mean(intensityReferenceBeforeDetection) (:485-486).  May be NULL. */
    float* detect_work;        /* see paresis_detect_counts; may be NULL for ordinary kernel sizes */
    const float* src_kernel; int src_half;
    const float* psf_kernel; int psf_half;
    int noise; uint64_t seed; uint64_t sequence;   /* Poisson stream: image k of bin b uses sequence + 4b + k */
    float* out_sample; float* out_ref; float* out_propag; float* out_white;   /* [n_bins][det_x][det_y].  All NULL: the
                                  energies are accumulated only and close_bin is ignored (the caller runs the detector,
                                  as the energy-sharded path does); acc_white is needed with outputs at position 0 only */
    float* dx_pad; float* dy_pad;   /* optional [(nx+30)][(ny+30)], both or neither: Dx, Dy of the sample-only beam, last
                                       energy (:492) */
    int* flag;
    /* optional timing probe: cudaEvent_t pair recorded around one kernel of the first energy / bin
     * (1 = membrane hop, 2 = sample+reference hop, 3 = detector launch of the first bin); 0 = off */
    int probe; void* probe_start; void* probe_end;
    int i_bs_dirty;            /* i_bs (and i_bs_group) hold garbage: zero them first (extra memsets) */
    float* i_bs_group[PARESIS_MAX_GROUP - 1];   /* optional: further [nx][ny] buffers like i_bs (same all-zero contract).
                                  With k of them, up to k+1 energies of a detector bin share one object hop
                                  (paresis_refract_group); the first NULL entry ends the list, and no entry may
                                  follow it. */
    int positions_per_launch;  /* paresis_rt_run_positions only: > 1 = membrane cut, hops and detector of up to this many
                                  positions (<= n_slots, <= PARESIS_MAX_HOP_BATCH) share ONE launch each (blockIdx.z =
                                  position) on the caller's stream, instead of one launch per position on per-slot
                                  streams.  Needs a sphere field and detector bins of one energy; position 0 (extra
                                  images) always runs on its own.  0 / 1 = off. */
    int throughput;            /* 1 = the hops use full-height tiles (paresis_refract_extras.throughput).  paresis_rt_run_positions
                                  sets it for every position of a call with more than one; a single paresis_rt_run keeps
                                  what the caller put here. */
} paresis_rt_job;

/* Per energy: the membrane hop into i_bs, the object hop into acc_sample / acc_ref (+ means[e]), at position 0 the
 * sample-only hop into acc_propag; at a bin close the detector on 2 or 4 images.  Accumulators start from zero and are
 * zeroed again after each detector run.  Each hop takes 1 .. PARESIS_MAX_LAYERS maps, none of them NULL.  Every argument
 * is checked before the first CUDA call (PARESIS_ERR_ARG). */
int paresis_rt_run(const paresis_rt_job* job_host, paresis_stream stream);

/* Many membrane positions in ONE call: for each position, rasterise its membrane
 * (paresis_raster_spheres) and run the per-energy pipeline (paresis_rt_run), positions dealt
 * round-robin over `n_slots` scratch sets, each on its own stream, so that consecutive positions
 * overlap on the GPU (positions are independent: main.py:63-110).  `stream` is the caller's
 * stream: every slot stream first waits for it, and it waits for every slot stream at the end.
 *
 * `job_host` is the template of paresis_rt_run: its scratch / detect_work / output / means / sequence / first_point /
 * probe event fields are ignored (they come from the slot and the position; with positions_per_launch the template's
 * detect_work serves every position).  A hop1 or hop2 layer whose `thickness` is NULL stands for "the membrane map of
 * this position"; a NULL propag map is an error.  Every argument is checked before the first CUDA call
 * (PARESIS_ERR_ARG), including that no image buffer belongs to two slots; n_positions == 0 does nothing. */
typedef struct {
    const int64_t* offsets_host;   /* [n_layers][2]: the np.random.randint draws of this position (x, y) */
    float* thickness;              /* [nx][ny] out: membrane grain map, metres */
    float* out_sample; float* out_ref; float* out_propag; float* out_white;   /* [n_bins][det_x][det_y] */
    double* means;                 /* [n_energies] or NULL */
    uint64_t sequence;
    int first_point;
    void* probe_start; void* probe_end;   /* optional cudaEvent_t pair for job_host->probe (4 = the membrane raster);
                                             a probed position runs alone: the other slots drain first and wait for it */
} paresis_rt_position;

typedef struct {
    float* i_bs; float* acc_sample; float* acc_ref; float* acc_propag; float* acc_white;   /* as in paresis_rt_job */
    void* raster_work; size_t raster_work_bytes;   /* needed only when the membrane has no sphere field: at least
                                                      paresis_raster_work_bytes(n_spheres, n_layers, nx, ny) */
    paresis_stream stream;
    int i_bs_dirty;                /* in/out: cleared once the slot has run a position */
    float* i_bs_group[PARESIS_MAX_GROUP - 1];   /* as in paresis_rt_job */
    float* detect_work;            /* as paresis_rt_job.detect_work, this slot's own (slots run concurrently); may be NULL
                                      for ordinary kernel sizes */
} paresis_rt_slot;

typedef struct {
    const double* spheres; int n_spheres; double pix_um; int n_layers; int margin;   /* see paresis_raster_spheres */
    const float* field; int field_x, field_y;   /* optional sphere field (paresis_raster_field): positions are then
                                                   cut from it (paresis_membrane_from_field) instead of rasterised */
} paresis_membrane;

int paresis_rt_run_positions(const paresis_rt_job* job_host, const paresis_membrane* membrane_host,
                             const paresis_rt_position* positions_host, int n_positions,
                             paresis_rt_slot* slots_host, int n_slots, paresis_stream stream);

/* ---------------------------------------------------------------------------------------
 * Fresnel model
 * ------------------------------------------------------------------------------------- */

/* AnalyticalSample.setWave (Sample.py:248-282): wave *= exp((-i k delta_m - k beta_m) t_m).
 * wave_in may be NULL (uniform real amplitude).  atten_m = k beta_m, phase_m = k delta_m. */
int paresis_transmit_wave(const paresis_c32* wave_in, float amplitude_uniform,
                          const float* const* thickness_host, const double* atten_host,
                          const double* phase_host, int n_layers,
                          paresis_c32* wave_out, size_t n, paresis_stream stream);

typedef struct paresis_fresnel_plan paresis_fresnel_plan;
typedef struct paresis_fresnel_kernel paresis_fresnel_kernel;

/* Experiment.wavePropagation (Experiment.py:219-252): reflect-pad by `margin` (<= 16), FFT at the padded size P = n + 2m,
 * multiply by the separable transfer function, inverse FFT, crop.  Evaluated as what it is -- a circular convolution of
 * period P along each axis, cropped to the n core samples -- with batched 1-D transforms of a convenient length
 * M >= 2n - 1 (a power of two at the benchmark grids, where P = 2 x prime) plus the 2m reflect-margin terms in closed
 * form (csrc/fresnel.cu).  The plan owns the cuFFT line plans, an n x M work buffer and an n x n intermediate. */
int paresis_fresnel_plan_create(int nx, int ny, int margin, paresis_fresnel_plan** plan);
int paresis_fresnel_plan_destroy(paresis_fresnel_plan* plan);
size_t paresis_fresnel_plan_bytes(const paresis_fresnel_plan* plan);

/* hx[nx+2m], hy[ny+2m]: per-axis transfer vectors in FFT (unshifted) order, prepared in fp64
 * on the host: hx[i]*hy[j] = exp(-i z (u_i^2+v_j^2)/(2kM)) / ((nx+2m)(ny+2m))
 * (Experiment.py:243-250; the frequency step uses the UNPADDED size, :246-247).
 * `phase` multiplies the result (the global exp(ikz/M) of :250, or 1).
 * If intensity_acc != NULL the kernel adds |wave|^2 into it (Experiment.py:351-358) and
 * wave_out may be NULL; wave_out may be wave_in. */
int paresis_fresnel_propagate(paresis_fresnel_plan* plan, const paresis_c32* wave_in,
                              const paresis_c32* hx, const paresis_c32* hy, paresis_c32 phase,
                              paresis_c32* wave_out, float* intensity_acc, paresis_stream stream);

/* The same in two steps, for a transfer function that is used more than once (every membrane position of a scan uses
 * the same distances and energies): paresis_fresnel_kernel_create turns (hx, hy) into the convolution kernels of both
 * axes (fp64 on the device, a few small launches on `stream`), paresis_fresnel_convolve propagates with them.  A kernel
 * belongs to plans of the size it was created with (anything else is PARESIS_ERR_ARG); it outlives the plan. */
int paresis_fresnel_kernel_create(paresis_fresnel_plan* plan, const paresis_c32* hx, const paresis_c32* hy, paresis_stream stream,
                                  paresis_fresnel_kernel** kernel);
int paresis_fresnel_kernel_destroy(paresis_fresnel_kernel* kernel);
int paresis_fresnel_convolve(paresis_fresnel_plan* plan, const paresis_c32* wave_in, const paresis_fresnel_kernel* kernel,
                             paresis_c32 phase, paresis_c32* wave_out, float* intensity_acc, paresis_stream stream);

/* The literal chain, kept as a cross-check of the above and for callers that want the padded spectrum: several
 * propagations of the SAME field over different distances (Experiment.py:340-341 and :349 both start from the wave
 * behind the membrane).  paresis_fresnel_spectrum keeps fft2(np.pad(wave, margin, 'reflect')) inside the plan (cuFFT 2-D
 * plan of size P x P and two padded buffers, allocated on first use), paresis_fresnel_from_spectrum applies one transfer
 * function to it, transforms back, crops and delivers like paresis_fresnel_propagate. */
int paresis_fresnel_spectrum(paresis_fresnel_plan* plan, const paresis_c32* wave_in, paresis_stream stream);
int paresis_fresnel_from_spectrum(paresis_fresnel_plan* plan, const paresis_c32* hx, const paresis_c32* hy, paresis_c32 phase,
                                  paresis_c32* wave_out, float* intensity_acc, paresis_stream stream);

/* Experiment.computeSampleAndReferenceImages_Fresnel for one membrane position in ONE call (Experiment.py:279-405).
 * The host prepares, per spectrum energy, the transmission coefficients (fp64) and the three transfer kernels with
 * their global phases exp(ikz/M) (:250); the library runs the whole launch sequence on `stream`. */
typedef struct {
    const float* thickness;
    double atten;              /* k beta, 1/m */
    double phase;              /* k delta, 1/m */
} paresis_wave_layer;

typedef struct {
    float amplitude_membrane;  /* sqrt(I0*flux*air*efficiency*plate) * exp(-k sum(beta u)) of the uniform membrane layers
                                  (:308-338; the plate scales every intensity linearly, :352-356) */
    float amplitude_propag;    /* sqrt(I0*flux*air*efficiency*plate): the sample-only beam (:365) */
    double white;              /* added to the white field of the bin (:372-375): amplitude_propag^2 in fp64 */
    const paresis_wave_layer* membrane_host;   /* the membrane's maps (:338), any number >= 1 */
    int n_membrane;
    paresis_wave_layer sample[PARESIS_MAX_LAYERS];   /* the sample's maps (:344, :365) */
    int n_sample;
    const paresis_fresnel_kernel* reference;   /* membrane -> detector, d2 + d3, magnification (:349) */
    paresis_c32 phase_reference;
    const paresis_fresnel_kernel* to_object;   /* membrane -> object, d2, magMemObj = (d1 + d2) / d1 (:340-341) */
    paresis_c32 phase_to_object;
    const paresis_fresnel_kernel* to_detector; /* object -> detector, d3, magnification (:348, :365) */
    paresis_c32 phase_to_detector;
    int close_bin;             /* run the detector after this energy (:378) */
} paresis_fresnel_energy;

typedef struct {
    paresis_fresnel_plan* plan;          /* nx x ny, the size of every map, wave and accumulator below */
    int oversampling, det_x, det_y;
    int first_point;                     /* membrane position 0: propagation and white images too (:359-375) */
    int n_energies;
    const paresis_fresnel_energy* energies_host;
    paresis_c32* wave_a; paresis_c32* wave_b;   /* [nx][ny] scratch */
    float* acc_sample; float* acc_ref; float* acc_propag; float* acc_white;   /* [nx][ny] accumulators (any content);
                                                                                 acc_propag: first_point only, acc_white:
                                                                                 first_point with outputs only */
    double* means;             /* [n_energies]: SUM over the image of |reference beam|^2 of each energy alone, formed
                                  while it is accumulated; divide by nx*ny for the per-energy mean (:351-358).  May be NULL. */
    float* detect_work;        /* see paresis_detect_counts; may be NULL for ordinary kernel sizes */
    const float* src_kernel; int src_half;
    const float* psf_kernel; int psf_half;
    int noise; uint64_t seed; uint64_t sequence;   /* Poisson stream: image k of bin b uses sequence + 4b + k */
    float* out_sample; float* out_ref; float* out_propag; float* out_white;   /* [n_bins][det_x][det_y].  All NULL: the
                                  energies are accumulated only and close_bin is ignored (the caller runs the detector,
                                  as the energy-sharded path does) */
} paresis_fresnel_job;

/* Per energy: transmission through the membrane -> wave_a; wave_a -> detector into acc_ref (+ means[e]); wave_a ->
 * object -> wave_b; transmission through the sample; wave_b -> detector into acc_sample; at position 0 the sample-only
 * beam into acc_propag.  Accumulators start from zero and are zeroed again after each detector run.  Every argument is
 * checked before the first CUDA call (PARESIS_ERR_ARG). */
int paresis_fresnel_run(const paresis_fresnel_job* job_host, paresis_stream stream);

/* Many membrane positions of the Fresnel model in ONE call, as paresis_rt_run_positions does for ray tracing: for each
 * position, its membrane map is cut from the sphere field (paresis_membrane_from_field) or, without a field, rasterised
 * (paresis_raster_spheres) into position.thickness; then the launch sequence of paresis_fresnel_run runs on the slot's
 * stream with the slot's plan and buffers and the position's outputs, means and sequence.  Position p goes to slot
 * p mod n_slots, so that consecutive positions overlap on the GPU.  `stream` is the caller's stream: every slot stream
 * first waits for it, and it waits for every slot stream at the end.
 *
 * `job_host` is the template of paresis_fresnel_run: its plan, wave, accumulator, detect_work, output, means, sequence
 * and first_point fields are ignored (they come from the slot and the position).  A membrane layer whose `thickness` is
 * NULL stands for "the membrane map of this position"; a NULL sample map is an error.  Positions take no probe events.
 * Every argument is checked before the first CUDA call (PARESIS_ERR_ARG); n_positions == 0 does nothing. */
typedef struct {
    paresis_fresnel_plan* plan;                 /* this slot's OWN plan (a plan owns its work buffers): the size of every
                                                   transfer kernel of the job; no two slots may share one */
    paresis_c32* wave_a; paresis_c32* wave_b;   /* [nx][ny] scratch */
    float* acc_sample; float* acc_ref; float* acc_propag; float* acc_white;   /* [nx][ny], any content */
    float* detect_work;                         /* per slot (slots run concurrently); may be NULL as in paresis_fresnel_job */
    void* raster_work; size_t raster_work_bytes;   /* needed only when the membrane has no sphere field: at least
                                                      paresis_raster_work_bytes(n_spheres, n_layers, nx, ny) */
    paresis_stream stream;
} paresis_fresnel_slot;

int paresis_fresnel_run_positions(const paresis_fresnel_job* job_host, const paresis_membrane* membrane_host,
                                  const paresis_rt_position* positions_host, int n_positions,
                                  paresis_fresnel_slot* slots_host, int n_slots, paresis_stream stream);

/* ---------------------------------------------------------------------------------------
 * Detector
 * ------------------------------------------------------------------------------------- */

/* Detector.detection up to (not including) the Poisson draw -- Detector.py:92-110 and the
 * crop of :118: reflect-pad 15*os, source blur (fftconvolve 'same' with
 * create_gaussian_shape(sigma), :96-99), resize = os x os SUM binning (:103, :185-198),
 * PSF blur (:106-108).  Kernels are the separable 1-D factors of create_gaussian_shape
 * (Detector.py:201-220), length 2*half+1, built on the host; half = 0 skips that blur.
 * `work` must hold paresis_detect_work_floats(...) floats.  expect_out[det_x][det_y]. */
size_t paresis_detect_work_floats(int nx, int ny, int oversampling, int det_x, int det_y);
int paresis_detect(const float* image, int nx, int ny, int oversampling, int det_x, int det_y,
                   const float* src_kernel, int src_half, const float* psf_kernel, int psf_half,
                   float* work, float* expect_out, paresis_stream stream);

/* Detector.detection in ONE kernel, Poisson draw included (Detector.py:92-118): the production
 * path.  A thread block stages the window of the oversampled image it needs in shared memory and
 * runs blur+bin, PSF and (noise != 0) the Philox Poisson draw for pixel p = a*det_y + b on chip.
 * `work` is only touched for kernels too wide for shared memory (then it must hold
 * paresis_detect_work_floats floats); it may be NULL otherwise.  out[det_x][det_y]: counts
 * (noise != 0) or the noise-free expectation. */
int paresis_detect_counts(const float* image, int nx, int ny, int oversampling, int det_x, int det_y,
                          const float* src_kernel, int src_half, const float* psf_kernel, int psf_half,
                          float* work, float* out, int noise, uint64_t seed, uint64_t sequence,
                          paresis_stream stream);

/* The same for up to 8 images of one detector (sample, reference, propagation, white:
 * Experiment.py:503-514 calls detection() once per image) in a single launch; image k draws its
 * noise from sequences_host[k]. */
int paresis_detect_counts_multi(const float* const* images_host, float* const* outs_host,
                                const uint64_t* sequences_host, int n_images, int nx, int ny, int oversampling,
                                int det_x, int det_y, const float* src_kernel, int src_half,
                                const float* psf_kernel, int psf_half, float* work, int noise, uint64_t seed,
                                paresis_stream stream);

/* rs.poisson(detectedImage) -- Detector.py:113-115.  Counter-based Philox4x32-10: the draw
 * for pixel p depends only on (seed, sequence, p), so results do not depend on launch shape
 * or on how positions are sharded over GPUs. */
int paresis_poisson(const float* expect, float* counts, size_t n, uint64_t seed, uint64_t sequence,
                    paresis_stream stream);

/* resize(img, sizeX, sizeY) stand-alone -- Detector.py:185-198. */
int paresis_bin_sum(const float* image, int nx, int ny, int size_x, int size_y, float* out,
                    paresis_stream stream);

/* ---------------------------------------------------------------------------------------
 * Geometry (projected thickness maps)
 * ------------------------------------------------------------------------------------- */

/* getMembraneSegmentedFromFile -- Samples/getMembraneFromFile.py:127-161,168: rasterise
 * spherical caps, all layers.  spheres[n][3] = (c0, c1, radius) in micrometres, already
 * rescaled / shifted / tiled (:95-124, done on the host).  offsets_host[layer][2] = the two
 * np.random.randint draws per layer (:139-140), x first.  thickness_out[dim_x][dim_y] is
 * overwritten, in metres.  `work` is device scratch for the list of bounding-box chunks
 * (paresis_raster_work_bytes suggests a size; a list that overflows is still rasterised
 * correctly, only slower). */
size_t paresis_raster_work_bytes(int n_spheres, int n_layers, int dim_x, int dim_y);
int paresis_raster_spheres(const double* spheres, int n_spheres, double pix_um,
                           const int64_t* offsets_host, int n_layers, int dim_x, int dim_y,
                           int margin, float* thickness_out, void* work, size_t work_bytes,
                           paresis_stream stream);

/* The same membrane without re-rasterising it at every position.  getMembraneFromFile.py:139-161 moves
 * the sphere list by INTEGER pixel offsets per layer, so the grain map of a position is a sum of shifted
 * windows of one "sphere field": the caps of the whole (tiled) list on its own canvas.
 *   paresis_raster_field        : field[field_x][field_y] = that canvas, metres (= paresis_raster_spheres with
 *                                 one layer, zero offsets, zero margin); once per experiment.
 *   paresis_membrane_from_field : thickness_out[r][c] = sum_l field[ox_l + margin + r][oy_l + margin + c]
 *                                 (0 outside the field); once per position.
 * Identical to paresis_raster_spheres up to fp32 summation order PROVIDED no grain reaches further than
 * margin/2 pixels (floor(r/pix) + 1 <= margin/2): the reference only accepts grains whose centre lies within
 * margin/2 of the field of view (:151), which then never clips a grain that touches it.  The caller checks
 * that (paresis_b200/geometry.py does) and uses paresis_raster_spheres otherwise. */
int paresis_raster_field(const double* spheres, int n_spheres, double pix_um, int field_x, int field_y,
                         float* field, void* work, size_t work_bytes, paresis_stream stream);
int paresis_membrane_from_field(const float* field, int field_x, int field_y, const int64_t* offsets_host,
                                int n_layers, int margin, int dim_x, int dim_y, float* thickness_out,
                                paresis_stream stream);
/* ... for up to PARESIS_MAX_HOP_BATCH positions in one launch: offsets_host[z] / thickness_out_host[z] as above. */
int paresis_membrane_from_field_batch(const float* field, int field_x, int field_y, const int64_t* const* offsets_host,
                                      float* const* thickness_out_host, int n_items, int n_layers, int margin, int dim_x,
                                      int dim_y, paresis_stream stream);

/* CreateSampleSphere -- Samples/createSampGeom.py:41-53. */
int paresis_sphere_map(double radius_um, int dim_x, int dim_y, double pix_um, float* out,
                       paresis_stream stream);

/* CreateSampleCylindre -- Samples/createSampGeom.py:87-106, including the cv2.warpAffine
 * (imutils.rotate) fixed-point sampling of the rotated 2N x 2N canvas. */
int paresis_cylinder_map(double radius_um, double angle_deg, int dim_x, int dim_y, double pix_um,
                         float* out, paresis_stream stream);

/* CreateSampleSpheresInCylinder (kind 0) / CreateSampleSpheresInParallelepiped (kind 1) --
 * Samples/createSampGeom.py:110-260: two 500 um spheres (materials 0, 1) in a vertical tube (material 2 =
 * tube - spheres; kind 1 is rotated by 15 degrees like imutils.rotate).  out3[3][dim_x][dim_y], metres. */
int paresis_two_sphere_phantom(int kind, int dim_x, int dim_y, double pix_um, float* out3, paresis_stream stream);

/* ---------------------------------------------------------------------------------------
 * Small utilities used by the host shim
 * ------------------------------------------------------------------------------------- */
/* ---------------------------------------------------------------------------------------
 * Dark-field branch of the ray-tracing model
 * --------------------------------------------------------------------------------------- */

/* The scattering-angle map of the Lung / 'cylinder_beeds' model (Sample.py:322-343), already in pixels at
 * the detector (refractionFileNumba2.py:114): df_px = coeff * sqrt(thickness[m]), coeff formed in fp64 on
 * the host = 2 delta sqrt(NsphereVol^(1/3) * 1e6) sqrt(ln(2/delta) + 1) * z / (pixel * M). */
int paresis_df_angle(const float* thickness, double coeff, float* df_px, size_t n, paresis_stream stream);

/* refractionFileNumba2.py:130, :143-146: df_clean = df_px with angles above limit_px (Nx/4) dropped;
 * i_plain = intensity where df_clean == 0 (else 0), i_df = intensity where df_clean != 0 (else 0).
 * intensity may be NULL (uniform `intensity_uniform`). */
int paresis_df_split(const float* intensity, float intensity_uniform, const float* df_px, float limit_px,
                     float* i_plain, float* i_df, float* df_clean, size_t n, paresis_stream stream);

/* refractionFileNumba2.py:171-186: out += for every pixel of `scattered` (the refracted dark-field
 * intensity) its value spread over a normalised Gaussian patch of sigma = df_px/2 at that pixel
 * (gaussian_shape, :14-23); df_px == 0 adds the value in place.  out[nx][ny] is accumulated into. */
int paresis_df_scatter(const float* scattered, const float* df_px, float* out, int nx, int ny, paresis_stream stream);

/* Experiment.computeSampleAndReferenceImages_RT for one membrane position of a scattering sample in ONE call
 * (Experiment.py:407-526 with fastRefractionDF, refractionFileNumba2.py:88-196).  Per energy, on `stream`:
 * paresis_df_angle on the scattering material's map -> `angle`; the membrane hop into i_bs; paresis_df_split of i_bs
 * (limit nx/4) into plain / scattered rays; two dual-beam object hops (hop2 layers): plain -> (acc_sample, acc_ref),
 * scattered -> (moved, acc_ref); paresis_df_scatter(moved, clean, acc_sample).  Both object hops add to means[e], which
 * is therefore the sum of the whole reference beam.  At position 0 the sample-only beam goes through the same split, two
 * single-beam hops (propag layers) and one scatter into acc_propag, and dark_field += dark_field_weight * angle.  At a
 * bin close the detector runs on 2 or 4 images as in paresis_rt_run.  Every argument is checked before the first CUDA
 * call (PARESIS_ERR_ARG). */
typedef struct {
    const float* scatter_map;  /* thickness map (metres) of the material whose angle applies: with several scattering
                                  materials, the last one (Sample.py:322-343 overwrites newDf).  Required. */
    double angle_coeff;        /* df_px = angle_coeff * sqrt(t): 2 delta sqrt(NsphereVol^(1/3) * 1e6) sqrt(ln(2/delta) + 1)
                                  * d3 / (pixel * M), formed in fp64 on the host (refractionFileNumba2.py:114) */
    double dark_field_weight;  /* flux * pixel * M / d3: the angle map of this energy back in radians, weighted by the
                                  spectrum (Experiment.py:491) */
} paresis_df_energy;

typedef struct {
    paresis_rt_job rt;         /* as for paresis_rt_run (out_* all NULL: accumulate only), except that i_bs_group,
                                  positions_per_launch, dx_pad, dy_pad and probe are ignored.  i_bs keeps paresis_rt_run's
                                  contract: all zero on entry unless i_bs_dirty is set, all zero on exit.  The object
                                  hops of each energy must fit in PARESIS_MAX_LAYERS maps (mix the sample's maps
                                  otherwise). */
    const paresis_df_energy* energies_df_host;   /* [rt.n_energies] */
    float* angle;              /* [nx][ny] scratch: the angle map in pixels; holds the last energy's when the job has run */
    float* plain; float* scattered; float* clean; float* moved;   /* [nx][ny] scratch, any content on entry */
    float* dark_field;         /* optional [nx][ny], position 0 only: += sum over the job's energies of
                                  dark_field_weight * angle (radians).  The caller zeroes it. */
} paresis_df_job;

int paresis_df_run(const paresis_df_job* job_host, paresis_stream stream);

/* Many membrane positions of a scattering sample in ONE call, as paresis_rt_run_positions does for a plain sample: for
 * each position, its membrane map is cut from the sphere field (paresis_membrane_from_field) or, without a field,
 * rasterised (paresis_raster_spheres) into position.rt.thickness; then the launch sequence of paresis_df_run runs on the
 * slot's stream with the slot's buffers and the position's outputs, means, sequence and dark-field map.  Position p goes
 * to slot p mod n_slots, so that consecutive positions overlap on the GPU.  `stream` is the caller's stream: every slot
 * stream first waits for it, and it waits for every slot stream at the end.  With more than one position the hops use
 * full-height tiles (paresis_rt_job.throughput = 1), as in paresis_rt_run_positions.
 *
 * `job_host` is the template of paresis_df_run: its i_bs, accumulator, detect_work, output, means, sequence, first_point,
 * scratch and dark_field fields are ignored (they come from the slot and the position).  A hop1 or hop2 layer whose
 * `thickness` is NULL stands for "the membrane map of this position"; a NULL propag or scattering map is an error.
 * Positions take no probe events.  Every argument is checked before the first CUDA call (PARESIS_ERR_ARG), including that
 * no image buffer belongs to two slots; n_positions == 0 does nothing. */
typedef struct {
    float* i_bs; float* acc_sample; float* acc_ref; float* acc_propag; float* acc_white;   /* as in paresis_rt_job */
    float* angle; float* plain; float* scattered; float* clean; float* moved;             /* as in paresis_df_job */
    float* detect_work;                    /* as paresis_rt_job.detect_work, this slot's own (slots run concurrently); may
                                              be NULL for ordinary kernel sizes */
    void* raster_work; size_t raster_work_bytes;   /* needed only when the membrane has no sphere field: at least
                                                      paresis_raster_work_bytes(n_spheres, n_layers, nx, ny) */
    paresis_stream stream;
    int i_bs_dirty;                        /* in/out, as paresis_rt_slot: cleared once the slot has run a position */
} paresis_df_slot;

typedef struct {
    paresis_rt_position rt;                /* probe events must be NULL */
    float* dark_field;                     /* optional [nx][ny], first_point only: += as paresis_df_job.dark_field */
} paresis_df_position;

int paresis_df_run_positions(const paresis_df_job* job_host, const paresis_membrane* membrane_host,
                             const paresis_df_position* positions_host, int n_positions,
                             paresis_df_slot* slots_host, int n_slots, paresis_stream stream);

/* Result transfers (the reference hands back host arrays: Experiment.py:405, :526, main.py:99): an
 * asynchronous device -> pinned-host copy on the library's copy stream, ordered after `producer`.
 * A lane holds the events of one copy in flight; reuse it once paresis_transfer_wait returned. */
int paresis_transfer_lane_create(void** lane_out);
int paresis_transfer_lane_destroy(void* lane);
int paresis_transfer_d2h(void* lane, void* dst_host_pinned, const void* src_device, size_t bytes, paresis_stream producer);
int paresis_transfer_wait(void* lane);

int paresis_fill(float* dst, float value, size_t n, paresis_stream stream);
int paresis_axpy(float* dst, const float* src, float scale, size_t n, paresis_stream stream); /* dst += scale*src */
/* mean of an image (np.mean at Experiment.py:485-486), result to a device double */
int paresis_mean(const float* src, size_t n, double* out, paresis_stream stream);
/* *out += scale * sum(src)  (out is NOT cleared) */
int paresis_sum_scaled(const float* src, size_t n, double scale, double* out, paresis_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* PARESIS_B200_H */
