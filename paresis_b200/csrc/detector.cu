// Detector model: source blur -> os x os sum binning -> PSF blur -> crop, then Poisson noise.
//
// Reference: Detector.py:79-119 (detection), :185-198 (resize), :201-220 (create_gaussian_shape).
// The reference pads by reflection (15*os), convolves with scipy.signal.fftconvolve(mode='same')
// (zero extension beyond the padded frame), bins, convolves again and crops 15 detector pixels.
// create_gaussian_shape is an outer product of a normalised 1-D Gaussian with itself, so both
// blurs are done as exact separable direct convolutions; blur + binning collapse into ONE strided
// pass per axis with the composite kernel W(d) = sum_{a<os} g(d - a).  The reflect padding is
// index arithmetic, never materialised.  Everything is fp32, HBM-bound streaming.
#include <math.h>

#include "detector_common.cuh"
#include "poisson.cuh"

namespace paresis {

__device__ __forceinline__ void build_composite(float* W, const float* __restrict__ g, int half, int os) {
    // W[t], t = d + half, d in [-half, os-1+half]
    const int taps = os + 2 * half;
    for (int t = threadIdx.x; t < taps; t += blockDim.x) {
        const int d = t - half;
        float s = 0.f;
        for (int a = 0; a < os; ++a) {
            const int e = d - a;
            if (e >= -half && e <= half) s += g ? g[e + half] : 1.f;
        }
        W[t] = s;
    }
    __syncthreads();
}

// Pass A: along columns.  T1[xp][v] = sum_d W(d) * P(xp, v*os + d), P = reflect-padded image, 0 outside.
__global__ void __launch_bounds__(DET_THREADS)
blur_bin_cols_kernel(const float* __restrict__ img, int nx, int ny, int os, const float* __restrict__ g, int half,
                     float* __restrict__ T1, int out_cols) {
    __shared__ float W[MAX_TAPS];
    build_composite(W, g, half, os);
    const int v = blockIdx.x * DET_THREADS + threadIdx.x;
    const int xp = blockIdx.y;
    if (v >= out_cols) return;
    const int pad = DET_PAD * os, npy = ny + 2 * pad;
    const float* row = img + (size_t)reflect_index(xp - pad, nx) * ny;
    const int taps = os + 2 * half;
    float acc = 0.f;
    for (int t = 0; t < taps; ++t) {
        const int yp = v * os + t - half;
        if (yp >= 0 && yp < npy) acc = fmaf(W[t], __ldg(row + reflect_index(yp - pad, ny)), acc);
    }
    T1[(size_t)xp * out_cols + v] = acc;
}

// Pass B: along rows.  B[u][v] = sum_d W(d) * T1[u*os + d][v], 0 outside.
__global__ void __launch_bounds__(DET_THREADS)
blur_bin_rows_kernel(const float* __restrict__ T1, int npx, int os, const float* __restrict__ g, int half,
                     float* __restrict__ B, int out_cols) {
    __shared__ float W[MAX_TAPS];
    build_composite(W, g, half, os);
    const int v = blockIdx.x * DET_THREADS + threadIdx.x;
    const int u = blockIdx.y;
    if (v >= out_cols) return;
    const int taps = os + 2 * half;
    float acc = 0.f;
    for (int t = 0; t < taps; ++t) {
        const int xp = u * os + t - half;
        if (xp >= 0 && xp < npx) acc = fmaf(W[t], __ldg(T1 + (size_t)xp * out_cols + v), acc);
    }
    B[(size_t)u * out_cols + v] = acc;
}

// PSF pass along columns with crop: C[u][b] = sum_e g(e) B[u][b + 15 + e], 0 outside [0, in_cols).
__global__ void __launch_bounds__(DET_THREADS)
psf_cols_kernel(const float* __restrict__ B, int in_cols, const float* __restrict__ g, int half,
                float* __restrict__ C, int det_y) {
    const int b = blockIdx.x * DET_THREADS + threadIdx.x;
    const int u = blockIdx.y;
    if (b >= det_y) return;
    float acc = 0.f;
    for (int e = -half; e <= half; ++e) {
        const int v = b + DET_PAD + e;
        if (v >= 0 && v < in_cols) acc = fmaf(__ldg(g + e + half), __ldg(B + (size_t)u * in_cols + v), acc);
    }
    C[(size_t)u * det_y + b] = acc;
}

// PSF pass along rows with crop: out[a][b] = sum_e g(e) C[a + 15 + e][b], 0 outside [0, in_rows).
__global__ void __launch_bounds__(DET_THREADS)
psf_rows_kernel(const float* __restrict__ C, int in_rows, const float* __restrict__ g, int half,
                float* __restrict__ out, int det_y) {
    const int b = blockIdx.x * DET_THREADS + threadIdx.x;
    const int a = blockIdx.y;
    if (b >= det_y) return;
    float acc = 0.f;
    for (int e = -half; e <= half; ++e) {
        const int u = a + DET_PAD + e;
        if (u >= 0 && u < in_rows) acc = fmaf(__ldg(g + e + half), __ldg(C + (size_t)u * det_y + b), acc);
    }
    out[(size_t)a * det_y + b] = acc;
}

__global__ void __launch_bounds__(DET_THREADS)
crop_kernel(const float* __restrict__ B, int in_cols, float* __restrict__ out, int det_y) {
    const int b = blockIdx.x * DET_THREADS + threadIdx.x;
    const int a = blockIdx.y;
    if (b < det_y) out[(size_t)a * det_y + b] = B[(size_t)(a + DET_PAD) * in_cols + b + DET_PAD];
}

// Detector.py:185-198 stand-alone: s = nx / size_x, plain block sums.
__global__ void __launch_bounds__(DET_THREADS)
bin_sum_kernel(const float* __restrict__ img, int nx, int ny, int s, float* __restrict__ out, int sx, int sy) {
    const int b = blockIdx.x * DET_THREADS + threadIdx.x;
    const int a = blockIdx.y;
    if (b >= sy) return;
    float acc = 0.f;
    for (int u = 0; u < s; ++u)
        for (int w = 0; w < s; ++w) {
            const int r = a * s + u, c = b * s + w;
            if (r < nx && c < ny) acc += __ldg(img + (size_t)r * ny + c);
        }
    out[(size_t)a * sy + b] = acc;
}

__global__ void __launch_bounds__(256)
poisson_kernel(const float* __restrict__ expect, float* __restrict__ counts, size_t n, uint64_t seed, uint64_t seq) {
    for (size_t p = blockIdx.x * (size_t)blockDim.x + threadIdx.x; p < n; p += (size_t)gridDim.x * blockDim.x)
        counts[p] = poisson_draw(expect[p], seed, seq, p);
}

// ---------------------------------------------------------------------------------------------
// Fused detector: one kernel from the oversampled image to detector counts.
//
// A block owns a TB x TB tile of detector pixels.  It stages the source window it needs in
// shared memory -- reflect padding resolved by index arithmetic, zeros beyond the padded frame
// exactly like fftconvolve(mode='same') sees them -- then runs blur+bin along columns, along
// rows, the PSF along columns, along rows, and (optionally) the Poisson draw, all on chip.
// Global traffic: the image once (plus the halo re-reads, served by L2) and the counts once.
// ---------------------------------------------------------------------------------------------
constexpr int TB = 32;
constexpr int FUSED_TX = 32, FUSED_TY = 8;
constexpr int FUSED_THREADS = FUSED_TX * FUSED_TY;

struct FusedShape {
    int nx, ny, os, det_x, det_y, src_half, psf_half;
    int bw;      // binned window side   = TB + 2*psf_half
    int sw;      // source window side   = bw*os + 2*src_half
};

// TAPS = os + 2*src_half when it is small (column offsets and weights live in registers);
// TAPS = 0 is the generic version for wider source kernels.
template <bool NOISE, int TAPS>
__global__ void __launch_bounds__(FUSED_THREADS)
detect_fused_kernel(const float* __restrict__ img, FusedShape s, const float* __restrict__ gsrc,
                    const float* __restrict__ gpsf, float* __restrict__ out, uint64_t seed, uint64_t seq) {
    extern __shared__ float smem[];
    float* A = smem;                              // [sw][bw]   blurred+binned along columns
    float* B = A + s.sw * s.bw;                   // [bw][bw]   blurred+binned both ways
    float* C = A;                                 // [bw][TB]   PSF along columns (reuses A)
    float* W = B + s.bw * s.bw;                   // composite kernel, os + 2*src_half taps
    float* P = W + (s.os + 2 * s.src_half);       // PSF kernel, 2*psf_half + 1 taps
    int* rowoff = (int*)(P + 2 * s.psf_half + 1); // [sw] source row offset (elements) or -1 = zero row
    int* queue = rowoff + s.sw;                   // [TB*TB][2] pixels whose Poisson draw needs the full PTRS test
    __shared__ int n_queued;
    if (threadIdx.x == 0 && threadIdx.y == 0) n_queued = 0;
    const int tid = threadIdx.y * FUSED_TX + threadIdx.x;
    const int taps = TAPS > 0 ? TAPS : s.os + 2 * s.src_half;
    const int pad = DET_PAD * s.os, npx = s.nx + 2 * pad, npy = s.ny + 2 * pad;
    const int bxn = s.det_x + 2 * DET_PAD, byn = s.det_y + 2 * DET_PAD;
    // first binned row / column of the window (coordinates of the padded, binned frame)
    const int u0 = blockIdx.y * TB + DET_PAD - s.psf_half, v0 = blockIdx.x * TB + DET_PAD - s.psf_half;
    const int x0 = u0 * s.os - s.src_half, y0 = v0 * s.os - s.src_half;
    for (int t = tid; t < taps; t += FUSED_THREADS) {
        const int d = t - s.src_half;
        float acc = 0.f;
        for (int a = 0; a < s.os; ++a) {
            const int e = d - a;
            if (e >= -s.src_half && e <= s.src_half) acc += gsrc ? gsrc[e + s.src_half] : 1.f;
        }
        W[t] = acc;
    }
    for (int t = tid; t < 2 * s.psf_half + 1; t += FUSED_THREADS) P[t] = gpsf ? gpsf[t] : 1.f;
    for (int a = tid; a < s.sw; a += FUSED_THREADS) {
        const int xp = x0 + a;
        rowoff[a] = (xp >= 0 && xp < npx) ? reflect_index(xp - pad, s.nx) * s.ny : -1;   // nx*ny < 2^30 (checked on the host)
    }
    __syncthreads();

    // blur + bin along columns, straight from global memory (each source pixel is read by <= 2 taps
    // of neighbouring threads: L1 serves the overlap).  A thread keeps one output column: its
    // source columns (reflected, or -1 beyond the padded frame) are fixed for the whole sweep.
    for (int v = threadIdx.x; v < s.bw; v += FUSED_TX) {
        const int yb = y0 + v * s.os;
        if (TAPS > 0) {
            int col[TAPS > 0 ? TAPS : 1];
            float w[TAPS > 0 ? TAPS : 1];
#pragma unroll
            for (int k = 0; k < TAPS; ++k) {
                const int yp = yb + k;
                const bool in = yp >= 0 && yp < npy;
                col[k] = in ? reflect_index(yp - pad, s.ny) : 0;
                w[k] = in ? W[k] : 0.f;
            }
            for (int a = threadIdx.y; a < s.sw; a += FUSED_TY) {
                const int ro = rowoff[a];
                float acc = 0.f;
                if (ro >= 0) {
                    const float* row = img + ro;
#pragma unroll
                    for (int k = 0; k < TAPS; ++k) acc = fmaf(w[k], __ldg(row + col[k]), acc);
                }
                A[a * s.bw + v] = acc;
            }
        } else {
            for (int a = threadIdx.y; a < s.sw; a += FUSED_TY) {
                const int ro = rowoff[a];
                float acc = 0.f;
                if (ro >= 0) {
                    const float* row = img + ro;
                    for (int k = 0; k < taps; ++k) {
                        const int yp = yb + k;
                        if (yp >= 0 && yp < npy) acc = fmaf(W[k], __ldg(row + reflect_index(yp - pad, s.ny)), acc);
                    }
                }
                A[a * s.bw + v] = acc;
            }
        }
    }
    __syncthreads();
    for (int v = threadIdx.x; v < s.bw; v += FUSED_TX) {                    // along rows
        const bool vin = (v0 + v >= 0) & (v0 + v < byn);
        for (int u = threadIdx.y; u < s.bw; u += FUSED_TY) {
            const float* src = A + u * s.os * s.bw + v;
            float acc = 0.f;
            if (TAPS > 0) {
#pragma unroll
                for (int k = 0; k < TAPS; ++k) acc = fmaf(W[k], src[k * s.bw], acc);
            } else {
                for (int k = 0; k < taps; ++k) acc = fmaf(W[k], src[k * s.bw], acc);
            }
            // binned pixels outside the padded frame are the zeros fftconvolve(mode='same') extends with
            const bool in = vin & (u0 + u >= 0) & (u0 + u < bxn);
            B[u * s.bw + v] = in ? acc : 0.f;
        }
    }
    __syncthreads();
    const int np = 2 * s.psf_half + 1;
    for (int u = threadIdx.y; u < s.bw; u += FUSED_TY) {                    // PSF along columns
        const float* src = B + u * s.bw + threadIdx.x;
        float acc = 0.f;
        for (int k = 0; k < np; ++k) acc = fmaf(P[k], src[k], acc);
        C[u * TB + threadIdx.x] = acc;
    }
    __syncthreads();
    const int db = blockIdx.x * TB + threadIdx.x;
    for (int a = threadIdx.y; a < TB; a += FUSED_TY) {                      // PSF along rows, noise, store
        const int da = blockIdx.y * TB + a;
        if (da >= s.det_x || db >= s.det_y) continue;
        const float* src = C + a * TB + threadIdx.x;
        float acc = 0.f;
        for (int k = 0; k < np; ++k) acc = fmaf(P[k], src[k * TB], acc);
        const size_t p = (size_t)da * s.det_y + db;
        if (!NOISE) { out[p] = acc; continue; }
        // ~86 % of the draws finish at the quick acceptance test; the rest are queued so that the
        // expensive tail runs on dense warps instead of dragging every warp through it
        float x;
        if (poisson_quick(acc, seed, seq, p, x)) {
            out[p] = x;
        } else {
            const int slot = atomicAdd(&n_queued, 1);
            queue[2 * slot] = a * TB + threadIdx.x;
            queue[2 * slot + 1] = __float_as_int(acc);
        }
    }
    if (NOISE) {
        __syncthreads();
        for (int qi = tid; qi < n_queued; qi += FUSED_THREADS) {
            const int local = queue[2 * qi];
            const float lam = __int_as_float(queue[2 * qi + 1]);
            const size_t p = (size_t)(blockIdx.y * TB + local / TB) * s.det_y + (blockIdx.x * TB + local % TB);
            out[p] = poisson_slow(lam, seed, seq, p);
        }
    }
}

template <bool NOISE, int TAPS>
static int launch_fused(const float* image, const FusedShape& s, const float* gs, const float* gp, float* out,
                        uint64_t seed, uint64_t seq, size_t smem, cudaStream_t st) {
    static size_t configured[32] = {0};    // per device: the attribute belongs to the device's copy of the kernel
    int dev = 0;
    PARESIS_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 32) dev = 0;
    if (smem > configured[dev]) {
        PARESIS_CUDA(cudaFuncSetAttribute(detect_fused_kernel<NOISE, TAPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured[dev] = smem;
    }
    const dim3 grid(div_up(s.det_y, TB), div_up(s.det_x, TB)), block(FUSED_TX, FUSED_TY);
    detect_fused_kernel<NOISE, TAPS><<<grid, block, smem, st>>>(image, s, gs, gp, out, seed, seq);
    PARESIS_LAUNCH_CHECK("detect_fused_kernel");
    return PARESIS_OK;
}

template <bool NOISE>
static int dispatch_fused(int taps, const float* image, const FusedShape& s, const float* gs, const float* gp, float* out,
                          uint64_t seed, uint64_t seq, size_t smem, cudaStream_t st) {
    (void)taps;   // the sizes PARESIS produces go through detect_tile_kernel; this is the any-size fallback
    return launch_fused<NOISE, 0>(image, s, gs, gp, out, seed, seq, smem, st);
}

}  // namespace paresis

using namespace paresis;

extern "C" size_t paresis_detect_work_floats(int nx, int ny, int os, int det_x, int det_y) {
    const size_t npx = (size_t)nx + 2 * DET_PAD * os;
    const size_t bx = det_x + 2 * DET_PAD, by = det_y + 2 * DET_PAD;
    (void)ny;
    return npx * by + bx * by + bx * (size_t)det_y;
}

extern "C" int paresis_detect(const float* image, int nx, int ny, int os, int det_x, int det_y,
                              const float* src_kernel, int src_half, const float* psf_kernel, int psf_half,
                              float* work, float* expect_out, paresis_stream stream) {
    if (!image || !work || !expect_out || os < 1 || det_x < 1 || det_y < 1) {
        set_last_error("paresis_detect: bad arguments");
        return PARESIS_ERR_ARG;
    }
    if (nx != det_x * os || ny != det_y * os) {
        set_last_error("paresis_detect: study grid %dx%d is not detector %dx%d times oversampling %d", nx, ny, det_x, det_y, os);
        return PARESIS_ERR_ARG;
    }
    if (DET_PAD * os > nx - 1 || DET_PAD * os > ny - 1) {
        set_last_error("paresis_detect: reflect margin %d exceeds the image", DET_PAD * os);
        return PARESIS_ERR_ARG;
    }
    if (src_half < 0 || psf_half < 0 || os + 2 * src_half > MAX_TAPS || (src_half > 0 && !src_kernel) || (psf_half > 0 && !psf_kernel)) {
        set_last_error("paresis_detect: kernel half-widths %d / %d unsupported", src_half, psf_half);
        return PARESIS_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const int pad = DET_PAD * os, npx = nx + 2 * pad;
    const int bx = det_x + 2 * DET_PAD, by = det_y + 2 * DET_PAD;
    float* T1 = work;
    float* B = T1 + (size_t)npx * by;
    float* C = B + (size_t)bx * by;
    const float* g = src_half > 0 ? src_kernel : nullptr;
    blur_bin_cols_kernel<<<dim3(div_up(by, DET_THREADS), npx), DET_THREADS, 0, s>>>(image, nx, ny, os, g, src_half, T1, by);
    PARESIS_LAUNCH_CHECK("blur_bin_cols_kernel");
    blur_bin_rows_kernel<<<dim3(div_up(by, DET_THREADS), bx), DET_THREADS, 0, s>>>(T1, npx, os, g, src_half, B, by);
    PARESIS_LAUNCH_CHECK("blur_bin_rows_kernel");
    if (psf_half > 0) {
        psf_cols_kernel<<<dim3(div_up(det_y, DET_THREADS), bx), DET_THREADS, 0, s>>>(B, by, psf_kernel, psf_half, C, det_y);
        PARESIS_LAUNCH_CHECK("psf_cols_kernel");
        psf_rows_kernel<<<dim3(div_up(det_y, DET_THREADS), det_x), DET_THREADS, 0, s>>>(C, bx, psf_kernel, psf_half, expect_out, det_y);
        PARESIS_LAUNCH_CHECK("psf_rows_kernel");
    } else {
        crop_kernel<<<dim3(div_up(det_y, DET_THREADS), det_x), DET_THREADS, 0, s>>>(B, by, expect_out, det_y);
        PARESIS_LAUNCH_CHECK("crop_kernel");
    }
    return PARESIS_OK;
}

static size_t fused_smem_bytes(const FusedShape& s) {
    const size_t floats = (size_t)s.sw * s.bw + (size_t)s.bw * s.bw + (s.os + 2 * s.src_half) + (2 * s.psf_half + 1) + s.sw
                          + 2 * TB * TB;
    return floats * sizeof(float);
}

static int dispatch_detect_tile(int os, int hs, int hp, PARESIS_DT_ARGS) {
    switch (os) {
        case 1: return dispatch_detect_tile_os1(hs, hp, im, n_images, nx, ny, det_x, det_y, gs, gp, noise, seed, st);
        case 2: return dispatch_detect_tile_os2(hs, hp, im, n_images, nx, ny, det_x, det_y, gs, gp, noise, seed, st);
        case 3: return dispatch_detect_tile_os3(hs, hp, im, n_images, nx, ny, det_x, det_y, gs, gp, noise, seed, st);
        case 4: return dispatch_detect_tile_os4(hs, hp, im, n_images, nx, ny, det_x, det_y, gs, gp, noise, seed, st);
        default: return -1;
    }
}

static int detect_args_ok(int nx, int ny, int os, int det_x, int det_y, const float* src_kernel, int src_half,
                          const float* psf_kernel, int psf_half) {
    return !(os < 1 || det_x < 1 || det_y < 1 || nx != det_x * os || ny != det_y * os ||
             DET_PAD * os > nx - 1 || DET_PAD * os > ny - 1 || src_half < 0 || psf_half < 0 ||
             (src_half > 0 && !src_kernel) || (psf_half > 0 && !psf_kernel) || (long)nx * ny >= (1L << 30));
}

extern "C" int paresis_detect_counts(const float* image, int nx, int ny, int os, int det_x, int det_y,
                                     const float* src_kernel, int src_half, const float* psf_kernel, int psf_half,
                                     float* work, float* out, int noise, uint64_t seed, uint64_t sequence,
                                     paresis_stream stream) {
    if (!image || !out || !detect_args_ok(nx, ny, os, det_x, det_y, src_kernel, src_half, psf_kernel, psf_half)) {
        set_last_error("paresis_detect_counts: bad arguments");
        return PARESIS_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const float* gs = src_half > 0 ? src_kernel : nullptr;
    const float* gp = psf_half > 0 ? psf_kernel : nullptr;
    DetImages im{};
    im.img[0] = image; im.out[0] = out; im.seq[0] = sequence;
    int rc = dispatch_detect_tile(os, src_half, psf_half, im, 1, nx, ny, det_x, det_y, gs, gp, noise, seed, st);
    if (rc >= 0) return rc;
    FusedShape s{nx, ny, os, det_x, det_y, src_half, psf_half, TB + 2 * psf_half, (TB + 2 * psf_half) * os + 2 * src_half};
    const size_t smem = fused_smem_bytes(s);
    if (smem > 200 * 1024) {
        // very wide kernels: separable passes through global memory, then the draw in place
        if (!work) { set_last_error("paresis_detect_counts: this kernel size needs the work buffer"); return PARESIS_ERR_ARG; }
        rc = paresis_detect(image, nx, ny, os, det_x, det_y, src_kernel, src_half, psf_kernel, psf_half, work, out, stream);
        if (rc != PARESIS_OK || !noise) return rc;
        return paresis_poisson(out, out, (size_t)det_x * det_y, seed, sequence, stream);
    }
    const int taps = os + 2 * src_half;
    return noise ? dispatch_fused<true>(taps, image, s, gs, gp, out, seed, sequence, smem, st)
                 : dispatch_fused<false>(taps, image, s, gs, gp, out, seed, sequence, smem, st);
}

extern "C" int paresis_detect_counts_multi(const float* const* images_host, float* const* outs_host,
                                           const uint64_t* sequences_host, int n_images, int nx, int ny, int os,
                                           int det_x, int det_y, const float* src_kernel, int src_half,
                                           const float* psf_kernel, int psf_half, float* work, int noise, uint64_t seed,
                                           paresis_stream stream) {
    if (!images_host || !outs_host || !sequences_host || n_images < 1 || n_images > DT_MAX_IMAGES ||
        !detect_args_ok(nx, ny, os, det_x, det_y, src_kernel, src_half, psf_kernel, psf_half)) {
        set_last_error("paresis_detect_counts_multi: bad arguments (1..%d images)", DT_MAX_IMAGES);
        return PARESIS_ERR_ARG;
    }
    DetImages im{};
    for (int k = 0; k < n_images; ++k) {
        if (!images_host[k] || !outs_host[k]) { set_last_error("paresis_detect_counts_multi: null image %d", k); return PARESIS_ERR_ARG; }
        im.img[k] = images_host[k]; im.out[k] = outs_host[k]; im.seq[k] = sequences_host[k];
    }
    int rc = dispatch_detect_tile(os, src_half, psf_half, im, n_images, nx, ny, det_x, det_y, src_half > 0 ? src_kernel : nullptr,
                                  psf_half > 0 ? psf_kernel : nullptr, noise, seed, (cudaStream_t)stream);
    if (rc >= 0) return rc;
    for (int k = 0; k < n_images; ++k) {   // unusual kernel sizes: one image at a time
        rc = paresis_detect_counts(images_host[k], nx, ny, os, det_x, det_y, src_kernel, src_half, psf_kernel, psf_half, work,
                                   outs_host[k], noise, seed, sequences_host[k], stream);
        if (rc != PARESIS_OK) return rc;
    }
    return PARESIS_OK;
}

extern "C" int paresis_poisson(const float* expect, float* counts, size_t n, uint64_t seed, uint64_t sequence,
                               paresis_stream stream) {
    if (!expect || !counts) { set_last_error("paresis_poisson: null pointer"); return PARESIS_ERR_ARG; }
    size_t blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (blocks < 1) blocks = 1;
    poisson_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(expect, counts, n, seed, sequence);
    PARESIS_LAUNCH_CHECK("poisson_kernel");
    return PARESIS_OK;
}

extern "C" int paresis_bin_sum(const float* image, int nx, int ny, int size_x, int size_y, float* out,
                               paresis_stream stream) {
    if (!image || !out || size_x < 1 || size_y < 1 || nx < size_x) {
        set_last_error("paresis_bin_sum: bad arguments");
        return PARESIS_ERR_ARG;
    }
    const int sfac = nx / size_x;  // Detector.py:192
    bin_sum_kernel<<<dim3(div_up(size_y, DET_THREADS), size_x), DET_THREADS, 0, (cudaStream_t)stream>>>(
        image, nx, ny, sfac, out, size_x, size_y);
    PARESIS_LAUNCH_CHECK("bin_sum_kernel");
    return PARESIS_OK;
}
