// Fresnel propagator (Experiment.py:219-252, wavePropagation): reflect-pad by 15, FFT at the padded size, separable
// transfer function, inverse FFT, crop.
//
// The reference's answer is tied to the padded size P = N + 30 (the reflect margin and the periodic wrap are part of
// it), and P is 2 x prime at every benchmark grid (4126 = 2 x 2063, 8222 = 2 x 4111): a cuFFT transform of that size
// runs Bluestein, ~7x the cost of a power of two (profiles/r02_summary.md section 7).  The transfer function is
// separable, exp(-i z u^2 / 2kM) * exp(-i z v^2 / 2kM), so the propagation is a circular convolution of period P along
// each axis with the 1-D kernel c = IDFT_P(h), and only the N cropped outputs of each line are wanted:
//     y[s] = sum_{s'} core[s'] c[(s - s') mod P]            (the N core samples: |s - s'| < N, 2N - 1 kernel values)
//          + sum_{t=1..m} core[t] c[s + t]                  (left reflect margin,  x_pad[m - t] = core[t])
//          + sum_{u=0..m-1} core[N-2-u] c[s + 2m - u]       (right reflect margin, x_pad[m + N + u] = core[N-2-u])
// The first sum is a linear convolution that fits a transform of size M >= 2N - 1 -- a power of two (2N) at the
// benchmark grids; the 2m margin terms are added in closed form where the line is read back.  The result is the same
// circular convolution (no truncation of the kernel, no change of the period); c and G = FFT_M(c arranged on
// [-(N-1), N-1]) are formed in fp64 on the device, once per transfer function.  Per axis:
//   * M a power of two in 512 .. 16384 (and within 1.5x of the next 7-smooth length): line_convolve_kernel
//     (fresnel_lines.cuh) takes a line through both transforms and the multiply in shared memory;
//   * otherwise: pad_lines_kernel, batched 1-D cuFFT in place, mul_lines_kernel, cuFFT back;
//   then post_lines_kernel adds the margin terms, applies the global phase, accumulates |.|^2 and writes transposed, so
//   that the second axis is a row pass again.
// paresis_fresnel_spectrum / _from_spectrum keep the literal pad -> fft2 -> transfer -> ifft2 -> crop chain.
#include <cufft.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "common.cuh"
#include "fresnel.cuh"
#include "fresnel_lines.cuh"

struct paresis_fresnel_kernel {
    float2* g[2];     // [0]: along x (lines of the second pass, M_x values), [1]: along y
    float2* c[2];     // the spatial kernels, P_x / P_y values
    float2* g_dr[2];  // g in the digit-reversed, pair-major order of the in-shared-memory transform (axes that use it)
    int len[2], fft_len[2];   // the plan geometry the kernel was prepared for
};

struct paresis_fresnel_plan {
    int nx, ny, margin, nxp, nyp;
    // separable path: axis 1 (y, rows of the wave) first, then axis 0 (x)
    int len[2], period[2], fft_len[2];        // N, P, M per axis
    cufftHandle lines[2];                     // batched 1-D C2C: [1] = nx lines of M_y, [0] = ny lines of M_x
    cufftHandle zp[2], zm[2];                 // 1-D Z2Z of P and of M (kernel preparation)
    bool made_lines[2], made_zp[2], made_zm[2];
    float2* work;                             // max(nx * M_y, ny * M_x)
    float2* mid;                              // ny x nx: the wave after the first pass, transposed
    double2* zbuf;                            // max(P, M) of both axes
    bool fused[2];                            // M is a power of two in [512, 16384]: line_convolve_kernel instead of cuFFT
    int log_m[2];
    float2* tw[2];                            // per-pass twiddle tables of line_convolve_kernel
    paresis_fresnel_kernel own;               // kernels of paresis_fresnel_propagate(hx, hy)
    size_t line_bytes;
    // literal path (spectrum / from_spectrum), created on first use
    bool have_2d;
    cufftHandle fft;
    float2* buf;
    float2* spec;     // spectrum of the last paresis_fresnel_spectrum() input
    size_t work_bytes;
};

namespace paresis {

__device__ __forceinline__ int reflect_idx(int q, int n) {
    if (q < 0) q = -q;
    if (q >= n) q = 2 * (n - 1) - q;
    return q;
}

// np.pad(wave, 15, mode='reflect')  (Experiment.py:236-237)
__global__ void __launch_bounds__(256)
pad_reflect_kernel(const float2* __restrict__ in, int nx, int ny, int m, float2* __restrict__ buf, int nyp) {
    const int yp = blockIdx.x * blockDim.x + threadIdx.x;
    const int xp = blockIdx.y;
    if (yp >= nyp) return;
    buf[(size_t)xp * nyp + yp] = in[(size_t)reflect_idx(xp - m, nx) * ny + reflect_idx(yp - m, ny)];
}

// exp(-i z (u^2+v^2)/(2kM)) * spectrum, with fftshift/ifftshift folded into the vectors (:250),
// out of place: spectrum (kept) -> work buffer
__global__ void __launch_bounds__(256)
transfer_from_kernel(const float2* __restrict__ spec, float2* __restrict__ buf, const float2* __restrict__ hx, const float2* __restrict__ hy,
                     int nyp) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    const int a = blockIdx.y;
    if (b >= nyp) return;
    const float2 p = hx[a], q = hy[b];
    const float2 h = make_float2(p.x * q.x - p.y * q.y, p.x * q.y + p.y * q.x);
    const float2 w = spec[(size_t)a * nyp + b];
    buf[(size_t)a * nyp + b] = make_float2(w.x * h.x - w.y * h.y, w.x * h.y + w.y * h.x);
}

// crop (:251), global phase (:250) and, optionally, |.|^2 accumulation (:351-358)
__global__ void __launch_bounds__(256)
crop_phase_kernel(const float2* __restrict__ buf, int nyp, int m, float2 phase, float2* __restrict__ out,
            float* __restrict__ acc, int ny) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = blockIdx.y;
    if (j >= ny) return;
    const float2 w = buf[(size_t)(i + m) * nyp + (j + m)];
    const float2 r = make_float2(w.x * phase.x - w.y * phase.y, w.x * phase.y + w.y * phase.x);
    const size_t p = (size_t)i * ny + j;
    if (out) out[p] = r;
    if (acc) acc[p] += r.x * r.x + r.y * r.y;
}

// ---- separable path --------------------------------------------------------------------------------------------

// work[l][s] = s < n ? in[l][s] : 0, two complex numbers per thread (n even: 128-bit loads and stores)
__global__ void __launch_bounds__(256)
pad_lines_kernel(const float2* __restrict__ in, int lines, int n, int M, float2* __restrict__ work) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;        // pair index in the line
    const int l = blockIdx.y;
    if (2 * q >= M) return;
    const int s = 2 * q;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (s + 1 < n && (n & 1) == 0) {
        v = *reinterpret_cast<const float4*>(in + (size_t)l * n + s);
    } else {
        if (s < n) { const float2 a = in[(size_t)l * n + s]; v.x = a.x; v.y = a.y; }
        if (s + 1 < n) { const float2 b = in[(size_t)l * n + s + 1]; v.z = b.x; v.w = b.y; }
    }
    *reinterpret_cast<float4*>(work + (size_t)l * M + s) = v;    // M is even, cudaMalloc alignment
}

// work[l][s] *= G[s]
__global__ void __launch_bounds__(256)
mul_lines_kernel(float2* __restrict__ work, const float2* __restrict__ G, int M) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    const int l = blockIdx.y;
    if (2 * q >= M) return;
    float4* w = reinterpret_cast<float4*>(work + (size_t)l * M) + q;
    const float4 g = *(reinterpret_cast<const float4*>(G) + q);
    const float4 v = *w;
    *w = make_float4(v.x * g.x - v.y * g.y, v.x * g.y + v.y * g.x, v.z * g.z - v.w * g.w, v.z * g.w + v.w * g.z);
}

// out[s][l] = (work[l][s] + margin terms) * phase for s < n, transposed through shared memory; the last pass can add
// |.|^2 into acc instead of (or besides) storing the field.  32 lines x 64 samples per block of 32 x 8 threads; a thread
// owns four lines (8 apart) of two samples (32 apart), so that one term costs two 128-bit broadcast loads of margin
// samples and two kernel values for 32 FMAs.  MARGIN > 0: compile-time margin (the loop over the 2m terms unrolls, every
// shared-memory offset is an immediate); MARGIN = 0: run-time margin m.  `sum` (nullable): *sum += the fp64 sum of the
// block's |.|^2 values, the same fp32 values that go into acc (warp shuffle, then one atomicAdd per block).
constexpr int POST_L = 32, POST_S = 64, POST_MAXM = 16;
template <int MARGIN>
__global__ void __launch_bounds__(256)
post_lines_kernel(const float2* __restrict__ work, const float2* __restrict__ in, const float2* __restrict__ c, int lines, int n, int m_rt,
                  int pitch, float2 phase, float2* __restrict__ out, float* __restrict__ acc, double* __restrict__ sum) {
    __shared__ float2 tile[POST_L][POST_S + 1];
    __shared__ __align__(16) float2 edge[2 * POST_MAXM][POST_L];   // [term][slot]: lines ty, ty+8 at slots 2ty, 2ty+1; ty+16, ty+24 at 16+2ty, 17+2ty
    __shared__ float2 cwin[POST_S + 2 * POST_MAXM];
    const int m = MARGIN > 0 ? MARGIN : m_rt;
    const int tx = threadIdx.x, ty = threadIdx.y, tid = ty * 32 + tx;
    const int s0 = blockIdx.x * POST_S, l0 = blockIdx.y * POST_L;
    // the 2m samples of each line that the reflect margins repeat, and the kernel values this tile meets
    for (int k = tid; k < POST_L * 2 * m; k += 256) {
        const int l = k / (2 * m), j = k - l * 2 * m;
        const int src = j < m ? j + 1 : n - 2 - (j - m);
        const int slot = (l & 16) + 2 * (l & 7) + ((l >> 3) & 1);
        PARESIS_BOUND(j, 2 * POST_MAXM); PARESIS_BOUND(slot, POST_L); PARESIS_BOUND(src, n);
        edge[j][slot] = l0 + l < lines ? in[(size_t)(l0 + l) * n + src] : make_float2(0.f, 0.f);
    }
    for (int k = tid; k < POST_S + 2 * m; k += 256) cwin[k] = c[min(s0 + 1 + k, n + 2 * m - 1)];
    __syncthreads();
    float2 v[4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int l = l0 + ty + 8 * i, s = s0 + tx + 32 * h;
            v[i][h] = (s < n && l < lines) ? work[(size_t)l * pitch + s] : make_float2(0.f, 0.f);
        }
    // term j < m: core[j + 1] c[s + j + 1];  term j >= m: core[n - 2 - (j - m)] c[s + 3m - j]
#pragma unroll
    for (int j = 0; j < (MARGIN > 0 ? 2 * MARGIN : 2 * POST_MAXM); ++j) {
        if (MARGIN == 0 && j >= 2 * m) break;
        const int ci = j < m ? tx + j : tx + 3 * m - j - 1;
        PARESIS_BOUND(ci, POST_S + 2 * POST_MAXM - 32); PARESIS_BOUND(ci + 32, POST_S + 2 * m);
        const float2 cv[2] = {cwin[ci], cwin[ci + 32]};
        const float4 ea = *reinterpret_cast<const float4*>(&edge[j][2 * ty]), eb = *reinterpret_cast<const float4*>(&edge[j][16 + 2 * ty]);
        const float2 e[4] = {make_float2(ea.x, ea.y), make_float2(ea.z, ea.w), make_float2(eb.x, eb.y), make_float2(eb.z, eb.w)};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                v[i][h].x = fmaf(e[i].x, cv[h].x, fmaf(-e[i].y, cv[h].y, v[i][h].x));
                v[i][h].y = fmaf(e[i].x, cv[h].y, fmaf(e[i].y, cv[h].x, v[i][h].y));
            }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int h = 0; h < 2; ++h) tile[ty + 8 * i][tx + 32 * h] = v[i][h];
    __syncthreads();
    double part = 0.0;
#pragma unroll
    for (int i = 0; i < POST_S / 8; ++i) {
        const int so = s0 + ty + 8 * i, lo = l0 + tx;
        if (so < n && lo < lines) {
            const float2 w = tile[tx][ty + 8 * i];
            const float2 r = make_float2(w.x * phase.x - w.y * phase.y, w.x * phase.y + w.y * phase.x);
            const size_t o = (size_t)so * lines + lo;
            const float i2 = r.x * r.x + r.y * r.y;
            if (out) out[o] = r;
            if (acc) acc[o] += i2;
            part += (double)i2;
        }
    }
    if (sum) {
        // the tile is no longer read: its first row holds the eight warp sums
        __syncthreads();
        for (int o = 16; o > 0; o >>= 1) part += __shfl_down_sync(0xffffffffu, part, o);
        double* warp_sums = reinterpret_cast<double*>(&tile[0][0]);
        if (tx == 0) warp_sums[ty] = part;
        __syncthreads();
        if (tid == 0) {
            double s = 0.0;
            for (int w = 0; w < 8; ++w) s += warp_sums[w];
            atomicAdd(sum, s);
        }
    }
}

// kernel preparation, fp64: h (fp32, unshifted order, 1/P folded in) -> c = IDFT_P(h) -> g on [-(n-1), n-1] -> G = FFT_M(g)/M
__global__ void widen_kernel(const float2* __restrict__ h, int P, double2* __restrict__ z) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a < P) z[a] = make_double2((double)h[a].x, (double)h[a].y);
}
__global__ void arrange_kernel(const double2* __restrict__ cz, int n, int P, int M, double2* __restrict__ g, float2* __restrict__ c32) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < P) c32[k] = make_float2((float)cz[k].x, (float)cz[k].y);
    if (k < M) {
        // index k of the M-periodic array holds lag d = k (k < n) or d = k - M (k > M - n); nothing in between
        double2 v = make_double2(0.0, 0.0);
        if (k < n) v = cz[k];
        else if (k > M - n) v = cz[k - M + P];
        g[k] = v;
    }
}
__global__ void narrow_kernel(const double2* __restrict__ g, int M, float2* __restrict__ G, float2* __restrict__ G_dr, int log_m) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= M) return;
    G[k] = make_float2((float)(g[k].x / M), (float)(g[k].y / M));
    if (G_dr) {
        // position k of the digit-reversed spectrum holds frequency fl_frequency_of(k); the middle pass reads group
        // b = k / R pair by pair, pair h of all groups together
        const int fr = fl_frequency_of(k, log_m), lr = fl_log_mid(log_m), R = 1 << lr, groups = M >> lr;
        const int b = k >> lr, within = k & (R - 1);
        G_dr[((within >> 1) * groups + b) * 2 + (within & 1)] = make_float2((float)(g[fr].x / M), (float)(g[fr].y / M));
    }
}

// Convolution length M >= 2n - 1: the next power of two when that is in the range of the in-shared-memory transform and
// not much longer than the smallest even length with prime factors 2, 3, 5, 7 (cuFFT's fast radices), else the latter.
static int conv_length(int n) {
    int smooth = (2 * n - 1 + 1) & ~1;
    for (;; smooth += 2) {
        int r = smooth;
        for (int q : {2, 3, 5, 7}) while (r % q == 0) r /= q;
        if (r == 1) break;
    }
    int pow2 = 512;
    while (pow2 < 2 * n - 1) pow2 *= 2;
    return (pow2 <= 16384 && 2 * pow2 <= 3 * smooth) ? pow2 : smooth;
}

template <int LOG_M>
static int launch_line_convolve(const float2* in, int lines, int n, const float2* tw, const float2* g_dr, float2* out, cudaStream_t s) {
    static bool configured[32] = {false};     // per device
    int dev = 0;
    PARESIS_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 32) dev = 0;
    const size_t smem = fl_smem_bytes(LOG_M);
    if (!configured[dev]) {
        PARESIS_CUDA(cudaFuncSetAttribute(line_convolve_kernel<LOG_M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured[dev] = true;
    }
    line_convolve_kernel<LOG_M><<<lines, fl_threads(LOG_M), smem, s>>>(in, n, tw, reinterpret_cast<const float4*>(g_dr), out);
    PARESIS_LAUNCH_CHECK("line_convolve_kernel");
    return PARESIS_OK;
}

static int fft_error(cufftResult r, const char* what) {
    set_last_error("%s failed (cuFFT code %d)", what, (int)r);
    return PARESIS_ERR_CUFFT;
}

static int kernel_alloc(const paresis_fresnel_plan* p, paresis_fresnel_kernel* k) {
    for (int ax = 0; ax < 2; ++ax) { k->g[ax] = nullptr; k->c[ax] = nullptr; k->g_dr[ax] = nullptr; k->len[ax] = p->len[ax]; k->fft_len[ax] = p->fft_len[ax]; }
    for (int ax = 0; ax < 2; ++ax) {
        PARESIS_CUDA(cudaMalloc(&k->g[ax], sizeof(float2) * p->fft_len[ax]));
        PARESIS_CUDA(cudaMalloc(&k->c[ax], sizeof(float2) * p->period[ax]));
        if (p->fused[ax]) PARESIS_CUDA(cudaMalloc(&k->g_dr[ax], sizeof(float2) * p->fft_len[ax]));
    }
    return PARESIS_OK;
}
static void kernel_free(paresis_fresnel_kernel* k) {
    for (int ax = 0; ax < 2; ++ax) {
        if (k->g[ax]) cudaFree(k->g[ax]);
        if (k->c[ax]) cudaFree(k->c[ax]);
        if (k->g_dr[ax]) cudaFree(k->g_dr[ax]);
        k->g[ax] = k->c[ax] = k->g_dr[ax] = nullptr;
    }
}

static int kernel_fill(paresis_fresnel_plan* p, const float2* hx, const float2* hy, paresis_fresnel_kernel* k, cudaStream_t s) {
    const float2* h[2] = {hx, hy};
    for (int ax = 0; ax < 2; ++ax) {
        const int n = p->len[ax], P = p->period[ax], M = p->fft_len[ax];
        double2* cz = p->zbuf;
        double2* gz = p->zbuf + P;
        widen_kernel<<<(P + 255) / 256, 256, 0, s>>>(h[ax], P, cz);
        PARESIS_LAUNCH_CHECK("widen_kernel");
        cufftResult r = cufftSetStream(p->zp[ax], s);
        if (r == CUFFT_SUCCESS) r = cufftExecZ2Z(p->zp[ax], (cufftDoubleComplex*)cz, (cufftDoubleComplex*)cz, CUFFT_INVERSE);
        if (r != CUFFT_SUCCESS) return fft_error(r, "cufftExecZ2Z (kernel, period)");
        const int top = P > M ? P : M;
        arrange_kernel<<<(top + 255) / 256, 256, 0, s>>>(cz, n, P, M, gz, k->c[ax]);
        PARESIS_LAUNCH_CHECK("arrange_kernel");
        r = cufftSetStream(p->zm[ax], s);
        if (r == CUFFT_SUCCESS) r = cufftExecZ2Z(p->zm[ax], (cufftDoubleComplex*)gz, (cufftDoubleComplex*)gz, CUFFT_FORWARD);
        if (r != CUFFT_SUCCESS) return fft_error(r, "cufftExecZ2Z (kernel, convolution length)");
        narrow_kernel<<<(M + 255) / 256, 256, 0, s>>>(gz, M, k->g[ax], p->fused[ax] ? k->g_dr[ax] : nullptr, p->log_m[ax]);
        PARESIS_LAUNCH_CHECK("narrow_kernel");
    }
    return PARESIS_OK;
}

static int launch_post(dim3 grid, const float2* work, const float2* in, const float2* c, int lines, int n, int m, int pitch, float2 phase,
                       float2* out, float* acc, double* sum, cudaStream_t s) {
    if (m == 15) post_lines_kernel<15><<<grid, dim3(32, 8), 0, s>>>(work, in, c, lines, n, m, pitch, phase, out, acc, sum);
    else post_lines_kernel<0><<<grid, dim3(32, 8), 0, s>>>(work, in, c, lines, n, m, pitch, phase, out, acc, sum);
    PARESIS_LAUNCH_CHECK("post_lines_kernel");
    return PARESIS_OK;
}

// one axis: `lines` lines of n samples (row-major `in`) -> out[s][l]
static int convolve_axis(paresis_fresnel_plan* p, int ax, const float2* in, int lines, const paresis_fresnel_kernel* k, float2 phase,
                         float2* out, float* acc, double* sum, cudaStream_t s) {
    const int n = p->len[ax], M = p->fft_len[ax], m = p->margin;
    const dim3 gt((n + POST_S - 1) / POST_S, (lines + POST_L - 1) / POST_L);
    if (p->fused[ax]) {
        int rc;
        switch (p->log_m[ax]) {
            case 9: rc = launch_line_convolve<9>(in, lines, n, p->tw[ax], k->g_dr[ax], p->work, s); break;
            case 10: rc = launch_line_convolve<10>(in, lines, n, p->tw[ax], k->g_dr[ax], p->work, s); break;
            case 11: rc = launch_line_convolve<11>(in, lines, n, p->tw[ax], k->g_dr[ax], p->work, s); break;
            case 12: rc = launch_line_convolve<12>(in, lines, n, p->tw[ax], k->g_dr[ax], p->work, s); break;
            case 13: rc = launch_line_convolve<13>(in, lines, n, p->tw[ax], k->g_dr[ax], p->work, s); break;
            default: rc = launch_line_convolve<14>(in, lines, n, p->tw[ax], k->g_dr[ax], p->work, s); break;
        }
        if (rc != PARESIS_OK) return rc;
        return launch_post(gt, p->work, in, k->c[ax], lines, n, m, n, phase, out, acc, sum, s);
    }
    const dim3 gl((M / 2 + 255) / 256, lines);
    pad_lines_kernel<<<gl, 256, 0, s>>>(in, lines, n, M, p->work);
    PARESIS_LAUNCH_CHECK("pad_lines_kernel");
    cufftResult r = cufftSetStream(p->lines[ax], s);
    if (r == CUFFT_SUCCESS) r = cufftExecC2C(p->lines[ax], p->work, p->work, CUFFT_FORWARD);
    if (r != CUFFT_SUCCESS) return fft_error(r, "cufftExecC2C forward (lines)");
    mul_lines_kernel<<<gl, 256, 0, s>>>(p->work, k->g[ax], M);
    PARESIS_LAUNCH_CHECK("mul_lines_kernel");
    r = cufftExecC2C(p->lines[ax], p->work, p->work, CUFFT_INVERSE);
    if (r != CUFFT_SUCCESS) return fft_error(r, "cufftExecC2C inverse (lines)");
    return launch_post(gt, p->work, in, k->c[ax], lines, n, m, M, phase, out, acc, sum, s);
}

}  // namespace paresis

// along y: the nx rows of the wave -> mid[ny][nx]; along x: the ny rows of mid -> out[nx][ny] (+ acc, + *sum)
int paresis::fresnel_convolve(paresis_fresnel_plan* p, const float2* wave_in, const paresis_fresnel_kernel* k, float2 phase,
                              float2* wave_out, float* acc, double* sum, cudaStream_t s) {
    const int rc = convolve_axis(p, 1, wave_in, p->nx, k, make_float2(1.f, 0.f), p->mid, nullptr, nullptr, s);
    if (rc != PARESIS_OK) return rc;
    return convolve_axis(p, 0, p->mid, p->ny, k, phase, wave_out, acc, sum, s);
}

bool paresis::fresnel_kernel_fits(const paresis_fresnel_plan* p, const paresis_fresnel_kernel* k) {
    for (int ax = 0; ax < 2; ++ax)
        if (k->len[ax] != p->len[ax] || k->fft_len[ax] != p->fft_len[ax]) return false;
    return true;
}

void paresis::fresnel_plan_dims(const paresis_fresnel_plan* p, int* nx, int* ny) { *nx = p->nx; *ny = p->ny; }

namespace paresis {

static int ensure_2d(paresis_fresnel_plan* p) {
    if (p->have_2d) return PARESIS_OK;
    cufftResult r = cufftCreate(&p->fft);
    if (r == CUFFT_SUCCESS) r = cufftMakePlan2d(p->fft, p->nxp, p->nyp, CUFFT_C2C, &p->work_bytes);
    if (r != CUFFT_SUCCESS) return fft_error(r, "cuFFT 2-D plan");
    PARESIS_CUDA(cudaMalloc(&p->buf, sizeof(float2) * (size_t)p->nxp * p->nyp));
    p->have_2d = true;
    return PARESIS_OK;
}

}  // namespace paresis

using namespace paresis;

extern "C" int paresis_fresnel_plan_create(int nx, int ny, int margin, paresis_fresnel_plan** plan) {
    if (!plan || nx < 2 || ny < 2 || margin < 0 || margin > POST_MAXM || margin > nx - 2 || margin > ny - 2) {
        set_last_error("paresis_fresnel_plan_create: need n >= 2, 0 <= margin <= min(%d, n - 2)", POST_MAXM);
        return PARESIS_ERR_ARG;
    }
    paresis_fresnel_plan* p = new paresis_fresnel_plan();
    p->nx = nx; p->ny = ny; p->margin = margin;
    p->nxp = nx + 2 * margin; p->nyp = ny + 2 * margin;
    p->have_2d = false; p->buf = nullptr; p->spec = nullptr; p->work_bytes = 0;
    p->work = nullptr; p->mid = nullptr; p->zbuf = nullptr;
    for (int ax = 0; ax < 2; ++ax) {
        p->own.g[ax] = p->own.c[ax] = p->own.g_dr[ax] = nullptr;
        p->made_lines[ax] = p->made_zp[ax] = p->made_zm[ax] = false;
        p->fused[ax] = false; p->tw[ax] = nullptr;
    }
    p->len[0] = nx; p->len[1] = ny;
    cufftResult r = CUFFT_SUCCESS;
    size_t line_ws = 0;
    for (int ax = 0; ax < 2 && r == CUFFT_SUCCESS; ++ax) {
        p->period[ax] = p->len[ax] + 2 * margin;
        p->fft_len[ax] = conv_length(p->len[ax]);
        int M = p->fft_len[ax];
        const int batch = ax == 1 ? nx : ny;
        size_t ws = 0;
        p->log_m[ax] = line_fft_log(M);
        p->fused[ax] = p->log_m[ax] != 0;
        if (!p->fused[ax]) {
            r = cufftCreate(&p->lines[ax]);
            p->made_lines[ax] = r == CUFFT_SUCCESS;
            if (r == CUFFT_SUCCESS) r = cufftMakePlanMany(p->lines[ax], 1, &M, nullptr, 1, M, nullptr, 1, M, CUFFT_C2C, batch, &ws);
            line_ws += ws;
        }
        if (r == CUFFT_SUCCESS) { r = cufftPlan1d(&p->zp[ax], p->period[ax], CUFFT_Z2Z, 1); p->made_zp[ax] = r == CUFFT_SUCCESS; }
        if (r == CUFFT_SUCCESS) { r = cufftPlan1d(&p->zm[ax], M, CUFFT_Z2Z, 1); p->made_zm[ax] = r == CUFFT_SUCCESS; }
    }
    const size_t work_elems = std::max((size_t)nx * (p->fused[1] ? ny : p->fft_len[1]), (size_t)ny * (p->fused[0] ? nx : p->fft_len[0]));
    const size_t z_elems = (size_t)std::max(p->period[0], p->period[1]) + (size_t)std::max(p->fft_len[0], p->fft_len[1]);
    cudaError_t e = cudaSuccess;
    if (r == CUFFT_SUCCESS) e = cudaMalloc(&p->work, sizeof(float2) * work_elems);
    if (r == CUFFT_SUCCESS && e == cudaSuccess) e = cudaMalloc(&p->mid, sizeof(float2) * (size_t)nx * ny);
    if (r == CUFFT_SUCCESS && e == cudaSuccess) e = cudaMalloc(&p->zbuf, sizeof(double2) * z_elems);
    int rc = PARESIS_OK;
    if (r != CUFFT_SUCCESS) rc = fft_error(r, "cuFFT line plans");
    else if (e != cudaSuccess) rc = check_cuda(e, "cudaMalloc(fresnel work buffers)");
    else rc = kernel_alloc(p, &p->own);
    for (int ax = 0; ax < 2 && rc == PARESIS_OK; ++ax) {
        if (!p->fused[ax]) continue;
        const int lm = p->log_m[ax], entries = fl_tw_entries(lm);
        std::vector<float2> tw((size_t)entries);
        for (int k = 0; k < fl_outer(lm); ++k) {          // pass k: S = M / 8^k, W = exp(-2 pi i / S), powers 1..4 of W^j
            const int S = 1 << (lm - 3 * k);
            float2* t = tw.data() + fl_tw_offset(lm, k);
            for (int j = 0; j < S / 8; ++j)
                for (int pw = 1; pw <= 4; ++pw) {
                    const double a = -2.0 * 3.14159265358979323846 * (double)((long long)j * pw % S) / (double)S;
                    t[4 * j + pw - 1] = make_float2((float)cos(a), (float)sin(a));
                }
        }
        e = cudaMalloc(&p->tw[ax], sizeof(float2) * entries);
        if (e == cudaSuccess) e = cudaMemcpy(p->tw[ax], tw.data(), sizeof(float2) * entries, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) rc = check_cuda(e, "twiddle table");
    }
    if (rc != PARESIS_OK) {
        paresis_fresnel_plan_destroy(p);
        return rc;
    }
    p->line_bytes = line_ws + sizeof(float2) * (work_elems + (size_t)nx * ny) + sizeof(double2) * z_elems;
    *plan = p;
    return PARESIS_OK;
}

extern "C" int paresis_fresnel_plan_destroy(paresis_fresnel_plan* p) {
    if (!p) return PARESIS_OK;
    for (int ax = 0; ax < 2; ++ax) {
        if (p->made_lines[ax]) cufftDestroy(p->lines[ax]);
        if (p->made_zp[ax]) cufftDestroy(p->zp[ax]);
        if (p->made_zm[ax]) cufftDestroy(p->zm[ax]);
    }
    kernel_free(&p->own);
    for (int ax = 0; ax < 2; ++ax) if (p->tw[ax]) cudaFree(p->tw[ax]);
    if (p->work) cudaFree(p->work);
    if (p->mid) cudaFree(p->mid);
    if (p->zbuf) cudaFree(p->zbuf);
    if (p->have_2d) { cufftDestroy(p->fft); cudaFree(p->buf); }
    if (p->spec) cudaFree(p->spec);
    delete p;
    return PARESIS_OK;
}

extern "C" size_t paresis_fresnel_plan_bytes(const paresis_fresnel_plan* p) {
    if (!p) return 0;
    return p->line_bytes + (p->have_2d ? p->work_bytes + sizeof(float2) * (size_t)p->nxp * p->nyp : 0);
}

extern "C" int paresis_fresnel_kernel_create(paresis_fresnel_plan* p, const paresis_c32* hx, const paresis_c32* hy, paresis_stream stream,
                                             paresis_fresnel_kernel** kernel) {
    if (!p || !hx || !hy || !kernel) { set_last_error("paresis_fresnel_kernel_create: null pointer"); return PARESIS_ERR_ARG; }
    paresis_fresnel_kernel* k = new paresis_fresnel_kernel();
    int rc = kernel_alloc(p, k);
    if (rc == PARESIS_OK) rc = kernel_fill(p, (const float2*)hx, (const float2*)hy, k, (cudaStream_t)stream);
    if (rc != PARESIS_OK) { kernel_free(k); delete k; return rc; }
    *kernel = k;
    return PARESIS_OK;
}

extern "C" int paresis_fresnel_kernel_destroy(paresis_fresnel_kernel* k) {
    if (!k) return PARESIS_OK;
    kernel_free(k);
    delete k;
    return PARESIS_OK;
}

extern "C" int paresis_fresnel_convolve(paresis_fresnel_plan* p, const paresis_c32* wave_in, const paresis_fresnel_kernel* kernel,
                                        paresis_c32 phase, paresis_c32* wave_out, float* intensity_acc, paresis_stream stream) {
    if (!p || !wave_in || !kernel || (!wave_out && !intensity_acc)) {
        set_last_error("paresis_fresnel_convolve: null pointer");
        return PARESIS_ERR_ARG;
    }
    if (!fresnel_kernel_fits(p, kernel)) {
        set_last_error("paresis_fresnel_convolve: the kernel was prepared for a %d x %d plan, this one is %d x %d", kernel->len[0],
                       kernel->len[1], p->len[0], p->len[1]);
        return PARESIS_ERR_ARG;
    }
    return fresnel_convolve(p, (const float2*)wave_in, kernel, make_float2(phase.re, phase.im), (float2*)wave_out, intensity_acc, nullptr,
                            (cudaStream_t)stream);
}

extern "C" int paresis_fresnel_propagate(paresis_fresnel_plan* p, const paresis_c32* wave_in,
                                         const paresis_c32* hx, const paresis_c32* hy, paresis_c32 phase,
                                         paresis_c32* wave_out, float* intensity_acc, paresis_stream stream) {
    if (!p || !wave_in || !hx || !hy || (!wave_out && !intensity_acc)) {
        set_last_error("paresis_fresnel_propagate: null pointer");
        return PARESIS_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const int rc = kernel_fill(p, (const float2*)hx, (const float2*)hy, &p->own, s);
    if (rc != PARESIS_OK) return rc;
    return fresnel_convolve(p, (const float2*)wave_in, &p->own, make_float2(phase.re, phase.im), (float2*)wave_out, intensity_acc, nullptr, s);
}

// Two propagations of the SAME field over different distances (Experiment.py:340-341 and :349 both start from the wave
// behind the membrane) share their reflect-pad and forward FFT: paresis_fresnel_spectrum() keeps fft2(pad(wave)) in the
// plan, paresis_fresnel_from_spectrum() applies a transfer function to it (out of place), transforms back and crops.
// On the Bluestein sizes this path is made of (4126 = 2 x 2063, 8222 = 2 x 4111) a 2-D transform is ~45 % of a
// propagation, so a position with three propagations saves one transform in six.
extern "C" int paresis_fresnel_spectrum(paresis_fresnel_plan* p, const paresis_c32* wave_in, paresis_stream stream) {
    if (!p || !wave_in) { set_last_error("paresis_fresnel_spectrum: null pointer"); return PARESIS_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    const int rc2 = ensure_2d(p);
    if (rc2 != PARESIS_OK) return rc2;
    if (!p->spec) PARESIS_CUDA(cudaMalloc(&p->spec, sizeof(float2) * (size_t)p->nxp * p->nyp));
    const dim3 gp((p->nyp + 255) / 256, p->nxp);
    pad_reflect_kernel<<<gp, 256, 0, s>>>((const float2*)wave_in, p->nx, p->ny, p->margin, p->spec, p->nyp);
    PARESIS_LAUNCH_CHECK("pad_reflect_kernel");
    cufftResult r = cufftSetStream(p->fft, s);
    if (r == CUFFT_SUCCESS) r = cufftExecC2C(p->fft, p->spec, p->spec, CUFFT_FORWARD);
    if (r != CUFFT_SUCCESS) { set_last_error("cufftExecC2C forward failed (code %d)", (int)r); return PARESIS_ERR_CUFFT; }
    return PARESIS_OK;
}

extern "C" int paresis_fresnel_from_spectrum(paresis_fresnel_plan* p, const paresis_c32* hx, const paresis_c32* hy, paresis_c32 phase,
                                             paresis_c32* wave_out, float* intensity_acc, paresis_stream stream) {
    if (!p || !p->spec || !hx || !hy || (!wave_out && !intensity_acc)) {
        set_last_error("paresis_fresnel_from_spectrum: null pointer, or no spectrum stored (call paresis_fresnel_spectrum first)");
        return PARESIS_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const dim3 gp((p->nyp + 255) / 256, p->nxp), gc((p->ny + 255) / 256, p->nx);
    transfer_from_kernel<<<gp, 256, 0, s>>>(p->spec, p->buf, (const float2*)hx, (const float2*)hy, p->nyp);
    PARESIS_LAUNCH_CHECK("transfer_from_kernel");
    cufftResult r = cufftSetStream(p->fft, s);
    if (r == CUFFT_SUCCESS) r = cufftExecC2C(p->fft, p->buf, p->buf, CUFFT_INVERSE);
    if (r != CUFFT_SUCCESS) { set_last_error("cufftExecC2C inverse failed (code %d)", (int)r); return PARESIS_ERR_CUFFT; }
    crop_phase_kernel<<<gc, 256, 0, s>>>(p->buf, p->nyp, p->margin, make_float2(phase.re, phase.im), (float2*)wave_out, intensity_acc, p->ny);
    PARESIS_LAUNCH_CHECK("crop_phase_kernel");
    return PARESIS_OK;
}
