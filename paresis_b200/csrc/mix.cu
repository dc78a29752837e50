// Per-energy phase / attenuation maps of a sample with more materials than a hop takes (Sample.py:279, :347-348):
// out[k][p] = bias[k] + sum_m w[k][m] * maps[m][p], accumulated in fp64 and rounded to fp32 once.
//
// Bandwidth bound: every material map is read once and both outputs are written in the same pass.  The map pointers and
// weights travel in one small device table; each block stages them through shared memory MIX_CHUNK maps at a time, so
// the number of maps has no upper limit.
#include <string.h>

#include <vector>

#include "common.cuh"

namespace paresis {

constexpr int MIX_THREADS = 256;
constexpr int MIX_CHUNK = 32;    // maps staged in shared memory at a time

struct MixOut {
    float* out[2];
    double bias[2];
};

// table: n_maps pointers, then n_out rows of n_maps weights (doubles).  One thread = 4 consecutive pixels.
template <int NOUT, bool VEC>
__global__ void __launch_bounds__(MIX_THREADS)
mix_maps_kernel(const void* __restrict__ table, int n_maps, MixOut o, size_t n) {
    __shared__ const float* s_map[MIX_CHUNK];
    __shared__ double s_w[NOUT][MIX_CHUNK];
    const float* const* maps = static_cast<const float* const*>(table);
    const double* w = reinterpret_cast<const double*>(maps + n_maps);
    const size_t p0 = 4 * (blockIdx.x * (size_t)MIX_THREADS + threadIdx.x);
    const bool full = p0 + 4 <= n;
    double acc[NOUT][4];
#pragma unroll
    for (int k = 0; k < NOUT; ++k)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[k][j] = o.bias[k];
    for (int c0 = 0; c0 < n_maps; c0 += MIX_CHUNK) {
        const int cn = min(MIX_CHUNK, n_maps - c0);
        __syncthreads();   // the previous chunk is consumed
        if (threadIdx.x < cn) {
            s_map[threadIdx.x] = maps[c0 + threadIdx.x];
#pragma unroll
            for (int k = 0; k < NOUT; ++k) s_w[k][threadIdx.x] = w[(size_t)k * n_maps + c0 + threadIdx.x];
        }
        __syncthreads();
        if (p0 >= n) continue;
#pragma unroll 4
        for (int m = 0; m < cn; ++m) {
            float t[4];
            if (VEC && full) {
                const float4 v = __ldcs(reinterpret_cast<const float4*>(s_map[m] + p0));
                t[0] = v.x; t[1] = v.y; t[2] = v.z; t[3] = v.w;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) t[j] = p0 + j < n ? ld_stream(s_map[m] + p0 + j) : 0.f;
            }
#pragma unroll
            for (int k = 0; k < NOUT; ++k)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[k][j] = fma(s_w[k][m], (double)t[j], acc[k][j]);
        }
    }
    if (p0 >= n) return;
#pragma unroll
    for (int k = 0; k < NOUT; ++k) {
        if (VEC && full) {
            *reinterpret_cast<float4*>(o.out[k] + p0) =
                make_float4((float)acc[k][0], (float)acc[k][1], (float)acc[k][2], (float)acc[k][3]);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (p0 + j < n) o.out[k][p0 + j] = (float)acc[k][j];
        }
    }
}

template <int NOUT>
static void launch_mix(bool vec, const void* table, int n_maps, const MixOut& o, size_t n, cudaStream_t s) {
    const size_t blocks = (n + 4 * (size_t)MIX_THREADS - 1) / (4 * (size_t)MIX_THREADS);
    if (vec)
        mix_maps_kernel<NOUT, true><<<(unsigned)blocks, MIX_THREADS, 0, s>>>(table, n_maps, o, n);
    else
        mix_maps_kernel<NOUT, false><<<(unsigned)blocks, MIX_THREADS, 0, s>>>(table, n_maps, o, n);
}

}  // namespace paresis

using namespace paresis;

extern "C" int paresis_mix_maps(const float* const* maps_host, int n_maps, const double* weights_host, const double* bias_host,
                                int n_out, float* const* out_host, size_t n, paresis_stream stream) {
    if (!maps_host || !weights_host || !out_host) {
        set_last_error("paresis_mix_maps: null pointer (maps, weights or outputs)");
        return PARESIS_ERR_ARG;
    }
    if (n_maps < 1) {
        set_last_error("paresis_mix_maps: need n_maps >= 1, got %d", n_maps);
        return PARESIS_ERR_ARG;
    }
    if (n_out < 1 || n_out > 2) {
        set_last_error("paresis_mix_maps: n_out must be 1 or 2, got %d", n_out);
        return PARESIS_ERR_ARG;
    }
    if ((n + 3) / 4 > (size_t)0x7fffffff * MIX_THREADS) {
        set_last_error("paresis_mix_maps: %zu pixels exceed one launch", n);
        return PARESIS_ERR_ARG;
    }
    MixOut o{};
    bool vec = true;
    for (int k = 0; k < n_out; ++k) {
        if (!out_host[k]) { set_last_error("paresis_mix_maps: null output map %d", k); return PARESIS_ERR_ARG; }
        o.out[k] = out_host[k];
        o.bias[k] = bias_host ? bias_host[k] : 0.0;
        vec = vec && ((uintptr_t)out_host[k] & 15) == 0;
    }
    for (int m = 0; m < n_maps; ++m) {
        if (!maps_host[m]) { set_last_error("paresis_mix_maps: null material map %d", m); return PARESIS_ERR_ARG; }
        vec = vec && ((uintptr_t)maps_host[m] & 15) == 0;
    }
    if (n == 0) return PARESIS_OK;
    // the table: pointers, then the weight rows; staged on the host, copied behind whatever the stream runs, freed in order
    const size_t bytes = sizeof(void*) * (size_t)n_maps + sizeof(double) * (size_t)n_out * n_maps;
    std::vector<unsigned char> host(bytes);
    memcpy(host.data(), maps_host, sizeof(void*) * (size_t)n_maps);
    memcpy(host.data() + sizeof(void*) * (size_t)n_maps, weights_host, sizeof(double) * (size_t)n_out * n_maps);
    cudaStream_t s = (cudaStream_t)stream;
    void* table = nullptr;
    PARESIS_CUDA(cudaMallocAsync(&table, bytes, s));
    PARESIS_CUDA(cudaMemcpyAsync(table, host.data(), bytes, cudaMemcpyHostToDevice, s));
    if (n_out == 1)
        launch_mix<1>(vec, table, n_maps, o, n, s);
    else
        launch_mix<2>(vec, table, n_maps, o, n, s);
    const cudaError_t launched = cudaPeekAtLastError();
    PARESIS_CUDA(cudaFreeAsync(table, s));
    PARESIS_CUDA(launched);
    return PARESIS_OK;
}
