// Training-side helpers of the float layer API (fastpcc_b200/autograd.py): the transposed neighbour table that the
// dgrad of a sparse / transposed convolution runs on, and the backward of an activation fused into a conv epilogue.
// Both are memory-bound single passes with no host synchronisation, so a training step that builds fresh kernel maps
// for every batch (MinkowskiEngine's per-batch coordinate manager) does not stall on them.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace fpcc {

// tt[k, table[k, m] - 1] = m + 1.  One thread per (output row, offset): the table read is coalesced, the store is a
// scatter.  Each (offset, input row) pair has at most one output row (the caller's precondition), so no two threads
// write one entry and the result does not depend on the order in which they run.
__global__ void __launch_bounds__(256) kmap_transpose_kernel(const int32_t *__restrict__ table, int n_out, int64_t ld, int n_in,
                                                             int32_t *__restrict__ tt, int64_t ld_t) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    const int k = blockIdx.y;
    if (m >= n_out) return;
    const int32_t v = __ldg(&table[(int64_t)k * ld + m]);
    if (v > 0 && v <= n_in) tt[(int64_t)k * ld_t + (v - 1)] = m + 1;
}

// element types: 0 fp16, 1 bf16, 2 fp32 (the out_type codes of fpcc_spconv_f16)
__device__ __forceinline__ float load_as_float(const void *p, int type, int64_t i) {
    if (type == 0) return __half2float(reinterpret_cast<const __half *>(p)[i]);
    if (type == 1) return __bfloat162float(reinterpret_cast<const __nv_bfloat16 *>(p)[i]);
    return reinterpret_cast<const float *>(p)[i];
}

constexpr int AG_ROWS = 256;  // rows per CTA: one fp64 partial row of the bias gradient per CTA

// dz[r, j] = dy[r, j] * act'(y[r, j]) rounded once to the compute dtype (0 in the pad columns c <= j < c_pad), and
// the column sums of the unrounded fp32 products per CTA in fp64.  Block (32, 8): threadIdx.x = column within a
// 32-column slice, threadIdx.y = row lane; each thread sums its rows in ascending order, the 8 lanes meet in a fixed
// order in shared memory, so the partial row does not depend on scheduling.
__global__ void __launch_bounds__(256) act_grad_kernel(const void *__restrict__ dy, int dy_type, int64_t ld_dy,
                                                       const void *__restrict__ y, int y_type, int64_t ld_y, int64_t n, int c,
                                                       int act, float slope, void *__restrict__ dz, int dz_type, int c_pad,
                                                       double *__restrict__ partial) {
    __shared__ double red[8][32];
    const int j = blockIdx.y * 32 + threadIdx.x;
    const int64_t r0 = (int64_t)blockIdx.x * AG_ROWS;
    const int64_t r1 = r0 + AG_ROWS < n ? r0 + AG_ROWS : n;
    double acc = 0.0;
    if (j < c_pad) {
        for (int64_t r = r0 + threadIdx.y; r < r1; r += 8) {
            float d = 0.f;
            if (j < c) {
                const float g = load_as_float(dy, dy_type, r * ld_dy + j);
                if (act == 0) {
                    d = g;
                } else {
                    // Y > 0 <=> pre-activation > 0 for ReLU and for LeakyReLU with slope >= 0; at 0 both derivative
                    // conventions agree with torch's (slope)
                    const float v = load_as_float(y, y_type, r * ld_y + j);
                    d = g * (v > 0.f ? 1.f : slope);
                }
                acc += (double)d;
            }
            if (dz_type == 0) reinterpret_cast<__half *>(dz)[r * c_pad + j] = __float2half_rn(d);
            else reinterpret_cast<__nv_bfloat16 *>(dz)[r * c_pad + j] = __float2bfloat16_rn(d);
        }
    }
    if (partial == nullptr) return;
    red[threadIdx.y][threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.y == 0 && j < c) {
        double s = red[0][threadIdx.x];
#pragma unroll
        for (int q = 1; q < 8; ++q) s += red[q][threadIdx.x];
        partial[(int64_t)blockIdx.x * c + j] = s;
    }
}

// dbias[j] = sum over the CTAs' partial rows, one CTA per column: strided sums in ascending order, then a fixed tree.
__global__ void __launch_bounds__(256) act_grad_bias_kernel(const double *__restrict__ partial, int n_parts, int c,
                                                            float *__restrict__ dbias) {
    __shared__ double red[256];
    const int j = blockIdx.x;
    double s = 0.0;
    for (int b = threadIdx.x; b < n_parts; b += 256) s += partial[(int64_t)b * c + j];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) dbias[j] = (float)red[0];
}

}  // namespace fpcc

using namespace fpcc;

extern "C" int fpcc_kmap_transpose(const int32_t *table, int kvol, int n_out, int64_t ld, int n_in, int32_t *tt, int64_t ld_t,
                                   void *stream) {
    FPCC_REQUIRE(table && tt, "kmap_transpose: NULL pointer");
    FPCC_REQUIRE(kvol > 0 && kvol <= 65535, "kmap_transpose: kvol %d must be in 1..65535", kvol);
    FPCC_REQUIRE(n_out >= 0 && n_in >= 0, "kmap_transpose: negative row count");
    FPCC_REQUIRE(ld >= n_out && ld_t >= n_in, "kmap_transpose: row pitch below the row count");
    if (n_in == 0) return FPCC_OK;
    cudaStream_t s = (cudaStream_t)stream;
    FPCC_CUDA(cudaMemset2DAsync(tt, (size_t)ld_t * sizeof(int32_t), 0, (size_t)n_in * sizeof(int32_t), kvol, s));
    if (n_out == 0) return FPCC_OK;
    kmap_transpose_kernel<<<dim3(ceil_div(n_out, 256), kvol), 256, 0, s>>>(table, n_out, ld, n_in, tt, ld_t);
    FPCC_LAUNCH_CHECK();
    return FPCC_OK;
}

extern "C" size_t fpcc_act_grad_workspace(int64_t n, int c) {
    if (n < 1 || c < 1) return 256;
    return (((size_t)((n + AG_ROWS - 1) / AG_ROWS) * (size_t)c * sizeof(double)) + 255) & ~(size_t)255;
}

extern "C" int fpcc_act_grad_f16(const void *dy, int dy_type, int64_t ld_dy, const void *y, int y_type, int64_t ld_y, int64_t n,
                                 int c, int act, float slope, void *dz, int dz_type, int c_pad, float *dbias, void *workspace,
                                 size_t workspace_bytes, void *stream) {
    FPCC_REQUIRE(dy && dz, "act_grad_f16: NULL pointer");
    FPCC_REQUIRE(act >= 0 && act <= 2, "act_grad_f16: unknown activation %d", act);
    FPCC_REQUIRE(act == 0 || y, "act_grad_f16: the activation needs its forward output y");
    FPCC_REQUIRE(act != 2 || (slope >= 0.f && slope <= 3.4e38f), "act_grad_f16: LeakyReLU slope must be finite and >= 0");
    FPCC_REQUIRE(dy_type >= 0 && dy_type <= 2 && y_type >= 0 && y_type <= 2, "act_grad_f16: dy / y types must be 0..2");
    FPCC_REQUIRE(dz_type == 0 || dz_type == 1, "act_grad_f16: dz type must be 0 (fp16) or 1 (bf16)");
    FPCC_REQUIRE(n >= 0 && n <= ((int64_t)INT32_MAX) * AG_ROWS, "act_grad_f16: bad row count");
    FPCC_REQUIRE(c > 0 && c_pad >= c && c_pad <= 65536, "act_grad_f16: need 0 < c <= c_pad <= 65536");
    FPCC_REQUIRE(ld_dy >= c && (act == 0 || ld_y >= c), "act_grad_f16: row pitch below the channel count");
    FPCC_REQUIRE(!dbias || (workspace && workspace_bytes >= fpcc_act_grad_workspace(n, c)), "act_grad_f16: workspace too small");
    cudaStream_t s = (cudaStream_t)stream;
    if (n == 0) {
        if (dbias) FPCC_CUDA(cudaMemsetAsync(dbias, 0, (size_t)c * sizeof(float), s));
        return FPCC_OK;
    }
    const int n_parts = ceil_div(n, AG_ROWS);
    double *partial = dbias ? (double *)workspace : nullptr;
    act_grad_kernel<<<dim3(n_parts, ceil_div(c_pad, 32)), dim3(32, 8), 0, s>>>(dy, dy_type, ld_dy, y, y_type, ld_y, n, c, act, slope,
                                                                              dz, dz_type, c_pad, partial);
    FPCC_LAUNCH_CHECK();
    if (dbias) {
        act_grad_bias_kernel<<<c, 256, 0, s>>>(partial, n_parts, c, dbias);
        FPCC_LAUNCH_CHECK();
    }
    return FPCC_OK;
}
