// Deep-factorized entropy model (the learned prior of fastpcc_b200/entropy_models.py; DESIGN 3.10).
//
// Definition (the project's own, after tensorflow_compression's DeepFactorized with filters = (3, 3, 3); parity with
// the reference's re-implementation is unpinned).  Per channel c, one row of params [C, 43] in this order:
//     H0[3x1] b0[3] a0[3] | H1[3x3] b1[3] a1[3] | H2[3x3] b2[3] a2[3] | H3[1x3] b3[1]      (H row-major [out][in])
// f_c(x): v = x; for each layer i: v <- softplus(H_i) v + b_i, and for i < 3 also v <- v + tanh(a_i) * tanh(v).
// f_c is monotone increasing (softplus >= 0, |tanh(a)| < 1).
// L_c(y) = |sigmoid(s u) - sigmoid(s l)|, u = f_c(y + 1/2), l = f_c(y - 1/2), s = -1 if u + l > 0 else +1 (both sigmoids in
// the lower tail; unlike -sign() it is never 0).
// bits = -log2(max(L, bound)).  Gradient at the bound: compressai's LowerBound -- dL passes where L >= bound, or where
// the incoming gradient would raise L (d bits / d max(L, bound) < 0, i.e. dbits > 0).
//
// Kernels.  Block 256 over a slice of at most SLICE channels: thread t -> channel t % cb, row lane t / cb (cb = the
// slice's channel count, 256 / cb row lanes), so a warp reads consecutive channels of consecutive rows.  The per-channel
// transforms softplus(H), b, tanh(a) are staged once per CTA in shared memory ([c][43], an odd stride: conflict-free).
// The gradient recomputes the forward at y +- 1/2 in registers (nothing is stored between the passes), writes dy, and
// accumulates the 43 parameter gradients of its elements in fp32 over at most FLUSH elements, then into the thread's
// own fp64 slots in shared memory.  The CTA's row lanes meet in ascending order into one fp64 partial row per
// (part, channel); the parts meet in act_grad_bias_kernel (train.cu): strided sums in ascending order, then a fixed
// tree.  No float atomics: dparams is the same bits run to run.
#include "common.cuh"

namespace fpcc {

// dbias[j] = sum over the partial rows [n_parts, c] in a fixed order (train.cu)
__global__ void act_grad_bias_kernel(const double *__restrict__ partial, int n_parts, int c, float *__restrict__ dbias);

constexpr int NP = 43;          // parameters per channel
constexpr int SLICE = 128;      // channels per CTA slice
constexpr int EM_THREADS = 256;
constexpr int FLUSH = 8;        // elements per fp32 accumulation before the fp64 slots
constexpr int MAX_PARTS = 296;  // row parts of the gradient (2 CTAs on each of 148 SMs per slice)

// 0: softplus(H), 1: b, 2: tanh(a)
__host__ __device__ __forceinline__ int param_kind(int k) {
    if (k >= 39) return k == 42 ? 1 : 0;
    const int base = k < 9 ? 0 : (k < 24 ? 9 : 24);
    const int nh = k < 9 ? 3 : 9;
    const int r = k - base;
    return r < nh ? 0 : (r < nh + 3 ? 1 : 2);
}

__device__ __forceinline__ float softplus_f(float x) { return x > 20.f ? x : log1pf(expf(x)); }

__device__ __forceinline__ float transform_param(float v, int k) {
    const int kind = param_kind(k);
    return kind == 0 ? softplus_f(v) : (kind == 1 ? v : tanhf(v));
}

// Forward of f at x with the transformed row q; keeps what the backward needs (t = tanh of each layer's
// pre-activation, v = each layer's output).
struct FState {
    float t[3][3], v[3][3];
};

template <bool KEEP>
__device__ __forceinline__ float f_eval(const float *q, float x, FState &st) {
    float v[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const float z = fmaf(q[j], x, q[3 + j]);
        const float t = tanhf(z);
        v[j] = fmaf(q[6 + j], t, z);
        if (KEEP) { st.t[0][j] = t; st.v[0][j] = v[j]; }
    }
#pragma unroll
    for (int i = 1; i < 3; ++i) {
        const int base = i == 1 ? 9 : 24;
        float w[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            float z = q[base + 9 + j];
#pragma unroll
            for (int k = 0; k < 3; ++k) z = fmaf(q[base + 3 * j + k], v[k], z);
            const float t = tanhf(z);
            w[j] = fmaf(q[base + 12 + j], t, z);
            if (KEEP) { st.t[i][j] = t; st.v[i][j] = w[j]; }
        }
#pragma unroll
        for (int j = 0; j < 3; ++j) v[j] = w[j];
    }
    float f = q[42];
#pragma unroll
    for (int k = 0; k < 3; ++k) f = fmaf(q[39 + k], v[k], f);
    return f;
}

__device__ __forceinline__ float sigmoid_f(float x) { return 1.f / (1.f + expf(-x)); }

// L_c(y) from u = f(y + 1/2), l = f(y - 1/2); *s_out = s, *d_out = sigmoid(s u) - sigmoid(s l)
__device__ __forceinline__ float likelihood_ul(float u, float l, float *s_out, float *su_out, float *sl_out) {
    const float s = u + l > 0.f ? -1.f : 1.f;
    const float su = sigmoid_f(s * u), sl = sigmoid_f(s * l);
    *s_out = s; *su_out = su; *sl_out = sl;
    return fabsf(su - sl);
}

__device__ __forceinline__ float likelihood(const float *q, float y) {
    FState st;
    const float u = f_eval<false>(q, y + 0.5f, st), l = f_eval<false>(q, y - 0.5f, st);
    float s, su, sl;
    return likelihood_ul(u, l, &s, &su, &sl);
}

// Backward of f at the kept state: acc += g * df/dq (in transformed-parameter space), returns g * df/dx.
__device__ __forceinline__ float f_backward(const float *q, float x, const FState &st, float g, float *acc) {
    float dv[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        acc[39 + k] = fmaf(g, st.v[2][k], acc[39 + k]);
        dv[k] = g * q[39 + k];
    }
    acc[42] += g;
#pragma unroll
    for (int i = 2; i >= 1; --i) {
        const int base = i == 1 ? 9 : 24;
        float dz[3], dprev[3] = {0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const float t = st.t[i][j];
            dz[j] = dv[j] * fmaf(q[base + 12 + j], fmaf(-t, t, 1.f), 1.f);
            acc[base + 12 + j] = fmaf(dv[j], t, acc[base + 12 + j]);
            acc[base + 9 + j] += dz[j];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                acc[base + 3 * j + k] = fmaf(dz[j], st.v[i - 1][k], acc[base + 3 * j + k]);
                dprev[k] = fmaf(dz[j], q[base + 3 * j + k], dprev[k]);
            }
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) dv[k] = dprev[k];
    }
    float dx = 0.f;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const float t = st.t[0][j];
        const float dz = dv[j] * fmaf(q[6 + j], fmaf(-t, t, 1.f), 1.f);
        acc[6 + j] = fmaf(dv[j], t, acc[6 + j]);
        acc[3 + j] += dz;
        acc[j] = fmaf(dz, x, acc[j]);
        dx = fmaf(dz, q[j], dx);
    }
    return dx;
}

// stages the transformed rows of channels [c0, c0 + cb) into q_s[cb][NP]
__device__ __forceinline__ void stage_params(const float *__restrict__ params, int c0, int cb, float *q_s) {
    for (int i = threadIdx.x; i < cb * NP; i += blockDim.x) q_s[i] = transform_param(__ldg(&params[(int64_t)c0 * NP + i]), i % NP);
    __syncthreads();
}

__global__ void __launch_bounds__(EM_THREADS) factorized_bits_kernel(const float *__restrict__ y, int64_t ld_y, int64_t n, int C,
                                                                     const float *__restrict__ params, float bound,
                                                                     int rows_per_cta, float *__restrict__ bits) {
    __shared__ float q_s[SLICE * NP];
    const int c0 = blockIdx.y * SLICE;
    const int cb = min(SLICE, C - c0), rl_n = EM_THREADS / cb;
    stage_params(params, c0, cb, q_s);
    const int cl = threadIdx.x % cb, rl = threadIdx.x / cb;
    if (rl >= rl_n) return;
    const float *q = q_s + cl * NP;
    const int c = c0 + cl;
    const int64_t r0 = (int64_t)blockIdx.x * rows_per_cta;
    const int64_t r1 = min(r0 + rows_per_cta, n);
    for (int64_t r = r0 + rl; r < r1; r += rl_n) {
        const float L = likelihood(q, __ldg(&y[r * ld_y + c]));
        bits[r * C + c] = -log2f(fmaxf(L, bound));
    }
}

__global__ void __launch_bounds__(EM_THREADS) factorized_grad_kernel(const float *__restrict__ y, int64_t ld_y,
                                                                        const float *__restrict__ dbits, int64_t ld_db, int64_t n,
                                                                        int C, const float *__restrict__ params, float bound,
                                                                        int rows_per_part, float *__restrict__ dy,
                                                                        double *__restrict__ partial) {
    __shared__ float q_s[SLICE * NP];
    extern __shared__ double slots[];  // [EM_THREADS][NP]: every thread's own fp64 sums
    const int c0 = blockIdx.y * SLICE;
    const int cb = min(SLICE, C - c0), rl_n = EM_THREADS / cb;
    stage_params(params, c0, cb, q_s);
    const int cl = threadIdx.x % cb, rl = threadIdx.x / cb;
    double *mine = slots + threadIdx.x * NP;
    for (int k = 0; k < NP; ++k) mine[k] = 0.0;
    if (rl < rl_n) {
        const float *q = q_s + cl * NP;
        const int c = c0 + cl;
        const int64_t r0 = (int64_t)blockIdx.x * rows_per_part;
        const int64_t r1 = min(r0 + rows_per_part, n);
        int64_t r = r0 + rl;
        while (r < r1) {
            float acc[NP];
#pragma unroll
            for (int k = 0; k < NP; ++k) acc[k] = 0.f;
            for (int e = 0; e < FLUSH && r < r1; ++e, r += rl_n) {
                const float x = __ldg(&y[r * ld_y + c]);
                const float g = __ldg(&dbits[r * ld_db + c]);
                FState su_st, sl_st;
                const float xu = x + 0.5f, xl = x - 0.5f;
                const float u = f_eval<true>(q, xu, su_st), l = f_eval<true>(q, xl, sl_st);
                float s, sgu, sgl;
                const float L = likelihood_ul(u, l, &s, &sgu, &sgl);
                const float Lb = fmaxf(L, bound);
                // d bits / d Lb = -1 / (Lb ln 2); LowerBound: passes where L >= bound or where it is negative
                float gL = -g / (Lb * 0.69314718055994531f);
                if (!(L >= bound || gL < 0.f)) gL = 0.f;
                const float d = sgu - sgl;
                const float sd = d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f);  // torch's abs' (0 at 0)
                const float gu = gL * sd * s * sgu * (1.f - sgu);
                const float gl = -gL * sd * s * sgl * (1.f - sgl);
                float dx = f_backward(q, xu, su_st, gu, acc);
                dx += f_backward(q, xl, sl_st, gl, acc);
                dy[r * C + c] = dx;
            }
#pragma unroll
            for (int k = 0; k < NP; ++k) mine[k] += (double)acc[k];
        }
        // raw-parameter chain: d softplus(H) / dH = sigmoid(H), d tanh(a) / da = 1 - tanh(a)^2
        for (int k = 0; k < NP; ++k) {
            const int kind = param_kind(k);
            if (kind == 1) continue;
            const float raw = __ldg(&params[(int64_t)c * NP + k]);
            float fct;
            if (kind == 0) fct = sigmoid_f(raw);
            else { const float t = q[k]; fct = fmaf(-t, t, 1.f); }
            mine[k] *= (double)fct;
        }
    }
    __syncthreads();
    // row lanes meet in ascending order: one fp64 partial row per (part, channel)
    for (int i = threadIdx.x; i < cb * NP; i += EM_THREADS) {
        const int ch = i / NP, k = i % NP;
        double s = 0.0;
        for (int l = 0; l < rl_n; ++l) s += slots[(l * cb + ch) * NP + k];
        partial[((int64_t)blockIdx.x * C + c0 + ch) * NP + k] = s;
    }
}

__global__ void __launch_bounds__(128) factorized_pmf_kernel(const float *__restrict__ params, int lo, int n_sym,
                                                             double *__restrict__ pmf) {
    __shared__ float q_s[NP];
    const int c = blockIdx.x;
    stage_params(params, c, 1, q_s);
    for (int k = threadIdx.x; k < n_sym; k += blockDim.x) pmf[(int64_t)c * n_sym + k] = (double)likelihood(q_s, (float)(lo + k));
}

static int grad_parts(int64_t n) {
    const int64_t p = (n + 255) / 256;
    return p < 1 ? 1 : (p > MAX_PARTS ? MAX_PARTS : (int)p);
}

}  // namespace fpcc

using namespace fpcc;

static bool bound_ok(float b) { return b > 0.f && b < 1.f; }  // false for NaN

extern "C" int fpcc_factorized_bits(const float *y, int64_t ld_y, int64_t n, int C, const float *params, float bound, float *bits,
                                    void *stream) {
    FPCC_REQUIRE(y && params && bits, "factorized_bits: NULL pointer");
    FPCC_REQUIRE(C > 0 && C <= (1 << 22), "factorized_bits: C %d must be in 1..2^22", C);
    FPCC_REQUIRE(n >= 0 && n <= ((int64_t)1 << 40), "factorized_bits: bad row count");
    FPCC_REQUIRE(ld_y >= C, "factorized_bits: row pitch below the channel count");
    FPCC_REQUIRE(bound_ok(bound), "factorized_bits: likelihood bound must be in (0, 1)");
    if (n == 0) return FPCC_OK;
    const int cb0 = C < SLICE ? C : SLICE;
    const int rows = (EM_THREADS / cb0) * 8;  // 8 elements per thread
    const int64_t ctas = (n + rows - 1) / rows;
    FPCC_REQUIRE(ctas <= INT32_MAX, "factorized_bits: too many rows");
    factorized_bits_kernel<<<dim3((unsigned)ctas, ceil_div(C, SLICE)), EM_THREADS, 0, (cudaStream_t)stream>>>(y, ld_y, n, C, params, bound,
                                                                                                            rows, bits);
    FPCC_LAUNCH_CHECK();
    return FPCC_OK;
}

extern "C" size_t fpcc_factorized_grad_workspace(int64_t n, int C) {
    if (n < 1 || C < 1) return 256;
    return (((size_t)grad_parts(n) * (size_t)C * NP * sizeof(double)) + 255) & ~(size_t)255;
}

extern "C" int fpcc_factorized_grad(const float *y, int64_t ld_y, const float *dbits, int64_t ld_db, int64_t n, int C,
                                    const float *params, float bound, float *dy, float *dparams, void *workspace,
                                    size_t workspace_bytes, void *stream) {
    FPCC_REQUIRE(y && dbits && params && dy && dparams, "factorized_grad: NULL pointer");
    FPCC_REQUIRE(C > 0 && C <= (1 << 22), "factorized_grad: C %d must be in 1..2^22", C);
    FPCC_REQUIRE(n >= 0 && n <= ((int64_t)1 << 40), "factorized_grad: bad row count");
    FPCC_REQUIRE(ld_y >= C && ld_db >= C, "factorized_grad: row pitch below the channel count");
    FPCC_REQUIRE(bound_ok(bound), "factorized_grad: likelihood bound must be in (0, 1)");
    FPCC_REQUIRE(workspace && workspace_bytes >= fpcc_factorized_grad_workspace(n, C), "factorized_grad: workspace too small");
    cudaStream_t s = (cudaStream_t)stream;
    if (n == 0) {
        FPCC_CUDA(cudaMemsetAsync(dparams, 0, (size_t)C * NP * sizeof(float), s));
        return FPCC_OK;
    }
    const size_t dyn = (size_t)EM_THREADS * NP * sizeof(double);
    static bool attr_set = false;  // per process; the attribute is a property of the kernel on every device
    if (!attr_set) {
        FPCC_CUDA(cudaFuncSetAttribute(factorized_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
        attr_set = true;
    }
    const int parts = grad_parts(n);
    const int rows = (int)((n + parts - 1) / parts);
    double *partial = (double *)workspace;
    factorized_grad_kernel<<<dim3(parts, ceil_div(C, SLICE)), EM_THREADS, dyn, s>>>(y, ld_y, dbits, ld_db, n, C, params, bound, rows, dy,
                                                                                   partial);
    FPCC_LAUNCH_CHECK();
    act_grad_bias_kernel<<<C * NP, 256, 0, s>>>(partial, parts, C * NP, dparams);
    FPCC_LAUNCH_CHECK();
    return FPCC_OK;
}

extern "C" int fpcc_factorized_pmf(const float *params, int C, int lo, int n_sym, double *pmf, void *stream) {
    FPCC_REQUIRE(params && pmf, "factorized_pmf: NULL pointer");
    FPCC_REQUIRE(C > 0 && C <= (1 << 22), "factorized_pmf: C %d must be in 1..2^22", C);
    FPCC_REQUIRE(n_sym > 0 && n_sym <= (1 << 16), "factorized_pmf: n_sym %d must be in 1..65536", n_sym);
    FPCC_REQUIRE(lo >= -(1 << 24) && (int64_t)lo + n_sym <= (1 << 24), "factorized_pmf: symbols lo .. lo + n_sym must lie in +-2^24");
    factorized_pmf_kernel<<<C, 128, 0, (cudaStream_t)stream>>>(params, lo, n_sym, pmf);
    FPCC_LAUNCH_CHECK();
    return FPCC_OK;
}
