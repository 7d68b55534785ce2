// train.cu -- kernels of the TRAINING path besides the GEMM (gemm_f32.cu): batch-statistics BatchNorm forward/backward,
// the EdgeConv edge gather / scatter, max-over-k with argmax and its backward, and row softmax forward/backward.
//
// Reference semantics (model.train(), train.py:614): every BatchNorm normalises with the statistics of the current batch
// (biased variance; over B*N*k edge elements for the EdgeConv BatchNorm2d layers, model/dgcnn.py:54-55), LeakyReLU(0.2),
// max over the k neighbours (model/dgcnn.py:118) routes its gradient to the arg-max edge, and the gather of
// model/dgcnn.py:35-41 back-propagates as a scatter-add.  Training tensors are fp32, channel-major (C, M) with M = points
// (or E = points * k edges, e = i*k + slot); this first version materialises the per-edge tensors (the reference does too).
#include "common.cuh"

namespace gfs {

// ------------------------------------------------------------------------------------------------------------------
// BatchNorm (batch statistics): one CTA per channel, fp64 accumulation, fixed order -> deterministic
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double block_sum(double v, double* red) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
    return t;
}

constexpr int BN_SPLIT = 16;   // CTAs per channel; partials are combined in index order -> deterministic

__global__ void __launch_bounds__(512)
bn_stats_kernel(const float* __restrict__ x, int64_t ld, int64_t M, double* __restrict__ part) {
    __shared__ double red[16];
    const float* row = x + (int64_t)blockIdx.x * ld;
    const int64_t per = (M + gridDim.y - 1) / gridDim.y;
    const int64_t i0 = per * blockIdx.y, i1 = (i0 + per) < M ? (i0 + per) : M;
    double s = 0.0, q = 0.0;
    for (int64_t i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        const double v = row[i];
        s += v;
        q += v * v;
    }
    s = block_sum(s, red);
    q = block_sum(q, red);
    if (threadIdx.x == 0) {
        part[((int64_t)blockIdx.x * gridDim.y + blockIdx.y) * 2 + 0] = s;
        part[((int64_t)blockIdx.x * gridDim.y + blockIdx.y) * 2 + 1] = q;
    }
}

__global__ void bn_stats_finish_kernel(const double* __restrict__ part, int C, int S, int64_t M, float* __restrict__ mean,
                                       float* __restrict__ var) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double s = 0.0, q = 0.0;
    for (int i = 0; i < S; ++i) {
        s += part[((int64_t)c * S + i) * 2 + 0];
        q += part[((int64_t)c * S + i) * 2 + 1];
    }
    const double m = s / (double)M;
    mean[c] = (float)m;
    var[c] = (float)fmax(q / (double)M - m * m, 0.0);
}

// the same finish plus what the training forward derives from the statistics (one launch instead of four elementwise ones):
// invstd = rsqrt(var + eps), scale = gamma * invstd, shift = beta - mean * scale   (fp32, the reference's operation order)
__global__ void bn_stats_coeffs_kernel(const double* __restrict__ part, int C, int S, int64_t M, const float* __restrict__ gamma,
                                       const float* __restrict__ beta, float eps, float* __restrict__ mean, float* __restrict__ var,
                                       float* __restrict__ invstd, float* __restrict__ scale, float* __restrict__ shift) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double s = 0.0, q = 0.0;
    for (int i = 0; i < S; ++i) {
        s += part[((int64_t)c * S + i) * 2 + 0];
        q += part[((int64_t)c * S + i) * 2 + 1];
    }
    const double m = s / (double)M;
    const float mf = (float)m, vf = (float)fmax(q / (double)M - m * m, 0.0);
    const float is = rsqrtf(vf + eps), sc = gamma[c] * is;
    mean[c] = mf;
    var[c] = vf;
    invstd[c] = is;
    scale[c] = sc;
    shift[c] = beta[c] - mf * sc;
}

// nn.BatchNorm running statistics (momentum form): r = (1 - mom) r + mom * batch, unbiased variance; ++num_batches_tracked
__global__ void bn_update_running_kernel(const float* __restrict__ mean, const float* __restrict__ var, int C, float unbias, float mom,
                                         float* __restrict__ rmean, float* __restrict__ rvar, long long* __restrict__ nbt) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c == 0 && nbt) *nbt += 1;
    if (c >= C) return;
    rmean[c] = rmean[c] * (1.0f - mom) + mom * mean[c];
    rvar[c] = rvar[c] * (1.0f - mom) + mom * (var[c] * unbias);
}

// y = act(x * scale[c] + shift[c]),  act(u) = u > 0 ? u : slope * u   (slope 0.2 LeakyReLU, 0 ReLU, 1 identity)
__global__ void bn_act_fwd_kernel(const float* __restrict__ x, int64_t ldx, float* __restrict__ y, int64_t ldy, int64_t M,
                                  const float* __restrict__ scale, const float* __restrict__ shift, float slope) {
    const int c = blockIdx.y;
    const float sc = scale[c], sh = shift[c];
    const float* xr = x + (int64_t)c * ldx;
    float* yr = y + (int64_t)c * ldy;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < M; i += (int64_t)gridDim.x * blockDim.x) {
        const float u = fmaf(xr[i], sc, sh);
        yr[i] = u > 0.0f ? u : slope * u;
    }
}

// g = dy * act'(u), u = gamma * xhat + beta;  sums[c] = (sum g, sum g * xhat)
__global__ void __launch_bounds__(512)
bn_bwd_reduce_kernel(const float* __restrict__ dy, int64_t lddy, const float* __restrict__ x, int64_t ldx, int64_t M,
                     const float* __restrict__ mean, const float* __restrict__ invstd, const float* __restrict__ gamma,
                     const float* __restrict__ beta, float slope, double* __restrict__ part) {
    __shared__ double red[16];
    const int c = blockIdx.x;
    const float mu = mean[c], is = invstd[c], ga = gamma[c], be = beta[c];
    const float* dr = dy + (int64_t)c * lddy;
    const float* xr = x + (int64_t)c * ldx;
    const int64_t per = (M + gridDim.y - 1) / gridDim.y;
    const int64_t i0 = per * blockIdx.y, i1 = (i0 + per) < M ? (i0 + per) : M;
    double s = 0.0, q = 0.0;
    for (int64_t i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        const float xh = (xr[i] - mu) * is;
        const float u = fmaf(ga, xh, be);
        const float g = dr[i] * (u > 0.0f ? 1.0f : slope);
        s += g;
        q += (double)g * xh;
    }
    s = block_sum(s, red);
    q = block_sum(q, red);
    if (threadIdx.x == 0) {
        part[((int64_t)c * gridDim.y + blockIdx.y) * 2 + 0] = s;
        part[((int64_t)c * gridDim.y + blockIdx.y) * 2 + 1] = q;
    }
}

__global__ void bn_bwd_finish_kernel(const double* __restrict__ part, int C, int S, float* __restrict__ sum_g, float* __restrict__ sum_gx) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double s = 0.0, q = 0.0;
    for (int i = 0; i < S; ++i) {
        s += part[((int64_t)c * S + i) * 2 + 0];
        q += part[((int64_t)c * S + i) * 2 + 1];
    }
    sum_g[c] = (float)s;
    sum_gx[c] = (float)q;
}

// The same two kernels for the BatchNorm that feeds max-over-k (model/dgcnn.py:55-58,118): the incoming gradient is dy (C, Mp)
// at the arg-max edge of every (channel, point) and zero on the other k-1 edges, so the (C, Mp*k) tensor gfs_max_over_k_bwd would
// write is never built: the sums run over the Mp arg-max edges only, the apply pass reads dy / arg per point.
__global__ void __launch_bounds__(512)
bn_bwd_reduce_argmax_kernel(const float* __restrict__ dy, int64_t lddy, const uint8_t* __restrict__ arg, int k,
                            const float* __restrict__ x, int64_t ldx, int64_t Mp, const float* __restrict__ mean,
                            const float* __restrict__ invstd, const float* __restrict__ gamma, const float* __restrict__ beta,
                            float slope, double* __restrict__ part) {
    __shared__ double red[16];
    const int c = blockIdx.x;
    const float mu = mean[c], is = invstd[c], ga = gamma[c], be = beta[c];
    const float* dr = dy + (int64_t)c * lddy;
    const uint8_t* ar = arg + (int64_t)c * Mp;
    const float* xr = x + (int64_t)c * ldx;
    const int64_t per = (Mp + gridDim.y - 1) / gridDim.y;
    const int64_t i0 = per * blockIdx.y, i1 = (i0 + per) < Mp ? (i0 + per) : Mp;
    double s = 0.0, q = 0.0;
    for (int64_t i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        const float xh = (xr[i * k + ar[i]] - mu) * is;
        const float u = fmaf(ga, xh, be);
        const float g = dr[i] * (u > 0.0f ? 1.0f : slope);
        s += g;
        q += (double)g * xh;
    }
    s = block_sum(s, red);
    q = block_sum(q, red);
    if (threadIdx.x == 0) {
        part[((int64_t)c * gridDim.y + blockIdx.y) * 2 + 0] = s;
        part[((int64_t)c * gridDim.y + blockIdx.y) * 2 + 1] = q;
    }
}

// VEC = 4: k % 4 == 0 and 16-byte aligned rows -> four consecutive edges of ONE point per thread (float4 in / out)
template <int VEC>
__global__ void bn_bwd_apply_argmax_kernel(const float* __restrict__ dy, int64_t lddy, const uint8_t* __restrict__ arg, int k,
                                           const float* __restrict__ x, int64_t ldx, float* __restrict__ dx, int64_t lddx, int64_t Mp,
                                           const float* __restrict__ mean, const float* __restrict__ invstd,
                                           const float* __restrict__ gamma, const float* __restrict__ beta, float slope,
                                           const float* __restrict__ sum_g, const float* __restrict__ sum_gx) {
    const int c = blockIdx.y;
    const int64_t E = Mp * k;
    const float mu = mean[c], is = invstd[c], ga = gamma[c], be = beta[c];
    const float a = sum_g[c] / (float)E, b = sum_gx[c] / (float)E, kk = ga * is;
    const float* dr = dy + (int64_t)c * lddy;
    const uint8_t* ar = arg + (int64_t)c * Mp;
    const float* xr = x + (int64_t)c * ldx;
    float* o = dx + (int64_t)c * lddx;
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v * VEC < E; v += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = v * VEC;
        const int64_t p = i / k;
        const int slot0 = (int)(i - p * k), hit = (int)__ldg(ar + p) - slot0;     // arg-max edge is element `hit` of this group
        float xin[VEC], out[VEC];
        if (VEC == 4) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(xr + i));
            xin[0] = t.x; xin[1] = t.y; xin[2] = t.z; xin[3] = t.w;
        } else {
            xin[0] = __ldg(xr + i);
        }
        const float d = (hit >= 0 && hit < VEC) ? __ldg(dr + p) : 0.0f;
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            const float xh = (xin[e] - mu) * is;
            const float u = fmaf(ga, xh, be);
            const float g = (e == hit) ? d * (u > 0.0f ? 1.0f : slope) : 0.0f;
            out[e] = kk * (g - a - xh * b);
        }
        if (VEC == 4) *reinterpret_cast<float4*>(o + i) = make_float4(out[0], out[1], out[2], out[3]);
        else o[i] = out[0];
    }
}

// dx = gamma * invstd * (g - sum_g / M - xhat * sum_gx / M)
__global__ void bn_bwd_apply_kernel(const float* __restrict__ dy, int64_t lddy, const float* __restrict__ x, int64_t ldx,
                                    float* __restrict__ dx, int64_t lddx, int64_t M, const float* __restrict__ mean,
                                    const float* __restrict__ invstd, const float* __restrict__ gamma, const float* __restrict__ beta,
                                    float slope, const float* __restrict__ sum_g, const float* __restrict__ sum_gx) {
    const int c = blockIdx.y;
    const float mu = mean[c], is = invstd[c], ga = gamma[c], be = beta[c];
    const float a = sum_g[c] / (float)M, b = sum_gx[c] / (float)M, k = ga * is;
    const float* dr = dy + (int64_t)c * lddy;
    const float* xr = x + (int64_t)c * ldx;
    float* o = dx + (int64_t)c * lddx;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < M; i += (int64_t)gridDim.x * blockDim.x) {
        const float xh = (xr[i] - mu) * is;
        const float u = fmaf(ga, xh, be);
        const float g = dr[i] * (u > 0.0f ? 1.0f : slope);
        o[i] = k * (g - a - xh * b);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// EdgeConv edge tensor: H[c, e] = P[j(e), c] + Q[i(e), c],  e = i*k + slot,  j = block(i)*N + idx[i, slot]
// pq: (M, 128) point-major [P | Q];  H: (64, E) channel-major.  CTA = 128 consecutive edges, transposed through smem.
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
edge_gather_kernel(const float* __restrict__ pq, const int32_t* __restrict__ idx, int N, int k, int64_t E, float* __restrict__ H,
                   float2* __restrict__ part) {
    __shared__ float T[64][129];
    const int64_t e0 = (int64_t)blockIdx.x * 128;
    const int q = threadIdx.x & 7, sub = threadIdx.x >> 3;
#pragma unroll 2
    for (int p = 0; p < 8; ++p) {
        const int el = p * 16 + sub;
        const int64_t e = e0 + el;
        float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0;
        if (e < E) {
            const int64_t i = e / k;
            const int64_t j = (i / N) * N + idx[e];
            const float4* P = reinterpret_cast<const float4*>(pq + j * 128 + q * 8);
            const float4* Q = reinterpret_cast<const float4*>(pq + i * 128 + 64 + q * 8);
            const float4 p0 = __ldg(P), p1 = __ldg(P + 1), q0 = __ldg(Q), q1 = __ldg(Q + 1);
            a0 = make_float4(p0.x + q0.x, p0.y + q0.y, p0.z + q0.z, p0.w + q0.w);
            a1 = make_float4(p1.x + q1.x, p1.y + q1.y, p1.z + q1.z, p1.w + q1.w);
        }
        const int c = q * 8;
        T[c + 0][el] = a0.x; T[c + 1][el] = a0.y; T[c + 2][el] = a0.z; T[c + 3][el] = a0.w;
        T[c + 4][el] = a1.x; T[c + 5][el] = a1.y; T[c + 6][el] = a1.z; T[c + 7][el] = a1.w;
    }
    __syncthreads();
    const int64_t e = e0 + threadIdx.x;
    if (e < E)
        for (int c = 0; c < 64; ++c) H[(int64_t)c * E + e] = T[c][threadIdx.x];
    if (part) {
        // BatchNorm statistics of H while the tile is on chip: thread (c, half) sums 64 edges of channel c (rows past E are
        // zero); partials [c][2 * CTA + half] are combined in index order in fp64 by bn_stats_partials_kernel (deterministic)
        const int c = threadIdx.x & 63, half = threadIdx.x >> 6;
        float sm = 0.0f, sq = 0.0f;
#pragma unroll 8
        for (int el = half * 64; el < half * 64 + 64; ++el) {
            const float v = T[c][el];
            sm += v;
            sq = fmaf(v, v, sq);
        }
        part[(int64_t)c * (2 * gridDim.x) + 2 * blockIdx.x + half] = make_float2(sm, sq);
    }
}

// per-channel statistics and affine coefficients from the partial (sum, sum of squares) pairs of edge_gather_kernel
__global__ void __launch_bounds__(256)
bn_stats_partials_kernel(const float2* __restrict__ part, int P, int64_t M, const float* __restrict__ gamma, const float* __restrict__ beta,
                         float eps, float* __restrict__ mean, float* __restrict__ var, float* __restrict__ invstd,
                         float* __restrict__ scale, float* __restrict__ shift) {
    __shared__ double red[16];
    const int c = blockIdx.x;
    const float2* row = part + (int64_t)c * P;
    double s = 0.0, q = 0.0;
    for (int i = threadIdx.x; i < P; i += blockDim.x) {       // fixed assignment + fixed-order tree: deterministic
        const float2 v = row[i];
        s += (double)v.x;
        q += (double)v.y;
    }
    s = block_sum(s, red);
    q = block_sum(q, red);
    if (threadIdx.x == 0) {
        const double m = s / (double)M;
        const float mf = (float)m, vf = (float)fmax(q / (double)M - m * m, 0.0);
        const float is = rsqrtf(vf + eps), sc = gamma[c] * is;
        mean[c] = mf;
        var[c] = vf;
        invstd[c] = is;
        scale[c] = sc;
        shift[c] = beta[c] - mf * sc;
    }
}

// backward of the gather: dP[j] += dH[:, e] (j = idx[e]), dQ[i] = sum_slot dH[:, i*k + slot]   (the P half of dpq must be zeroed)
// A CTA owns ES_PPB consecutive points = ES_PPB*k consecutive edges, staged channel-major through shared memory.  The Q half
// needs no atomics (all k edges of a point are in the tile: one plain store per channel, fixed summation order); the P half goes
// out as 16-byte vector reductions (red.global.add.v4.f32, sm_90+): 16 per edge instead of 64 scalar atomics.  The order in which
// different CTAs add into one dP row is not fixed -- the only non-deterministic summation of the training path; the ordered
// scatter below (gfs_edge_scatter_bn_ordered) replaces it when the caller asks for reproducible bits.
constexpr int ES_PPB = 8;

__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};\n" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

__global__ void __launch_bounds__(256)
edge_scatter_kernel(const float* __restrict__ dH, const int32_t* __restrict__ idx, int N, int k, int64_t Mp, int64_t E,
                    float* __restrict__ dpq) {
    extern __shared__ float T[];                        // [64][EL + 1]
    const int EL = ES_PPB * k, LD = EL + 1;
    const int64_t i0 = (int64_t)blockIdx.x * ES_PPB;
    const int64_t e0 = i0 * k;
    const int np = (int)((Mp - i0) < ES_PPB ? (Mp - i0) : ES_PPB);
    const int ne = np * k;
    for (int t = threadIdx.x; t < 64 * EL; t += 256) {
        const int c = t / EL, el = t - c * EL;
        T[c * LD + el] = el < ne ? __ldg(dH + (int64_t)c * E + e0 + el) : 0.0f;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < 64 * np; t += 256) {
        const int p = t >> 6, c = t & 63;
        const float* r = T + c * LD + p * k;
        float sum = 0.0f;
        for (int sl = 0; sl < k; ++sl) sum += r[sl];
        dpq[(i0 + p) * 128 + 64 + c] = sum;
    }
    for (int t = threadIdx.x; t < ne * 16; t += 256) {
        const int el = t >> 4, q = t & 15;
        const int64_t i = i0 + el / k;
        const int64_t j = (i / N) * N + __ldg(idx + e0 + el);
        const float* r = T + (4 * q) * LD + el;
        red_add_v4(dpq + j * 128 + 4 * q, r[0], r[LD], r[2 * LD], r[3 * LD]);
    }
}

// The same scatter with the BatchNorm + activation backward of the layer in front of it applied on the fly: the tile is
//   dH[c, e] = gamma[c] invstd[c] (g - sum_g[c]/E - xhat sum_gx[c]/E),   g = dy[c, e] * act'(gamma xhat + beta),  xhat = (x - mean) invstd
// computed from dy (= d h1) and x (= H) while staging, so the (64, E) tensor dH is never written or re-read.
// ORDERED = false: the P half goes out as red.global.add.v4.f32 (dpq's P half zeroed by the caller).
// ORDERED = true (phase 1 of gfs_edge_scatter_bn_ordered): the P-half terms are stored edge-major instead, terms[e, 0:64] (rows of
// 256 B, 16-byte stores); edge_gather_rows_kernel then sums them per target in ascending edge order.
template <bool ORDERED>
__global__ void __launch_bounds__(256)
edge_scatter_bn_kernel(const float* __restrict__ dy, const float* __restrict__ x, const int32_t* __restrict__ idx, int N, int k, int64_t Mp,
                       int64_t E, const float* __restrict__ mean, const float* __restrict__ invstd, const float* __restrict__ gamma,
                       const float* __restrict__ beta, float slope, const float* __restrict__ sum_g, const float* __restrict__ sum_gx,
                       float* __restrict__ dpq, float* __restrict__ terms) {
    extern __shared__ float T[];                        // [64][EL + 1]
    __shared__ float cf[5][64];                         // mean, invstd, gamma, beta | gamma*invstd ; a ; b  (packed below)
    __shared__ float ca[64], cb[64];
    const int EL = ES_PPB * k, LD = EL + 1;
    if (threadIdx.x < 64) {
        const int c = threadIdx.x;
        cf[0][c] = mean[c];
        cf[1][c] = invstd[c];
        cf[2][c] = gamma[c];
        cf[3][c] = beta[c];
        cf[4][c] = gamma[c] * invstd[c];
        ca[c] = sum_g[c] / (float)E;
        cb[c] = sum_gx[c] / (float)E;
    }
    __syncthreads();
    const int64_t i0 = (int64_t)blockIdx.x * ES_PPB;
    const int64_t e0 = i0 * k;
    const int np = (int)((Mp - i0) < ES_PPB ? (Mp - i0) : ES_PPB);
    const int ne = np * k;
    for (int t = threadIdx.x; t < 64 * EL; t += 256) {
        const int c = t / EL, el = t - c * EL;
        float v = 0.0f;
        if (el < ne) {
            const int64_t o = (int64_t)c * E + e0 + el;
            const float xh = (__ldg(x + o) - cf[0][c]) * cf[1][c];
            const float u = fmaf(cf[2][c], xh, cf[3][c]);
            const float g = __ldg(dy + o) * (u > 0.0f ? 1.0f : slope);
            v = cf[4][c] * (g - ca[c] - xh * cb[c]);      // same expression as bn_bwd_apply_kernel
        }
        T[c * LD + el] = v;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < 64 * np; t += 256) {
        const int p = t >> 6, c = t & 63;
        const float* r = T + c * LD + p * k;
        float sum = 0.0f;
        for (int sl = 0; sl < k; ++sl) sum += r[sl];
        dpq[(i0 + p) * 128 + 64 + c] = sum;
    }
    for (int t = threadIdx.x; t < ne * 16; t += 256) {
        const int el = t >> 4, q = t & 15;
        const float* r = T + (4 * q) * LD + el;
        if (ORDERED) {
            reinterpret_cast<float4*>(terms + (e0 + el) * 64)[q] = make_float4(r[0], r[LD], r[2 * LD], r[3 * LD]);
        } else {
            const int64_t i = i0 + el / k;
            const int64_t j = (i / N) * N + __ldg(idx + e0 + el);
            red_add_v4(dpq + j * 128 + 4 * q, r[0], r[LD], r[2 * LD], r[3 * LD]);
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Ordered (deterministic) scatter: reverse index of the graph + per-target sums in ascending edge order
// ------------------------------------------------------------------------------------------------------------------
// CSR of the incoming edges of every target, identical to a stable sort of the targets: rev_ptr[j] = sum of the in-degrees of
// the targets before j, rev_edge[rev_ptr[j] .. rev_ptr[j+1]) = the edges e with target j in ascending order.  Every edge of block b
// targets block b, so block b's edges fill rev_edge[b*N*k, (b+1)*N*k) and one CTA builds its block alone.  Its NW warps split the
// block's edges into NW consecutive segments: pass 1 counts per (segment, target) in shared memory, a scan over (target, segment)
// turns the counts into write cursors, pass 2 walks each segment again 32 edges at a time and places every edge at its cursor
// plus its rank among the lanes with the same target (__match_any_sync).  No atomics decide an order: the result is the same
// on every run.
constexpr int RI_THREADS = 512;
constexpr size_t RI_SMEM_MAX = 226 * 1024;           // dynamic part; the static wsum and the 227 KB cap leave room

__global__ void __launch_bounds__(RI_THREADS)
edge_reverse_index_kernel(const int32_t* __restrict__ idx, int N, int k, int NW, int32_t* __restrict__ rev_ptr,
                          int32_t* __restrict__ rev_edge) {
    extern __shared__ int32_t cnt[];                    // [NW][N]
    __shared__ int32_t wsum[RI_THREADS / 32];
    const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t EB = (int64_t)N * k, base = (int64_t)b * EB;
    const int32_t* ib = idx + base;
    const int64_t seg = (EB + NW - 1) / NW;
    const int64_t lo = warp < NW ? (int64_t)warp * seg : EB, hi = lo + seg < EB ? lo + seg : EB;
    for (int i = tid; i < NW * N; i += RI_THREADS) cnt[i] = 0;
    __syncthreads();
    for (int64_t e = lo + lane; e < hi; e += 32) atomicAdd(&cnt[warp * N + __ldg(ib + e)], 1);   // integer counts: order-free
    __syncthreads();
    // thread t owns targets [t*R, t*R + R): exclusive prefix over the segments, then over the targets (block-wide scan)
    const int R = (N + RI_THREADS - 1) / RI_THREADS;
    const int l0 = tid * R < N ? tid * R : N, l1 = l0 + R < N ? l0 + R : N;
    int own = 0;
    for (int l = l0; l < l1; ++l) {
        int run = 0;
        for (int w = 0; w < NW; ++w) {
            const int c = cnt[w * N + l];
            cnt[w * N + l] = run;
            run += c;
        }
        rev_ptr[(int64_t)b * N + l] = run;              // in-degree, replaced by the start below
        own += run;
    }
    int inc = own;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += v;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    int before = inc - own;
    for (int w = 0; w < warp; ++w) before += wsum[w];
    int64_t start = base + before;
    for (int l = l0; l < l1; ++l) {
        const int deg = rev_ptr[(int64_t)b * N + l];
        rev_ptr[(int64_t)b * N + l] = (int32_t)start;
        for (int w = 0; w < NW; ++w) cnt[w * N + l] += (int32_t)start;
        start += deg;
    }
    if (b == gridDim.x - 1 && tid == 0) rev_ptr[(int64_t)gridDim.x * N] = (int32_t)(base + EB);
    __syncthreads();
    if (warp >= NW) return;
    const unsigned lt = (1u << lane) - 1u;
    for (int64_t e0 = lo; e0 < hi; e0 += 32) {
        const int64_t e = e0 + lane;
        const int l = e < hi ? __ldg(ib + e) : -1 - lane;          // lanes past the segment: a key no other lane has
        const unsigned same = __match_any_sync(0xffffffffu, l);
        if (e < hi) {
            const int at = cnt[warp * N + l];
            rev_edge[at + __popc(same & lt)] = (int32_t)(base + e);
            __syncwarp(same);
            if ((same & lt) == 0) cnt[warp * N + l] = at + __popc(same);   // the lowest lane of each group advances the cursor
        }
        __syncwarp();
    }
}

// Phase 2 of the ordered scatter: dpq[j, 0:64] = sum over r of terms[rev_edge[r], 0:64], r ascending from rev_ptr[j], starting
// from +0.0.  Half a warp per target, a float4 (four channels) per lane; the edge ids and rows of ES_AHEAD edges are loaded
// before their adds, so a long list is bound by load latency per batch, not per edge.
constexpr int ES_AHEAD = 8;

__global__ void __launch_bounds__(256)
edge_gather_rows_kernel(const float* __restrict__ terms, const int32_t* __restrict__ rev_ptr, const int32_t* __restrict__ rev_edge,
                        int64_t Mp, float* __restrict__ dpq) {
    const int64_t j = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    const int q = threadIdx.x & 15;
    if (j >= Mp) return;
    const int32_t s = __ldg(rev_ptr + j), t = __ldg(rev_ptr + j + 1);
    float4 acc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    int32_t r = s;
    for (; r + ES_AHEAD <= t; r += ES_AHEAD) {
        float4 v[ES_AHEAD];
#pragma unroll
        for (int u = 0; u < ES_AHEAD; ++u) v[u] = __ldg(reinterpret_cast<const float4*>(terms + (int64_t)__ldg(rev_edge + r + u) * 64) + q);
#pragma unroll
        for (int u = 0; u < ES_AHEAD; ++u) {
            acc.x += v[u].x;
            acc.y += v[u].y;
            acc.z += v[u].z;
            acc.w += v[u].w;
        }
    }
    for (; r < t; ++r) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(terms + (int64_t)__ldg(rev_edge + r) * 64) + q);
        acc.x += v.x;
        acc.y += v.y;
        acc.z += v.z;
        acc.w += v.w;
    }
    reinterpret_cast<float4*>(dpq + j * 128)[q] = acc;
}

// y[c, i] = max_slot a[c, i*k + slot] (first maximum), arg[c, i] = slot
__global__ void max_over_k_fwd_kernel(const float* __restrict__ a, int64_t M, int k, float* __restrict__ y, int64_t ldy,
                                      uint8_t* __restrict__ arg) {
    const int c = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    const float* r = a + (int64_t)c * M * k + i * k;
    float best = r[0];
    int bi = 0;
    for (int s = 1; s < k; ++s) {
        const float v = r[s];
        if (v > best) {
            best = v;
            bi = s;
        }
    }
    y[(int64_t)c * ldy + i] = best;
    arg[(int64_t)c * M + i] = (uint8_t)bi;
}

// BN + activation + max over k in one pass over the pre-BN tensor (model/dgcnn.py:55-58,118): the (C, M*k) activated tensor is
// never written.  The activation is applied BEFORE the max (the folded scale may be negative, SURVEY H4).
__global__ void bn_act_max_kernel(const float* __restrict__ z, int64_t M, int k, const float* __restrict__ scale,
                                  const float* __restrict__ shift, float slope, float* __restrict__ y, int64_t ldy,
                                  uint8_t* __restrict__ arg) {
    const int c = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    const float sc = scale[c], sh = shift[c];
    const float* r = z + (int64_t)c * M * k + i * k;
    float best = -INFINITY;
    int bi = 0;
    for (int s = 0; s < k; ++s) {
        const float u = fmaf(r[s], sc, sh);
        const float v = u > 0.0f ? u : slope * u;
        if (v > best) {                              // first maximum, as max_over_k_fwd_kernel
            best = v;
            bi = s;
        }
    }
    y[(int64_t)c * ldy + i] = best;
    arg[(int64_t)c * M + i] = (uint8_t)bi;
}

__global__ void max_over_k_bwd_kernel(const float* __restrict__ dy, int64_t lddy, const uint8_t* __restrict__ arg, int64_t M, int k,
                                      float* __restrict__ da) {
    const int c = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    const float g = dy[(int64_t)c * lddy + i];
    const int w = arg[(int64_t)c * M + i];
    float* r = da + (int64_t)c * M * k + i * k;
    for (int s = 0; s < k; ++s) r[s] = s == w ? g : 0.0f;
}

// ------------------------------------------------------------------------------------------------------------------
// row softmax (attention, model/attention.py:45):  p = softmax(s * scale) [* mask];  one warp per row
// backward: ds = scale * p0 * (dp*mask - sum(dp*mask*p0)),  p0 = softmax without the mask
// ------------------------------------------------------------------------------------------------------------------
// Dropout without a mask tensor: keep / drop of element (row r, column j) is a counter-based hash of (seed, r, j), so the
// forward and the backward pass regenerate the same decision and the (rows x n) mask (537 MB at B = 32, N = 2048) is neither
// drawn, stored nor read.  Returns the factor 1/keep or 0.  (The stream differs from torch's Philox: dropout is stochastic in
// the reference too, SURVEY H5; parity tests run with p = 0 or with an explicit mask.)
__device__ __forceinline__ float drop_factor(uint32_t seed, uint32_t r, uint32_t j, float keep, float inv_keep) {
    uint32_t h = (r * 0x9E3779B1u) ^ (j * 0x85EBCA77u) ^ seed;
    h ^= h >> 15;
    h *= 0x2C1B3C6Du;
    h ^= h >> 12;
    h *= 0x297A2D39u;
    h ^= h >> 15;
    return (float)(h >> 8) * (1.0f / 16777216.0f) < keep ? inv_keep : 0.0f;
}

// the mask the hash defines, materialised (tests)
__global__ void dropout_mask_kernel(int64_t rows, int n, uint32_t seed, float keep, float* __restrict__ mask) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * n) return;
    mask[i] = drop_factor(seed, (uint32_t)(i / n), (uint32_t)(i % n), keep, 1.0f / keep);
}

__global__ void softmax_rows_fwd_kernel(const float* __restrict__ s, int64_t rows, int n, float scale, const float* __restrict__ mask,
                                        uint32_t seed, float keep, float* __restrict__ p0, float* __restrict__ p) {
    const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= rows) return;
    const float* sr = s + r * n;
    float mx = -INFINITY;
    for (int j = lane; j < n; j += 32) mx = fmaxf(mx, sr[j] * scale);
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.0f;
    for (int j = lane; j < n; j += 32) sum += expf(sr[j] * scale - mx);
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float inv = 1.0f / sum;
    for (int j = lane; j < n; j += 32) {
        const float v = expf(sr[j] * scale - mx) * inv;
        p0[r * n + j] = v;
        if (p != p0) p[r * n + j] = mask ? v * mask[r * n + j] : (keep < 1.0f ? v * drop_factor(seed, (uint32_t)r, (uint32_t)j, keep, 1.0f / keep) : v);
    }
}

__global__ void softmax_rows_bwd_kernel(const float* __restrict__ p0, const float* __restrict__ dp, const float* __restrict__ mask,
                                        uint32_t seed, float keep, int64_t rows, int n, float scale, float* __restrict__ ds) {
    const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= rows) return;
    const float* pr = p0 + r * n;
    const float* dr = dp + r * n;
    const float* mr = mask ? mask + r * n : nullptr;
    const bool hashed = !mr && keep < 1.0f;
    const float ik = 1.0f / keep;
    float dot = 0.0f;
    for (int j = lane; j < n; j += 32)
        dot += pr[j] * dr[j] * (mr ? mr[j] : (hashed ? drop_factor(seed, (uint32_t)r, (uint32_t)j, keep, ik) : 1.0f));
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
    for (int j = lane; j < n; j += 32)
        ds[r * n + j] = scale * pr[j] * (dr[j] * (mr ? mr[j] : (hashed ? drop_factor(seed, (uint32_t)r, (uint32_t)j, keep, ik) : 1.0f)) - dot);
}

}  // namespace gfs

using namespace gfs;

extern "C" int gfs_bn_stats(const float* x, int64_t ld, int C, int64_t M, double* workspace, float* mean, float* var, void* stream) {
    GFS_REQUIRE(x && mean && var && workspace && C > 0 && M > 0, GFS_ERR_BAD_ARG, "gfs_bn_stats: bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int S = M >= 65536 ? BN_SPLIT : 1;
    bn_stats_kernel<<<dim3(C, S), 512, 0, st>>>(x, ld, M, workspace);
    GFS_LAUNCH_OK("bn_stats_kernel");
    bn_stats_finish_kernel<<<(C + 127) / 128, 128, 0, st>>>(workspace, C, S, M, mean, var);
    GFS_LAUNCH_OK("bn_stats_finish_kernel");
    return GFS_OK;
}

extern "C" int gfs_bn_stats_coeffs(const float* x, int64_t ld, int C, int64_t M, double* workspace, const float* gamma,
                                   const float* beta, float eps, float* mean, float* var, float* invstd, float* scale, float* shift,
                                   void* stream) {
    GFS_REQUIRE(x && workspace && gamma && beta && mean && var && invstd && scale && shift && C > 0 && M > 0, GFS_ERR_BAD_ARG,
                "gfs_bn_stats_coeffs: bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int S = M >= 65536 ? BN_SPLIT : 1;
    bn_stats_kernel<<<dim3(C, S), 512, 0, st>>>(x, ld, M, workspace);
    GFS_LAUNCH_OK("bn_stats_kernel");
    bn_stats_coeffs_kernel<<<(C + 127) / 128, 128, 0, st>>>(workspace, C, S, M, gamma, beta, eps, mean, var, invstd, scale, shift);
    GFS_LAUNCH_OK("bn_stats_coeffs_kernel");
    return GFS_OK;
}

extern "C" int gfs_bn_update_running(const float* mean, const float* var, int C, int64_t n, float momentum, float* running_mean,
                                     float* running_var, int64_t* num_batches_tracked, void* stream) {
    GFS_REQUIRE(mean && var && running_mean && running_var && C > 0 && n > 0, GFS_ERR_BAD_ARG, "gfs_bn_update_running: bad argument");
    const float unbias = (float)((double)n / (double)(n > 1 ? n - 1 : 1));
    bn_update_running_kernel<<<(C + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
        mean, var, C, unbias, momentum, running_mean, running_var, reinterpret_cast<long long*>(num_batches_tracked));
    GFS_LAUNCH_OK("bn_update_running_kernel");
    return GFS_OK;
}

extern "C" int gfs_bn_act_fwd(const float* x, int64_t ldx, float* y, int64_t ldy, int C, int64_t M, const float* scale,
                              const float* shift, float slope, void* stream) {
    GFS_REQUIRE(x && y && scale && shift && C > 0 && M > 0, GFS_ERR_BAD_ARG, "gfs_bn_act_fwd: bad argument");
    const unsigned gx = (unsigned)((M + 1023) / 1024 < 1024 ? (M + 1023) / 1024 : 1024);
    bn_act_fwd_kernel<<<dim3(gx, C), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, ldx, y, ldy, M, scale, shift, slope);
    GFS_LAUNCH_OK("bn_act_fwd_kernel");
    return GFS_OK;
}

extern "C" int gfs_bn_act_bwd(const float* dy, int64_t lddy, const float* x, int64_t ldx, float* dx, int64_t lddx, int C, int64_t M,
                              const float* mean, const float* invstd, const float* gamma, const float* beta, float slope,
                              double* workspace, float* sum_g, float* sum_gx, void* stream) {
    GFS_REQUIRE(dy && x && dx && mean && invstd && gamma && beta && workspace && sum_g && sum_gx && C > 0 && M > 0, GFS_ERR_BAD_ARG,
                "gfs_bn_act_bwd: bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int S = M >= 65536 ? BN_SPLIT : 1;
    bn_bwd_reduce_kernel<<<dim3(C, S), 512, 0, st>>>(dy, lddy, x, ldx, M, mean, invstd, gamma, beta, slope, workspace);
    GFS_LAUNCH_OK("bn_bwd_reduce_kernel");
    bn_bwd_finish_kernel<<<(C + 127) / 128, 128, 0, st>>>(workspace, C, S, sum_g, sum_gx);
    GFS_LAUNCH_OK("bn_bwd_finish_kernel");
    const unsigned gx = (unsigned)((M + 1023) / 1024 < 1024 ? (M + 1023) / 1024 : 1024);
    bn_bwd_apply_kernel<<<dim3(gx, C), 256, 0, st>>>(dy, lddy, x, ldx, dx, lddx, M, mean, invstd, gamma, beta, slope, sum_g, sum_gx);
    GFS_LAUNCH_OK("bn_bwd_apply_kernel");
    return GFS_OK;
}

extern "C" int gfs_bn_act_bwd_argmax(const float* dy, int64_t lddy, const uint8_t* arg, int k, const float* x, int64_t ldx, float* dx,
                                     int64_t lddx, int C, int64_t Mp, const float* mean, const float* invstd, const float* gamma,
                                     const float* beta, float slope, double* workspace, float* sum_g, float* sum_gx, void* stream) {
    GFS_REQUIRE(dy && arg && x && dx && mean && invstd && gamma && beta && workspace && sum_g && sum_gx && C > 0 && Mp > 0 && k > 0 && k <= 255,
                GFS_ERR_BAD_ARG, "gfs_bn_act_bwd_argmax: bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int S = Mp >= 65536 ? BN_SPLIT : 1;
    bn_bwd_reduce_argmax_kernel<<<dim3(C, S), 512, 0, st>>>(dy, lddy, arg, k, x, ldx, Mp, mean, invstd, gamma, beta, slope, workspace);
    GFS_LAUNCH_OK("bn_bwd_reduce_argmax_kernel");
    bn_bwd_finish_kernel<<<(C + 127) / 128, 128, 0, st>>>(workspace, C, S, sum_g, sum_gx);
    GFS_LAUNCH_OK("bn_bwd_finish_kernel");
    const int64_t E = Mp * k;
    const bool vec = (k % 4 == 0) && (ldx % 4 == 0) && (lddx % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) &&
                     ((reinterpret_cast<uintptr_t>(dx) & 15) == 0);
    const int64_t items = vec ? E / 4 : E;
    const unsigned gx = (unsigned)((items + 1023) / 1024 < 2048 ? (items + 1023) / 1024 : 2048);
    if (vec)
        bn_bwd_apply_argmax_kernel<4><<<dim3(gx, C), 256, 0, st>>>(dy, lddy, arg, k, x, ldx, dx, lddx, Mp, mean, invstd, gamma, beta, slope,
                                                                   sum_g, sum_gx);
    else
        bn_bwd_apply_argmax_kernel<1><<<dim3(gx, C), 256, 0, st>>>(dy, lddy, arg, k, x, ldx, dx, lddx, Mp, mean, invstd, gamma, beta, slope,
                                                                   sum_g, sum_gx);
    GFS_LAUNCH_OK("bn_bwd_apply_argmax_kernel");
    return GFS_OK;
}

extern "C" int gfs_bn_bwd_sums(const float* dy, int64_t lddy, const float* x, int64_t ldx, int C, int64_t M, const float* mean,
                               const float* invstd, const float* gamma, const float* beta, float slope, double* workspace, float* sum_g,
                               float* sum_gx, void* stream) {
    GFS_REQUIRE(dy && x && mean && invstd && gamma && beta && workspace && sum_g && sum_gx && C > 0 && M > 0, GFS_ERR_BAD_ARG,
                "gfs_bn_bwd_sums: bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int S = M >= 65536 ? BN_SPLIT : 1;
    bn_bwd_reduce_kernel<<<dim3(C, S), 512, 0, st>>>(dy, lddy, x, ldx, M, mean, invstd, gamma, beta, slope, workspace);
    GFS_LAUNCH_OK("bn_bwd_reduce_kernel");
    bn_bwd_finish_kernel<<<(C + 127) / 128, 128, 0, st>>>(workspace, C, S, sum_g, sum_gx);
    GFS_LAUNCH_OK("bn_bwd_finish_kernel");
    return GFS_OK;
}

extern "C" int gfs_edge_scatter_bn(const float* dy, const float* x, const int32_t* idx, int B, int N, int k, const float* mean,
                                   const float* invstd, const float* gamma, const float* beta, float slope, const float* sum_g,
                                   const float* sum_gx, float* dpq, void* stream) {
    GFS_REQUIRE(dy && x && idx && dpq && mean && invstd && gamma && beta && sum_g && sum_gx && B > 0 && N > 0 && k > 0, GFS_ERR_BAD_ARG,
                "gfs_edge_scatter_bn: bad argument");
    GFS_REQUIRE(k <= 64, GFS_ERR_UNSUPPORTED, "gfs_edge_scatter_bn: k <= 64");
    const int64_t Mp = (int64_t)B * N, E = Mp * k;
    const size_t smem = (size_t)64 * (ES_PPB * k + 1) * sizeof(float);
    GFS_CUDA_OK(allow_smem(reinterpret_cast<const void*>(edge_scatter_bn_kernel<false>), (size_t)64 * (ES_PPB * 64 + 1) * sizeof(float)));
    edge_scatter_bn_kernel<false><<<(unsigned)((Mp + ES_PPB - 1) / ES_PPB), 256, smem, static_cast<cudaStream_t>(stream)>>>(
        dy, x, idx, N, k, Mp, E, mean, invstd, gamma, beta, slope, sum_g, sum_gx, dpq, nullptr);
    GFS_LAUNCH_OK("edge_scatter_bn_kernel");
    return GFS_OK;
}

// shared-memory budget of the reverse index: NW segment counters of N ints per CTA
static int reverse_index_segments(int N) {
    const int64_t fit = (int64_t)(RI_SMEM_MAX / sizeof(int32_t)) / N;
    return (int)(fit < RI_THREADS / 32 ? fit : RI_THREADS / 32);
}

extern "C" int gfs_edge_reverse_index(const int32_t* idx, int B, int N, int k, int32_t* rev_ptr, int32_t* rev_edge, void* stream) {
    GFS_REQUIRE(idx && rev_ptr && rev_edge, GFS_ERR_BAD_ARG, "gfs_edge_reverse_index: null pointer");
    GFS_REQUIRE(B > 0 && N > 0 && k > 0, GFS_ERR_BAD_ARG, "gfs_edge_reverse_index: non-positive size (B=%d N=%d k=%d)", B, N, k);
    GFS_REQUIRE(k <= 64, GFS_ERR_UNSUPPORTED, "gfs_edge_reverse_index: k=%d > 64 is not built", k);
    GFS_REQUIRE((int64_t)B * N * k < ((int64_t)1 << 31), GFS_ERR_UNSUPPORTED,
                "gfs_edge_reverse_index: E = B*N*k = %lld edges >= 2^31 (int32 edge ids)", (long long)B * N * k);
    const int NW = reverse_index_segments(N);
    GFS_REQUIRE(NW >= 1, GFS_ERR_UNSUPPORTED, "gfs_edge_reverse_index: N=%d > %d (per-target counters live in shared memory)", N,
                (int)(RI_SMEM_MAX / sizeof(int32_t)));
    const size_t smem = (size_t)NW * N * sizeof(int32_t);
    GFS_CUDA_OK(allow_smem(reinterpret_cast<const void*>(edge_reverse_index_kernel), RI_SMEM_MAX));
    edge_reverse_index_kernel<<<B, RI_THREADS, smem, static_cast<cudaStream_t>(stream)>>>(idx, N, k, NW, rev_ptr, rev_edge);
    GFS_LAUNCH_OK("edge_reverse_index_kernel");
    return GFS_OK;
}

extern "C" int gfs_edge_scatter_bn_ordered(const float* dy, const float* x, const int32_t* idx, const int32_t* rev_ptr,
                                           const int32_t* rev_edge, int B, int N, int k, const float* mean, const float* invstd,
                                           const float* gamma, const float* beta, float slope, const float* sum_g, const float* sum_gx,
                                           float* edge_terms, float* dpq, void* stream) {
    GFS_REQUIRE(dy && x && idx && rev_ptr && rev_edge && mean && invstd && gamma && beta && sum_g && sum_gx && edge_terms && dpq,
                GFS_ERR_BAD_ARG, "gfs_edge_scatter_bn_ordered: null pointer");
    GFS_REQUIRE(B > 0 && N > 0 && k > 0, GFS_ERR_BAD_ARG, "gfs_edge_scatter_bn_ordered: non-positive size (B=%d N=%d k=%d)", B, N, k);
    GFS_REQUIRE(k <= 64, GFS_ERR_UNSUPPORTED, "gfs_edge_scatter_bn_ordered: k=%d > 64 is not built", k);
    GFS_REQUIRE((int64_t)B * N * k < ((int64_t)1 << 31), GFS_ERR_UNSUPPORTED,
                "gfs_edge_scatter_bn_ordered: E = B*N*k = %lld edges >= 2^31 (int32 edge ids)", (long long)B * N * k);
    GFS_REQUIRE(((reinterpret_cast<uintptr_t>(edge_terms) | reinterpret_cast<uintptr_t>(dpq)) & 15) == 0, GFS_ERR_BAD_ARG,
                "gfs_edge_scatter_bn_ordered: edge_terms and dpq must be 16-byte aligned");
    const int64_t Mp = (int64_t)B * N, E = Mp * k;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t smem = (size_t)64 * (ES_PPB * k + 1) * sizeof(float);
    GFS_CUDA_OK(allow_smem(reinterpret_cast<const void*>(edge_scatter_bn_kernel<true>), (size_t)64 * (ES_PPB * 64 + 1) * sizeof(float)));
    edge_scatter_bn_kernel<true><<<(unsigned)((Mp + ES_PPB - 1) / ES_PPB), 256, smem, st>>>(
        dy, x, idx, N, k, Mp, E, mean, invstd, gamma, beta, slope, sum_g, sum_gx, dpq, edge_terms);
    GFS_LAUNCH_OK("edge_scatter_bn_kernel<ordered>");
    edge_gather_rows_kernel<<<(unsigned)((Mp * 16 + 255) / 256), 256, 0, st>>>(edge_terms, rev_ptr, rev_edge, Mp, dpq);
    GFS_LAUNCH_OK("edge_gather_rows_kernel");
    return GFS_OK;
}

extern "C" int gfs_bn_act_max_fwd(const float* z, int C, int64_t M, int k, const float* scale, const float* shift, float slope, float* y,
                                  int64_t ldy, uint8_t* arg, void* stream) {
    GFS_REQUIRE(z && scale && shift && y && arg && C > 0 && M > 0 && k > 0 && k <= 255, GFS_ERR_BAD_ARG, "gfs_bn_act_max_fwd: bad argument");
    bn_act_max_kernel<<<dim3((unsigned)((M + 255) / 256), C), 256, 0, static_cast<cudaStream_t>(stream)>>>(z, M, k, scale, shift, slope, y,
                                                                                                          ldy, arg);
    GFS_LAUNCH_OK("bn_act_max_kernel");
    return GFS_OK;
}

extern "C" int gfs_edge_gather(const float* pq, const int32_t* idx, int B, int N, int k, float* H, void* stream) {
    GFS_REQUIRE(pq && idx && H && B > 0 && N > 0 && k > 0, GFS_ERR_BAD_ARG, "gfs_edge_gather: bad argument");
    const int64_t E = (int64_t)B * N * k;
    edge_gather_kernel<<<(unsigned)((E + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(pq, idx, N, k, E, H, nullptr);
    GFS_LAUNCH_OK("edge_gather_kernel");
    return GFS_OK;
}

extern "C" int gfs_edge_gather_stats(const float* pq, const int32_t* idx, int B, int N, int k, float* H, float* partials,
                                     const float* gamma, const float* beta, float eps, float* mean, float* var, float* invstd,
                                     float* scale, float* shift, void* stream) {
    GFS_REQUIRE(pq && idx && H && partials && gamma && beta && mean && var && invstd && scale && shift && B > 0 && N > 0 && k > 0,
                GFS_ERR_BAD_ARG, "gfs_edge_gather_stats: bad argument");
    const int64_t E = (int64_t)B * N * k;
    const unsigned grid = (unsigned)((E + 127) / 128);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    edge_gather_kernel<<<grid, 128, 0, st>>>(pq, idx, N, k, E, H, reinterpret_cast<float2*>(partials));
    GFS_LAUNCH_OK("edge_gather_kernel");
    bn_stats_partials_kernel<<<64, 256, 0, st>>>(reinterpret_cast<const float2*>(partials), (int)(2 * grid), E, gamma, beta, eps, mean, var,
                                                 invstd, scale, shift);
    GFS_LAUNCH_OK("bn_stats_partials_kernel");
    return GFS_OK;
}

extern "C" int gfs_edge_scatter(const float* dH, const int32_t* idx, int B, int N, int k, float* dpq, void* stream) {
    GFS_REQUIRE(dH && idx && dpq && B > 0 && N > 0 && k > 0, GFS_ERR_BAD_ARG, "gfs_edge_scatter: bad argument");
    GFS_REQUIRE(k <= 64, GFS_ERR_UNSUPPORTED, "gfs_edge_scatter: k <= 64");
    const int64_t Mp = (int64_t)B * N, E = Mp * k;
    const size_t smem = (size_t)64 * (ES_PPB * k + 1) * sizeof(float);
    GFS_CUDA_OK(allow_smem(reinterpret_cast<const void*>(edge_scatter_kernel), (size_t)64 * (ES_PPB * 64 + 1) * sizeof(float)));
    edge_scatter_kernel<<<(unsigned)((Mp + ES_PPB - 1) / ES_PPB), 256, smem, static_cast<cudaStream_t>(stream)>>>(dH, idx, N, k, Mp, E, dpq);
    GFS_LAUNCH_OK("edge_scatter_kernel");
    return GFS_OK;
}

extern "C" int gfs_max_over_k_fwd(const float* a, int C, int64_t M, int k, float* y, int64_t ldy, uint8_t* arg, void* stream) {
    GFS_REQUIRE(a && y && arg && C > 0 && M > 0 && k > 0 && k <= 255, GFS_ERR_BAD_ARG, "gfs_max_over_k_fwd: bad argument");
    max_over_k_fwd_kernel<<<dim3((unsigned)((M + 255) / 256), C), 256, 0, static_cast<cudaStream_t>(stream)>>>(a, M, k, y, ldy, arg);
    GFS_LAUNCH_OK("max_over_k_fwd_kernel");
    return GFS_OK;
}

extern "C" int gfs_max_over_k_bwd(const float* dy, int64_t lddy, const uint8_t* arg, int C, int64_t M, int k, float* da, void* stream) {
    GFS_REQUIRE(dy && arg && da && C > 0 && M > 0 && k > 0, GFS_ERR_BAD_ARG, "gfs_max_over_k_bwd: bad argument");
    max_over_k_bwd_kernel<<<dim3((unsigned)((M + 255) / 256), C), 256, 0, static_cast<cudaStream_t>(stream)>>>(dy, lddy, arg, M, k, da);
    GFS_LAUNCH_OK("max_over_k_bwd_kernel");
    return GFS_OK;
}

extern "C" int gfs_dropout_mask(int64_t rows, int n, uint32_t seed, float keep, float* mask, void* stream) {
    GFS_REQUIRE(mask && rows > 0 && n > 0 && keep > 0.0f && keep <= 1.0f, GFS_ERR_BAD_ARG, "gfs_dropout_mask: bad argument");
    dropout_mask_kernel<<<(unsigned)((rows * n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(rows, n, seed, keep, mask);
    GFS_LAUNCH_OK("dropout_mask_kernel");
    return GFS_OK;
}

extern "C" int gfs_softmax_rows_fwd(const float* s, int64_t rows, int n, float scale, const float* mask, uint32_t seed, float keep,
                                    float* p0, float* p, void* stream) {
    GFS_REQUIRE(s && p0 && p && rows > 0 && n > 0 && keep > 0.0f, GFS_ERR_BAD_ARG, "gfs_softmax_rows_fwd: bad argument");
    GFS_REQUIRE(p != p0 || (!mask && keep >= 1.0f), GFS_ERR_BAD_ARG, "gfs_softmax_rows_fwd: dropout needs a separate p");
    softmax_rows_fwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(s, rows, n, scale, mask, seed, keep,
                                                                                                     p0, p);
    GFS_LAUNCH_OK("softmax_rows_fwd_kernel");
    return GFS_OK;
}

extern "C" int gfs_softmax_rows_bwd(const float* p0, const float* dp, const float* mask, uint32_t seed, float keep, int64_t rows, int n,
                                    float scale, float* ds, void* stream) {
    GFS_REQUIRE(p0 && dp && ds && rows > 0 && n > 0 && keep > 0.0f, GFS_ERR_BAD_ARG, "gfs_softmax_rows_bwd: bad argument");
    softmax_rows_bwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(p0, dp, mask, seed, keep, rows, n,
                                                                                                     scale, ds);
    GFS_LAUNCH_OK("softmax_rows_bwd_kernel");
    return GFS_OK;
}
