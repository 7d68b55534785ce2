// rowsel_tc.cu -- the "points x dictionary" contractions of rowsel.cu on tcgen05, with the integer result still bit-exact.
//
//   gfs_gw_project_tc    model/capl.py:344-353   cos = <gp_l2[g], ec>/max(|ec|,1e-12) -> softmax_g(10 cos), argmax_g
//   gfs_kmeans_assign_tc sklearn _k_means_lloyd.pyx:196-218 (behind get_basis.py:210): argmin_c (|c|^2 - 2 x.c)
//
// The (points x D) . (D x <=192) product is a real GEMM (2*192*192 flop per point against 768 bytes): on CUDA cores it
// is FFMA bound (rowsel.cu: 69 % FMA pipe), on the tensor cores it drops under the time HBM needs to deliver the points.
// What must not change is the INTEGER result (GW assignment / k-means label): it is defined by the pinned fp32 fma chain
// of oracle/gfs_oracle.c.  So the tensor cores compute S ~= x.g with a bf16 hi/lo split of both operands
// (x_h.g_h + x_h.g_l + x_l.g_h, fp32 accumulation in TMEM, |S - x.g| <= 2^-13.6 |x||g| even if every rounding aligned),
// every row keeps its best and second best score, and a row whose two best scores are closer than the error bound allows
// is appended to a re-check list: gfs::rowsel_recheck_kernel evaluates the pinned chain for exactly those rows (a warp per
// row) and overwrites their result.  Features (the softmax of the cosines) carry a 2e-2 tolerance and are taken from the
// tensor-core values directly.
//
// Persistent CTA, 24 warps:
//   warps 0-15  producers: fp32 channel-major points (coalesced over the 128 points of the tile) -> bf16 hi / lo operand
//               tiles in shared memory (K-major SWIZZLE_128B, 64 channels per stage), partial squared norms
//   (the dictionary's packed hi / lo image, rowsel_pack_kernel, is loaded ONCE per CTA by TMA and stays resident: 48 KiB per 64 channels)
//   warp  16    MMA issue (warp-uniform loop, one elected lane): 12 x tcgen05.mma 128x192x16 per stage
//   warps 20-23 epilogue: tcgen05.ld, best / second best, (GW) softmax features as bf16 act tiles, ambiguity test
#include <cstddef>

#include "fp32_tile.cuh"

namespace gfs {

constexpr int RT_ROWS = 128;      // points per tile
constexpr int RT_N = 192;         // dictionary columns of one MMA (zero padded)
constexpr int RT_PW = 16;          // producer warps: four 16-channel quarters of a 64-channel stage x 128 points
constexpr int RT_THREADS = 32 * RT_PW + 32 + 96 + 128;   // + MMA warp (16), 3 idle warps, 4 epilogue warps (20-23)
constexpr uint32_t RT_BTILE = RT_N * 128;   // bytes of one 64-channel dictionary tile (hi or lo)

struct RtCtl {
    uint64_t a_full[2], a_empty[2], b_full, accf[2], acce[2];
    uint32_t tmem_base;
};
struct RtSmem {                   // 1024-byte aligned; every operand tile starts on a 1024-byte boundary (SWIZZLE_128B)
    uint8_t A[2][2][16384];       // [stage][hi | lo]  128 points x 64 channels
    float xn[4][4][RT_ROWS];      // [tile & 3][channel quarter] partial squared norms
    float cn[RT_N + 64];          // k-means: squared norms of the centres (padded: B below stays 1024-byte aligned)
    uint8_t B[1][2][RT_BTILE];    // [k-block][hi | lo]  192 entries x 64 channels: the WHOLE dictionary stays resident (D/64 k-blocks,
                                  // then the RtCtl block)
};
static_assert(offsetof(RtSmem, B) % 1024 == 0, "dictionary tiles must be 1024-byte aligned");

enum { RT_GW = 0, RT_KMEANS = 1, RT_KMEANS_PM = 2 };   // _PM: points are rows of a row-major (n, D) matrix (contiguous 128-point tiles)
// RT_PANEL (or-ed into a layout): one panel of <= 192 words of a dictionary of up to 512 (see rt_run_wide).  The panel
// instances reuse three arguments the single-panel ones leave unused in their layout: kb0 = the panel's first word,
// cos_cm = the per-row scratch the panels share, kblocks != 0 on the last panel (k-means).
constexpr int RT_PANEL = 4;
constexpr int RT_MAXK = 512;      // widest dictionary: ceil(512 / 192) = 3 panels

// dict_t (D, Gp) fp32 channel-major -> per 64-channel block: [hi tile | lo tile], 192 rows x 128 B, K-major SWIZZLE_128B.
// Also the largest squared norm of an entry (k-means: scales the ambiguity bound).
__global__ void rowsel_pack_kernel(const float* __restrict__ dict_t, int D, int G, int Gp, uint8_t* __restrict__ img) {
    pdl_enter();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int chunks = D >> 3;
    if (i >= RT_N * chunks) return;
    const int j = i / chunks, qq = i - j * chunks;          // entry, 8-channel chunk
    const int kb = qq >> 3, q = qq & 7;
    uint32_t hp[4], lp[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int c = qq * 8 + 2 * e;
        const float v0 = j < G ? dict_t[(int64_t)c * Gp + j] : 0.0f, v1 = j < G ? dict_t[(int64_t)(c + 1) * Gp + j] : 0.0f;
        const __nv_bfloat16 h0 = __float2bfloat16_rn(v0), h1 = __float2bfloat16_rn(v1);
        __nv_bfloat162 hh;
        hh.x = h0;
        hh.y = h1;
        hp[e] = *reinterpret_cast<uint32_t*>(&hh);
        lp[e] = pack_bf16x2(v0 - __bfloat162float(h0), v1 - __bfloat162float(h1));
    }
    uint8_t* t = img + (size_t)kb * 2 * RT_BTILE;
    *reinterpret_cast<uint4*>(t + sw128(j, q)) = make_uint4(hp[0], hp[1], hp[2], hp[3]);
    *reinterpret_cast<uint4*>(t + RT_BTILE + sw128(j, q)) = make_uint4(lp[0], lp[1], lp[2], lp[3]);
}
// k-means: the largest squared norm of a centre scales the ambiguity bound; also clears the re-check counter
__global__ void rowsel_cmax_kernel(const float* __restrict__ cnorm, int G, float* __restrict__ cmax2, int32_t* __restrict__ cnt) {
    pdl_enter();
    float m = 0.0f;
    if (cnorm)
        for (int j = threadIdx.x; j < G; j += 32) m = fmaxf(m, cnorm[j]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (threadIdx.x == 0) {
        cmax2[0] = m;
        *cnt = 0;
    }
}

__device__ __forceinline__ float rt_ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// best, second best and the FIRST index of the best among 32 scores held in registers.  MAXM: larger is better.
// A tournament tree (a pair keeps its best and its runner-up; merging two pairs is three independent min/max), not a
// running update: the epilogue thread is alone on its scheduler slot and would otherwise crawl along one dependent chain.
template <bool MAXM>
__device__ __forceinline__ void rt_best2(const float (&v)[32], float& best, float& second, int& idx) {
    float m[16], r2[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        m[i] = MAXM ? fmaxf(v[2 * i], v[2 * i + 1]) : fminf(v[2 * i], v[2 * i + 1]);
        r2[i] = MAXM ? fminf(v[2 * i], v[2 * i + 1]) : fmaxf(v[2 * i], v[2 * i + 1]);
    }
#pragma unroll
    for (int w = 8; w >= 1; w >>= 1) {
#pragma unroll
        for (int i = 0; i < w; ++i) {
            const float a = m[i], b = m[i + w];
            if (MAXM) {
                m[i] = fmaxf(a, b);
                r2[i] = fmaxf(fmaxf(fminf(a, b), r2[i]), r2[i + w]);
            } else {
                m[i] = fminf(a, b);
                r2[i] = fminf(fminf(fmaxf(a, b), r2[i]), r2[i + w]);
            }
        }
    }
    best = m[0];
    second = r2[0];
    int ix = 31;
#pragma unroll
    for (int c = 30; c >= 0; --c) ix = v[c] == best ? c : ix;
    idx = ix;
}

template <int MODE>
__global__ void __launch_bounds__(RT_THREADS, 1)
rowsel_tc_kernel(const float* __restrict__ x, int64_t bstride, int64_t cstride, int D, int N, int64_t M, int ntiles,
                 const uint8_t* __restrict__ img, int G, int Gp, const float* __restrict__ cnorm, const float* __restrict__ cmax2,
                 uint8_t* __restrict__ cos_act, int kblocks, int kb0, float* __restrict__ cos_cm, int32_t* __restrict__ sel,
                 int32_t* __restrict__ recheck, int32_t* __restrict__ recheck_cnt) {
    constexpr int L = MODE & 3;
    constexpr bool PANEL = (MODE & RT_PANEL) != 0;
    pdl_enter();
    extern __shared__ unsigned char smem_raw[];
    RtSmem& sm = *reinterpret_cast<RtSmem*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nkb = D >> 6;
    RtCtl& s = *reinterpret_cast<RtCtl*>(reinterpret_cast<uint8_t*>(&sm) + offsetof(RtSmem, B) + (size_t)nkb * 2 * RT_BTILE);

    if (tid < RT_N) sm.cn[tid] = (cnorm && tid < G) ? cnorm[tid] : 0.0f;
    if (warp == RT_PW) {
        if (lane == 0) {
            for (int i = 0; i < 2; ++i) {
                mbar_init(&s.a_full[i], RT_PW);
                mbar_init(&s.a_empty[i], 1);
                mbar_init(&s.accf[i], 1);
                mbar_init(&s.acce[i], 4);
            }
            mbar_init(&s.b_full, 1);
            mbar_fence_init();
            // the dictionary image: one TMA bulk copy per k-block, once per CTA
            mbar_arrive_expect_tx(&s.b_full, (uint32_t)nkb * 2u * RT_BTILE);
            for (int kb = 0; kb < nkb; ++kb) tma_load_1d(sm.B[kb][0], img + (size_t)kb * 2 * RT_BTILE, 2u * RT_BTILE, &s.b_full);
        }
        __syncwarp();
        tmem_alloc(&s.tmem_base, 512);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s.tmem_base;

    if (warp < RT_PW) {
        // =============================== producers ===============================
        // One flat sequence of (tile, 64-channel block) stages; the channels of the next TWO stages (also across a tile
        // boundary) are in flight in registers while the current one is converted: the loop is bound by DRAM latency otherwise.
        const int r = tid & 127, qt = tid >> 7;             // point row, 16-channel quarter of the 64-channel stage
        const int my_tiles = blockIdx.x < ntiles ? (ntiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;
        const int S = my_tiles * nkb;
        auto load16 = [&](int it, float (&dst)[16]) {         // stage it = (tile it / nkb, block it % nkb)
            const int lt_ = it / nkb, kb_ = it - lt_ * nkb;
            const int64_t m = ((int64_t)blockIdx.x + (int64_t)lt_ * gridDim.x) * RT_ROWS + r;
            const bool valid = it < S && m < M;
            const int64_t mm = valid ? m : 0;
            if (L == RT_KMEANS_PM) {
                // point-major: the thread's 16 channels are 64 contiguous bytes of its own row
                const float4* xp4 = reinterpret_cast<const float4*>(x + mm * D + kb_ * 64 + qt * 16);
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float4 t = valid ? __ldg(xp4 + c) : make_float4(0.f, 0.f, 0.f, 0.f);
                    dst[4 * c] = t.x;
                    dst[4 * c + 1] = t.y;
                    dst[4 * c + 2] = t.z;
                    dst[4 * c + 3] = t.w;
                }
                return;
            }
            const float* xp;
            if (L == RT_GW) {
                const int64_t b = mm / N;
                xp = x + b * bstride + (mm - b * N);
            } else {
                xp = x + mm;
            }
            xp += (int64_t)(kb_ * 64 + qt * 16) * cstride;
#pragma unroll
            for (int c = 0; c < 16; ++c) dst[c] = valid ? __ldg(xp + (int64_t)c * cstride) : 0.0f;
        };
        float v0[16], v1[16], v2[16];
        load16(0, v0);
        load16(1, v1);
        float nrm = 0.0f;
        int lt = 0, kb = 0;
        for (int it = 0; it < S; ++it) {
            const int st = it & 1;
            load16(it + 2, v2);
            mbar_wait(&s.a_empty[st], ((it >> 1) & 1) ^ 1);
            uint8_t* ah = sm.A[st][0];
            uint8_t* al = sm.A[st][1];
            if (kb == 0) nrm = 0.0f;
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                uint32_t hp[4], lp[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float a0 = v0[q * 8 + 2 * e], a1 = v0[q * 8 + 2 * e + 1];
                    // hi = the two values rounded to bf16 (one packed conversion), lo = the rounded residuals
                    const uint32_t h = pack_bf16x2(a0, a1);
                    hp[e] = h;
                    lp[e] = pack_bf16x2(a0 - __uint_as_float(h << 16), a1 - __uint_as_float(h & 0xffff0000u));
                    nrm = fmaf(a0, a0, fmaf(a1, a1, nrm));
                }
                const uint32_t o = sw128(r, qt * 2 + q);
                *reinterpret_cast<uint4*>(ah + o) = make_uint4(hp[0], hp[1], hp[2], hp[3]);
                *reinterpret_cast<uint4*>(al + o) = make_uint4(lp[0], lp[1], lp[2], lp[3]);
            }
            // the partial norm goes out BEFORE the tile's last arrive: that release orders it before the epilogue's read
            if (kb == nkb - 1) sm.xn[lt & 3][qt][r] = nrm;
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(&s.a_full[st]);
#pragma unroll
            for (int c = 0; c < 16; ++c) {
                v0[c] = v1[c];
                v1[c] = v2[c];
            }
            if (++kb == nkb) {
                kb = 0;
                ++lt;
            }
        }
    } else if (warp < RT_PW + 4) {
        // =============================== MMA issue (warp 16; warps 17-19 only complete its warpgroup for setmaxnreg) ===============================
        reg_dealloc<24>();
        if (warp == RT_PW) {
        const uint32_t idesc = umma_idesc_bf16(128, RT_N);
        const uint64_t a0 = umma_desc_sw128(smem_u32(sm.A[0][0]));
        const uint64_t b0 = umma_desc_sw128(smem_u32(sm.B[0][0]));
        constexpr uint32_t A_ST = 2 * 16384 >> 4, A_LO = 16384 >> 4, B_ST = 2 * RT_BTILE >> 4, B_LO = RT_BTILE >> 4;
        int it = 0, lt = 0;
        mbar_wait(&s.b_full, 0);
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++lt) {
            const int acc = lt & 1;
            mbar_wait(&s.acce[acc], ((lt >> 1) & 1) ^ 1);
            tc_fence_after();
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                const int st = it & 1;
                mbar_wait(&s.a_full[st], (it >> 1) & 1);
                tc_fence_after();
                if (elect_one()) {
                    const uint64_t aB = a0 + (uint64_t)(st * A_ST), bB = b0 + (uint64_t)(kb * B_ST);
                    const uint32_t d = tmem + acc * 256;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        umma_bf16(d, aB + ks * 2, bB + ks * 2, idesc, (kb | ks) ? 1u : 0u);
                        umma_bf16(d, aB + ks * 2, bB + B_LO + ks * 2, idesc, 1u);
                        umma_bf16(d, aB + A_LO + ks * 2, bB + ks * 2, idesc, 1u);
                    }
                    umma_commit(&s.a_empty[st]);
                    if (kb == nkb - 1) umma_commit(&s.accf[acc]);
                }
                __syncwarp();
            }
        }
        }
    } else if (warp >= RT_PW + 4) {
        // =============================== epilogue: one thread per point ===============================
        reg_alloc<128>();                                     // 24 warps x 80 registers at launch: the MMA group's dec frees 4 x 32 x 56 = 7168,
                                                              // this inc takes 4 x 32 x 48 = 6144 (asking for more than was freed never returns)
        const int quarter = warp & 3;
        const int row = quarter * 32 + lane;
        const uint32_t tbase = tmem + ((uint32_t)(quarter * 32) << 16);
        const float cmax = L != RT_GW ? sqrtf(__ldg(cmax2)) : 0.0f;
        int lt = 0;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++lt) {
            const int acc = lt & 1;
            mbar_wait_backoff(&s.accf[acc], (lt >> 1) & 1, 64);
            tc_fence_after();
            const int64_t m = (int64_t)tile * RT_ROWS + row;
            const bool valid = m < M;
            const float nrm = (sm.xn[lt & 3][0][row] + sm.xn[lt & 3][1][row]) + (sm.xn[lt & 3][2][row] + sm.xn[lt & 3][3][row]);
            const uint32_t t0 = tbase + acc * 256;
            uint32_t rr[32];
            float b1, b2;
            int i1 = 0;
            if constexpr (PANEL && L == RT_GW) {
                // this panel's 10 cos into the column-major scratch [|x|^2 | word 0 | word 1 | ...] (rows of M): the softmax
                // needs every word of the row, rowsel_gw_finish_kernel takes it from there
                const float inv = 10.0f / fmaxf(sqrtf(nrm), 1e-12f);
                float* out = cos_cm + (int64_t)(1 + kb0) * M + m;
                if (valid && kb0 == 0) cos_cm[m] = nrm;
                for (int ch = 0; ch * 32 < G; ++ch) {
                    tmem_ld32(t0 + ch * 32, rr);
                    tmem_ld_wait32(rr);
                    if (valid) {
#pragma unroll
                        for (int c = 0; c < 32; ++c)
                            if (ch * 32 + c < G) out[(int64_t)(ch * 32 + c) * M] = __uint_as_float(rr[c]) * inv;
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&s.acce[acc]);
                continue;
            }
            if (L == RT_GW) {
                const float inv = 10.0f / fmaxf(sqrtf(nrm), 1e-12f);
                b1 = -INFINITY;
                b2 = -INFINITY;
                for (int ch = 0; ch * 32 < G; ++ch) {
                    tmem_ld32(t0 + ch * 32, rr);
                    tmem_ld_wait32(rr);
                    float lg[32];
#pragma unroll
                    for (int c = 0; c < 32; ++c) lg[c] = ch * 32 + c < G ? __uint_as_float(rr[c]) * inv : -INFINITY;
                    float cb, cs;
                    int ci;
                    rt_best2<true>(lg, cb, cs, ci);
                    if (cb > b1) {                       // an equal best in a later chunk keeps the earlier (lower) index
                        b2 = fmaxf(b1, cs);
                        b1 = cb;
                        i1 = ch * 32 + ci;
                    } else {
                        b2 = fmaxf(b2, cb);
                    }
                }
                // softmax over the words: exp(10 cos - max) as ONE fma and ONE ex2.approx per element (the library expf carries a
                // range fix-up: two predicated multiplies and a compare per element, and this single-warp-per-scheduler epilogue is
                // what the kernel waits for -- ncu source page, r2); chunks entirely inside G run without the column predicate
                const float inv2 = inv * 1.4426950408889634f, nb2 = -b1 * 1.4426950408889634f;
                float sum4[4] = {0.0f, 0.0f, 0.0f, 0.0f};           // four independent add chains instead of one 150 long
                for (int ch = 0; ch * 32 < G; ++ch) {
                    tmem_ld32(t0 + ch * 32, rr);
                    tmem_ld_wait32(rr);
                    if (ch * 32 + 32 <= G) {
#pragma unroll
                        for (int c = 0; c < 32; ++c) sum4[c & 3] += rt_ex2(fmaf(__uint_as_float(rr[c]), inv2, nb2));
                    } else {
#pragma unroll
                        for (int c = 0; c < 32; ++c) sum4[c & 3] += ch * 32 + c < G ? rt_ex2(fmaf(__uint_as_float(rr[c]), inv2, nb2)) : 0.0f;
                    }
                }
                const float rs = 1.0f / ((sum4[0] + sum4[1]) + (sum4[2] + sum4[3]));
                for (int ch = 0; ch * 32 < Gp; ++ch) {
                    tmem_ld32(t0 + ch * 32, rr);
                    tmem_ld_wait32(rr);
                    if (valid) {
                        float e[32];
                        if (ch * 32 + 32 <= G) {
#pragma unroll
                            for (int c = 0; c < 32; ++c) e[c] = rt_ex2(fmaf(__uint_as_float(rr[c]), inv2, nb2)) * rs;
                        } else {
#pragma unroll
                            for (int c = 0; c < 32; ++c) e[c] = ch * 32 + c < G ? rt_ex2(fmaf(__uint_as_float(rr[c]), inv2, nb2)) * rs : 0.0f;
                        }
                        if (cos_act) {
                            uint8_t* tl = cos_act + (((m >> 7) * kblocks + kb0 + (ch >> 1)) * 16384);
                            const uint32_t rw = (uint32_t)(m & 127);
#pragma unroll
                            for (int q = 0; q < 4; ++q)
                                *reinterpret_cast<uint4*>(tl + sw128(rw, (ch & 1) * 4 + q)) =
                                    make_uint4(pack_bf16x2(e[q * 8], e[q * 8 + 1]), pack_bf16x2(e[q * 8 + 2], e[q * 8 + 3]),
                                               pack_bf16x2(e[q * 8 + 4], e[q * 8 + 5]), pack_bf16x2(e[q * 8 + 6], e[q * 8 + 7]));
                        }
                        if (cos_cm) {
                            const int64_t b = m / N, n = m - b * N;
#pragma unroll
                            for (int c = 0; c < 32; ++c)
                                if (ch * 32 + c < G) cos_cm[(b * G + ch * 32 + c) * N + n] = e[c];
                        }
                    }
                }
            } else {
                b1 = INFINITY;
                b2 = INFINITY;
                for (int ch = 0; ch * 32 < G; ++ch) {
                    tmem_ld32(t0 + ch * 32, rr);
                    tmem_ld_wait32(rr);
                    float sc[32];
#pragma unroll
                    for (int c = 0; c < 32; c += 4) {
                        const float4 cn4 = *reinterpret_cast<const float4*>(sm.cn + ch * 32 + c);
                        sc[c] = ch * 32 + c < G ? fmaf(-2.0f, __uint_as_float(rr[c]), cn4.x) : INFINITY;
                        sc[c + 1] = ch * 32 + c + 1 < G ? fmaf(-2.0f, __uint_as_float(rr[c + 1]), cn4.y) : INFINITY;
                        sc[c + 2] = ch * 32 + c + 2 < G ? fmaf(-2.0f, __uint_as_float(rr[c + 2]), cn4.z) : INFINITY;
                        sc[c + 3] = ch * 32 + c + 3 < G ? fmaf(-2.0f, __uint_as_float(rr[c + 3]), cn4.w) : INFINITY;
                    }
                    float cb, cs;
                    int ci;
                    rt_best2<false>(sc, cb, cs, ci);
                    if (cb < b1) {                       // an equal best in a later chunk keeps the earlier (lower) index
                        b2 = fminf(b1, cs);
                        b1 = cb;
                        i1 = ch * 32 + ci;
                    } else {
                        b2 = fminf(b2, cb);
                    }
                }
            }
            // hand the accumulator back
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&s.acce[acc]);
            if (valid) {
                if constexpr (PANEL) {
                    // (best, second best, index) of the panels so far, merged in ascending panel order: the earlier panels
                    // hold the lower indices, so an equal score keeps theirs
                    float* rs = cos_cm + 4 * m;
                    i1 += kb0;
                    if (kb0 > 0) {
                        const float pb1 = rs[0];
                        if (b1 < pb1) {
                            b2 = fminf(b2, pb1);
                        } else {
                            b2 = fminf(rs[1], b1);
                            b1 = pb1;
                            i1 = __float_as_int(rs[2]);
                        }
                    }
                    if (!kblocks) {
                        *reinterpret_cast<float4*>(rs) = make_float4(b1, b2, __int_as_float(i1), 0.0f);
                        continue;
                    }
                }
                sel[m] = i1;
                // the two best scores closer than the error bound of the tensor-core product (x 3 safety, see the header):
                // the pinned fp32 chain decides (rowsel_recheck_kernel)
                bool amb;
                if (L == RT_GW) amb = !(b1 - b2 > 5e-3f) || !(nrm > 1e-20f);
                else amb = !(b2 - b1 > 0x1p-10f * sqrtf(nrm) * cmax);
                if (amb) recheck[atomicAdd(recheck_cnt, 1)] = (int32_t)m;
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == RT_PW) {
        tc_fence_after();
        tmem_dealloc(tmem, 512);
    }
}

// One warp per listed row: the pinned fp32 chains (c ascending) of every dictionary entry, exactly as rowsel.cu evaluates
// them; the winner (ties -> lowest index) overwrites the tensor-core result.  A row is a chain of D/8 dictionary batches
// (48 L2 loads each); the batches are double buffered in registers so that the loads of batch b+1 fly while the 8 x 7 fmas
// of batch b issue, and the row itself is staged in shared memory once (broadcast LDS instead of a shuffle per channel).
// (Measured alternatives, r2: four rows per warp to reuse the dictionary values divides the L2 traffic by four but leaves
// only ~250 warps on the GPU for ~1000 ambiguous rows: slower.  The re-check is latency bound, not traffic bound.)
constexpr int RC_WARPS = 8;
// RT_PANEL instance (dictionaries of 193..512 words): the row is staged once, then the 192-column groups run one after
// the other with the same chains and the same per-lane pick; a later group replaces the running best only with a strictly
// better score, so ties still go to the lowest index over all words.
template <int MODE>
__global__ void __launch_bounds__(32 * RC_WARPS)
rowsel_recheck_kernel(const float* __restrict__ x, int64_t bstride, int64_t cstride, int D, int N, const float* __restrict__ dict_t,
                      int G, int Gp, const float* __restrict__ cnorm, const int32_t* __restrict__ recheck,
                      const int32_t* __restrict__ recheck_cnt, int32_t* __restrict__ sel) {
    constexpr int L = MODE & 3;
    constexpr bool PANEL = (MODE & RT_PANEL) != 0;
    pdl_enter();
    __shared__ float xs_all[RC_WARPS][256];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    float* xs = xs_all[wib];
    const int nrows = *recheck_cnt;
    const int nb = (D + 7) >> 3;
    int g0 = 0;                                      // first column of the current group (always 0 without RT_PANEL)
    auto load = [&](float (&g)[8][6], int bk) {
#pragma unroll
        for (int c2 = 0; c2 < 8; ++c2) {
            const int c = bk * 8 + c2;
            const float* gp = dict_t + (int64_t)c * Gp + g0;
#pragma unroll
            for (int j = 0; j < 6; ++j) g[c2][j] = (g0 + j * 32 + lane < G && c < D) ? __ldg(gp + j * 32 + lane) : 0.0f;
        }
    };
    for (int w = blockIdx.x * RC_WARPS + wib; w < nrows; w += gridDim.x * RC_WARPS) {
        const int64_t m = recheck[w];
        const float* xp;
        if (L == RT_GW) {
            const int64_t b = m / N;
            xp = x + b * bstride + (m - b * N);
        } else if (L == RT_KMEANS_PM) {
            xp = x + m * D;                          // cstride == 1
        } else {
            xp = x + m;
        }
        float ga[8][6], gb[8][6];
        g0 = 0;
        load(ga, 0);
        __syncwarp();
        for (int c = lane; c < D; c += 32) xs[c] = __ldg(xp + (int64_t)c * cstride);
        __syncwarp();
        float best = L == RT_GW ? -INFINITY : INFINITY;
        int bi = 0x7fffffff;
        for (;;) {
            float acc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            float nrm = 0.0f;
            auto compute = [&](const float (&g)[8][6], int bk) {
#pragma unroll
                for (int c2 = 0; c2 < 8; ++c2) {
                    const int c = bk * 8 + c2;
                    if (c < D) {                         // uniform
                        const float a = xs[c];
                        nrm = fmaf(a, a, nrm);
#pragma unroll
                        for (int j = 0; j < 6; ++j)
                            if (g0 + j * 32 + lane < G) acc[j] = fmaf(a, g[c2][j], acc[j]);
                    }
                }
            };
#pragma unroll 1
            for (int bk = 0; bk < nb; bk += 2) {
                if (bk + 1 < nb) load(gb, bk + 1);
                compute(ga, bk);
                if (bk + 2 < nb) load(ga, bk + 2);
                if (bk + 1 < nb) compute(gb, bk + 1);
            }
            const float inv = 10.0f / fmaxf(sqrtf(nrm), 1e-12f);
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                const int col = g0 + j * 32 + lane;
                if (col < G) {
                    const float sc = L == RT_GW ? acc[j] * inv : fmaf(-2.0f, acc[j], __ldg(cnorm + col));
                    const bool better = L == RT_GW ? (sc > best || (sc == best && col < bi)) : (sc < best || (sc == best && col < bi));
                    if (better) {
                        best = sc;
                        bi = col;
                    }
                }
            }
            if constexpr (!PANEL) break;
            g0 += RT_N;
            if (g0 >= G) break;
            load(ga, 0);
        }
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            const bool better = L == RT_GW ? (ob > best || (ob == best && oi < bi)) : (ob < best || (ob == best && oi < bi));
            if (better) {
                best = ob;
                bi = oi;
            }
        }
        if (lane == 0) sel[m] = bi;
    }
}

// GW projection over a panelled dictionary, one thread per row, after the last panel: best / second best / first index of
// the best over the scratch's G columns, the ambiguity test of rowsel_tc_kernel, and the softmax features (bf16 act tiles
// at kb0 with the padding columns zero, optional (B, G, N) fp32 copy) -- the single-panel epilogue, taken from the scratch.
__global__ void __launch_bounds__(256)
rowsel_gw_finish_kernel(const float* __restrict__ scr, int64_t M, int N, int G, int Gp, uint8_t* __restrict__ cos_act, int kblocks,
                        int kb0, float* __restrict__ cos_cm, int32_t* __restrict__ sel, int32_t* __restrict__ recheck,
                        int32_t* __restrict__ recheck_cnt) {
    pdl_enter();
    const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    const float nrm = scr[m];
    const float* v = scr + M + m;                    // word j at v[j * M]
    float b1 = -INFINITY, b2 = -INFINITY;
    int i1 = 0;
    for (int j = 0; j < G; ++j) {
        const float t = v[(int64_t)j * M];
        if (t > b1) {
            b2 = b1;
            b1 = t;
            i1 = j;
        } else {
            b2 = fmaxf(b2, t);
        }
    }
    const float l2e = 1.4426950408889634f, nb2 = -b1 * l2e;
    float s0 = 0.0f, s1 = 0.0f;
    int j = 0;
    for (; j + 1 < G; j += 2) {
        s0 += rt_ex2(fmaf(v[(int64_t)j * M], l2e, nb2));
        s1 += rt_ex2(fmaf(v[(int64_t)(j + 1) * M], l2e, nb2));
    }
    if (j < G) s0 += rt_ex2(fmaf(v[(int64_t)j * M], l2e, nb2));
    const float rs = 1.0f / (s0 + s1);
    const int64_t b = m / N, n = m - b * N;
    for (int j0 = 0; j0 < Gp; j0 += 8) {
        float e[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) e[c] = j0 + c < G ? rt_ex2(fmaf(v[(int64_t)(j0 + c) * M], l2e, nb2)) * rs : 0.0f;
        if (cos_act) {
            uint8_t* tl = cos_act + (((m >> 7) * kblocks + kb0 + (j0 >> 6)) * 16384);
            *reinterpret_cast<uint4*>(tl + sw128((uint32_t)(m & 127), (j0 >> 3) & 7)) =
                make_uint4(pack_bf16x2(e[0], e[1]), pack_bf16x2(e[2], e[3]), pack_bf16x2(e[4], e[5]), pack_bf16x2(e[6], e[7]));
        }
        if (cos_cm) {
#pragma unroll
            for (int c = 0; c < 8; ++c)
                if (j0 + c < G) cos_cm[(b * G + j0 + c) * N + n] = e[c];
        }
    }
    sel[m] = i1;
    if (!(b1 - b2 > 5e-3f) || !(nrm > 1e-20f)) recheck[atomicAdd(recheck_cnt, 1)] = (int32_t)m;
}

struct RtPlan {
    size_t off_img, off_cmax, off_cnt, off_list, off_scr, total;
};
// Kp > 192 (rt_run_wide): one packed image per panel and the per-row scratch the panels share -- (best, second best, index)
// as a float4 for k-means, |x|^2 and the 10 cos of every word (column-major, (1 + Kp) x rows fp32) for the GW projection
static RtPlan rt_plan(int64_t rows, int D, int Kp = RT_N, bool gw = false) {
    const int panels = Kp > RT_N ? (Kp + RT_N - 1) / RT_N : 1;
    RtPlan p;
    p.off_img = 0;
    size_t o = (size_t)panels * (D >> 6) * 2 * RT_BTILE;
    p.off_cmax = o;
    o += 256;
    p.off_cnt = o;
    o += 256;
    p.off_list = o;
    o += (size_t)rows * 4;
    o = (o + 255) / 256 * 256;
    p.off_scr = o;
    if (panels > 1) o += gw ? (size_t)(1 + Kp) * rows * 4 : (size_t)rows * 16;
    p.total = (o + 255) / 256 * 256;
    return p;
}

template <int MODE>
static int rt_run(const char* who, const float* x, int64_t bstride, int64_t cstride, int D, int N, int64_t M, const float* dict_t, int G,
                  int Gp, const float* cnorm, void* cos_act, int kblocks, int kb0, float* cos_cm, int32_t* sel, void* workspace,
                  int64_t workspace_bytes, cudaStream_t st) {
    const RtPlan p = rt_plan(M, D);
    GFS_REQUIRE(workspace && workspace_bytes >= (int64_t)p.total && (reinterpret_cast<uintptr_t>(workspace) & 255) == 0, GFS_ERR_BAD_ARG,
                "%s: workspace of %lld bytes (256-byte aligned) needed, got %lld", who, (long long)p.total, (long long)workspace_bytes);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    float* cmax2 = reinterpret_cast<float*>(ws + p.off_cmax);
    int32_t* cnt = reinterpret_cast<int32_t*>(ws + p.off_cnt);
    int32_t* list = reinterpret_cast<int32_t*>(ws + p.off_list);
    const int pk = RT_N * (D >> 3);
    launch_pdl(rowsel_pack_kernel, dim3((unsigned)((pk + 255) / 256)), dim3(256), 0, st,
        dict_t, D, G, Gp, ws);
    GFS_LAUNCH_OK("rowsel_pack_kernel");
    launch_pdl(rowsel_cmax_kernel, dim3((unsigned)(1)), dim3(32), 0, st,
        MODE != RT_GW ? cnorm : nullptr, G, cmax2, cnt);
    GFS_LAUNCH_OK("rowsel_cmax_kernel");
    const int ntiles = (int)((M + RT_ROWS - 1) / RT_ROWS);
    const int sms = sm_count();
    GFS_REQUIRE(sms > 0, GFS_ERR_CUDA, "%s: cannot query the device", who);
    const size_t smem = offsetof(RtSmem, B) + (size_t)(D >> 6) * 2 * RT_BTILE + sizeof(RtCtl) + 1024;
    GFS_REQUIRE(smem <= 227 * 1024, GFS_ERR_UNSUPPORTED, "%s: D=%d: the resident dictionary does not fit shared memory (use the fp32 entry point)", who, D);
    GFS_CUDA_OK(allow_smem(reinterpret_cast<const void*>(rowsel_tc_kernel<MODE>), smem));
    launch_pdl(rowsel_tc_kernel<MODE>, dim3((unsigned)(ntiles < sms ? ntiles : sms)), dim3(RT_THREADS), smem, st,
        x, bstride, cstride, D, N, M, ntiles, ws, G, Gp, cnorm, cmax2, static_cast<uint8_t*>(cos_act), kblocks, kb0, cos_cm, sel, list, cnt);
    GFS_LAUNCH_OK("rowsel_tc_kernel");
    launch_pdl(rowsel_recheck_kernel<MODE>, dim3((unsigned)(sms * 2)), dim3(256), 0, st,
        x, bstride, cstride, D, N, dict_t, G, Gp, cnorm, list, cnt, sel);
    GFS_LAUNCH_OK("rowsel_recheck_kernel");
    return GFS_OK;
}

// Dictionaries of 193..512 words: panels of 192 words, each packed into its own image.  Every panel is one persistent pass
// of rowsel_tc_kernel over all the points with that panel resident (ceil(G / 192) passes over X); k-means merges the panels
// row by row in ascending order inside the epilogue (the last panel writes the label and applies the ambiguity bound, with
// max|c| over all K), the GW projection writes the scores of every word and rowsel_gw_finish_kernel takes the softmax.  The
// re-check then evaluates the pinned chains over all the words.
template <int L>
static int rt_run_wide(const char* who, const float* x, int64_t bstride, int64_t cstride, int D, int N, int64_t M, const float* dict_t,
                       int G, int Gp, const float* cnorm, void* cos_act, int kblocks, int kb0, float* cos_cm, int32_t* sel, void* workspace,
                       int64_t workspace_bytes, cudaStream_t st) {
    const RtPlan p = rt_plan(M, D, Gp, L == RT_GW);
    GFS_REQUIRE(workspace && workspace_bytes >= (int64_t)p.total && (reinterpret_cast<uintptr_t>(workspace) & 255) == 0, GFS_ERR_BAD_ARG,
                "%s: workspace of %lld bytes (256-byte aligned) needed, got %lld", who, (long long)p.total, (long long)workspace_bytes);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    float* cmax2 = reinterpret_cast<float*>(ws + p.off_cmax);
    int32_t* cnt = reinterpret_cast<int32_t*>(ws + p.off_cnt);
    int32_t* list = reinterpret_cast<int32_t*>(ws + p.off_list);
    float* scr = reinterpret_cast<float*>(ws + p.off_scr);
    const int npan = (G + RT_N - 1) / RT_N;
    const size_t pimg = (size_t)(D >> 6) * 2 * RT_BTILE;
    const int pk = RT_N * (D >> 3);
    for (int q = 0; q < npan; ++q) {
        const int off = q * RT_N, w = G - off < RT_N ? G - off : RT_N;
        launch_pdl(rowsel_pack_kernel, dim3((unsigned)((pk + 255) / 256)), dim3(256), 0, st,
            dict_t + off, D, w, Gp, ws + q * pimg);
        GFS_LAUNCH_OK("rowsel_pack_kernel");
    }
    launch_pdl(rowsel_cmax_kernel, dim3((unsigned)(1)), dim3(32), 0, st,
        L != RT_GW ? cnorm : nullptr, G, cmax2, cnt);
    GFS_LAUNCH_OK("rowsel_cmax_kernel");
    const int ntiles = (int)((M + RT_ROWS - 1) / RT_ROWS);
    const int sms = sm_count();
    GFS_REQUIRE(sms > 0, GFS_ERR_CUDA, "%s: cannot query the device", who);
    const size_t smem = offsetof(RtSmem, B) + pimg + sizeof(RtCtl) + 1024;
    GFS_REQUIRE(smem <= 227 * 1024, GFS_ERR_UNSUPPORTED, "%s: D=%d: the resident dictionary panel does not fit shared memory", who, D);
    GFS_CUDA_OK(allow_smem(reinterpret_cast<const void*>(rowsel_tc_kernel<L | RT_PANEL>), smem));
    for (int q = 0; q < npan; ++q) {
        const int off = q * RT_N, w = G - off < RT_N ? G - off : RT_N;
        launch_pdl(rowsel_tc_kernel<L | RT_PANEL>, dim3((unsigned)(ntiles < sms ? ntiles : sms)), dim3(RT_THREADS), smem, st,
            x, bstride, cstride, D, N, M, ntiles, ws + q * pimg, w, Gp, L != RT_GW ? cnorm + off : nullptr, cmax2, nullptr,
            q == npan - 1 ? 1 : 0, off, scr, sel, list, cnt);
        GFS_LAUNCH_OK("rowsel_tc_kernel<panel>");
    }
    if (L == RT_GW) {
        launch_pdl(rowsel_gw_finish_kernel, dim3((unsigned)((M + 255) / 256)), dim3(256), 0, st,
            scr, M, N, G, Gp, static_cast<uint8_t*>(cos_act), kblocks, kb0, cos_cm, sel, list, cnt);
        GFS_LAUNCH_OK("rowsel_gw_finish_kernel");
    }
    launch_pdl(rowsel_recheck_kernel<L | RT_PANEL>, dim3((unsigned)(sms * 2)), dim3(256), 0, st,
        x, bstride, cstride, D, N, dict_t, G, Gp, cnorm, list, cnt, sel);
    GFS_LAUNCH_OK("rowsel_recheck_kernel<panel>");
    return GFS_OK;
}

}  // namespace gfs

extern "C" int64_t gfs_rowsel_tc_workspace_bytes(int64_t rows, int D) {
    if (rows <= 0 || D <= 0 || D % 64 != 0 || D > 192) return 0;
    return (int64_t)gfs::rt_plan(rows, D).total;
}

extern "C" int64_t gfs_rowsel_tc_workspace_bytes_kp(int64_t rows, int D, int Kp, int gw_project) {
    if (rows <= 0 || D <= 0 || D % 64 != 0 || D > 192 || Kp <= 0 || Kp > gfs::RT_MAXK) return 0;
    return (int64_t)gfs::rt_plan(rows, D, Kp, gw_project != 0).total;
}

extern "C" int gfs_gw_project_tc(const float* ec, int64_t ec_bstride, int B, int D, int N, const float* gp_l2t, int G, int Gp,
                                 void* cosine_act, int kblocks, int kb0, float* cosine_cm, int32_t* assignment, void* workspace,
                                 int64_t workspace_bytes, void* stream) {
    using namespace gfs;
    GFS_REQUIRE(ec && gp_l2t && assignment, GFS_ERR_BAD_ARG, "gfs_gw_project_tc: null pointer");
    GFS_REQUIRE(B > 0 && D > 0 && N > 0 && G > 0, GFS_ERR_BAD_ARG, "gfs_gw_project_tc: non-positive size");
    GFS_REQUIRE(D % 64 == 0 && D <= 192, GFS_ERR_UNSUPPORTED, "gfs_gw_project_tc: D=%d (need a multiple of 64, <= 192; use gfs_gw_project)", D);
    GFS_REQUIRE(N % 128 == 0, GFS_ERR_UNSUPPORTED, "gfs_gw_project_tc: N=%d (need a multiple of 128; use gfs_gw_project)", N);
    GFS_REQUIRE(G <= Gp && Gp <= RT_MAXK && Gp % 64 == 0, GFS_ERR_UNSUPPORTED, "gfs_gw_project_tc: G=%d Gp=%d (need G <= Gp <= 512, Gp %% 64 == 0)", G, Gp);
    GFS_REQUIRE((reinterpret_cast<uintptr_t>(cosine_act) & 15) == 0, GFS_ERR_BAD_ARG, "gfs_gw_project_tc: cosine_act must be 16-byte aligned");
    if (cosine_act) GFS_REQUIRE(kb0 >= 0 && kb0 + Gp / 64 <= kblocks, GFS_ERR_BAD_ARG, "gfs_gw_project_tc: output blocks out of range");
    if (Gp > RT_N)
        return rt_run_wide<RT_GW>("gfs_gw_project_tc", ec, ec_bstride, N, D, N, (int64_t)B * N, gp_l2t, G, Gp, nullptr, cosine_act, kblocks, kb0,
                                  cosine_cm, assignment, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
    return rt_run<RT_GW>("gfs_gw_project_tc", ec, ec_bstride, N, D, N, (int64_t)B * N, gp_l2t, G, Gp, nullptr, cosine_act, kblocks, kb0, cosine_cm,
                         assignment, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int gfs_kmeans_assign_tc(const float* X, int64_t n, int64_t ld, int point_major, int D, const float* centers_t, int K, int Kp,
                                    float* cnorm, int32_t* labels, void* workspace, int64_t workspace_bytes, void* stream) {
    using namespace gfs;
    GFS_REQUIRE(X && centers_t && cnorm && labels, GFS_ERR_BAD_ARG, "gfs_kmeans_assign_tc: null pointer");
    GFS_REQUIRE(n > 0 && D > 0 && K > 0, GFS_ERR_BAD_ARG, "gfs_kmeans_assign_tc: non-positive size");
    GFS_REQUIRE(point_major ? ld == D : ld >= n, GFS_ERR_BAD_ARG, "gfs_kmeans_assign_tc: leading dimension %lld does not fit the layout", (long long)ld);
    GFS_REQUIRE(n < (int64_t)1 << 31, GFS_ERR_UNSUPPORTED, "gfs_kmeans_assign_tc: n=%lld exceeds 2^31 per shard", (long long)n);
    GFS_REQUIRE(D % 64 == 0 && D <= 192, GFS_ERR_UNSUPPORTED, "gfs_kmeans_assign_tc: D=%d (need a multiple of 64, <= 192; use gfs_kmeans_assign)", D);
    GFS_REQUIRE(K <= Kp && Kp <= RT_MAXK, GFS_ERR_UNSUPPORTED, "gfs_kmeans_assign_tc: K=%d Kp=%d (need K <= Kp <= 512)", K, Kp);
    GFS_REQUIRE((reinterpret_cast<uintptr_t>(X) & 15) == 0, GFS_ERR_BAD_ARG, "gfs_kmeans_assign_tc: X must be 16-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    sqnorm_kernel<<<dim3((Kp + 255) / 256, 1), 256, 0, st>>>(centers_t, 0, D, Kp, cnorm);
    GFS_LAUNCH_OK("sqnorm_kernel");
    if (Kp > RT_N) {
        if (point_major)
            return rt_run_wide<RT_KMEANS_PM>("gfs_kmeans_assign_tc", X, 0, 1, D, 1, n, centers_t, K, Kp, cnorm, nullptr, 0, 0, nullptr, labels,
                                             workspace, workspace_bytes, st);
        return rt_run_wide<RT_KMEANS>("gfs_kmeans_assign_tc", X, 0, ld, D, 1, n, centers_t, K, Kp, cnorm, nullptr, 0, 0, nullptr, labels,
                                      workspace, workspace_bytes, st);
    }
    if (point_major)
        return rt_run<RT_KMEANS_PM>("gfs_kmeans_assign_tc", X, 0, 1, D, 1, n, centers_t, K, Kp, cnorm, nullptr, 0, 0, nullptr, labels, workspace,
                                    workspace_bytes, st);
    return rt_run<RT_KMEANS>("gfs_kmeans_assign_tc", X, 0, ld, D, 1, n, centers_t, K, Kp, cnorm, nullptr, 0, 0, nullptr, labels, workspace,
                             workspace_bytes, st);
}
