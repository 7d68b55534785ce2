// kmeans.cu -- deterministic M-step sums for the global k-means of get_basis.py:210 (sklearn _k_means_lloyd.pyx:209-218).
//
// Each persistent CTA owns a contiguous range of points, streams it through shared memory with TMA bulk copies and adds
// the points, in ascending point order, into a private (K x D) fp32 table in shared memory: thread d owns column d, so
// there are no floating-point atomics and no bank conflicts.  The
// per-CTA tables are then reduced in CTA order in fp64.  The result does not depend on scheduling, and across GPU
// counts it differs only by the (fp64) order of the partial sums.
#include "common.cuh"

namespace gfs {

constexpr int KM_CH = 32;          // points per TMA chunk
constexpr int KM_THREADS = 288;    // warps 0-7: one thread per feature column; warp 8: TMA issue, label staging, counts

// X is row-major, so a chunk of 32 points is ONE contiguous cp.async.bulk (TMA) of 32*D*4 bytes; two chunks are in flight
// while the column threads add the current one into the shared-memory table.
//
// WEIGHTED (sklearn _k_means_lloyd.pyx:216-218, sums[l] += x * w, wsum[l] += w): the helper warp stages the chunk's 32
// weights next to its labels, the column threads add __fmul_rn(x, w) with __fadd_rn (a product, then an add: no fused
// multiply-add, as sklearn's C), and the helper warp's lane 0 adds the weights into a per-CTA fp64 table in ascending
// point order instead of counting.  The unweighted instance is the kernel as it was.
//
// SPLIT (kmeans_partial_split_kernel, for K x D tables beyond shared memory): the CTAs form groups of `slices`; a group owns
// one contiguous point range, every CTA of it streams the whole range and keeps the table of its own contiguous slice of
// `kslice` centres, adding only the points labelled in that slice.  Each (centre, column) sum is then the same ascending-
// order fp32 sum the undivided table would hold.  The helper warp stages an out-of-slice label as -1.
template <bool WEIGHTED, bool SPLIT>
__device__ __forceinline__ void kmeans_partial_body(const float* __restrict__ X, int64_t n, int D, const int32_t* __restrict__ labels,
                                                    const float* __restrict__ weights, int K, int slices, int kslice,
                                                    float* __restrict__ partial, int32_t* __restrict__ pcount, double* __restrict__ pweight) {
    extern __shared__ __align__(128) unsigned char sm_raw[];
    const int range = SPLIT ? blockIdx.x / slices : blockIdx.x, nranges = SPLIT ? gridDim.x / slices : gridDim.x;
    const int c0 = SPLIT ? (blockIdx.x - range * slices) * kslice : 0;
    const int kc = SPLIT ? (K - c0 < kslice ? K - c0 : kslice) : K;     // centres of this CTA's table
    float* stg = reinterpret_cast<float*>(sm_raw);                          // [2][KM_CH][D]   (first: keeps 128 B alignment)
    float* tab = stg + 2 * KM_CH * D;                                       // [kc][D]
    int* cnt = reinterpret_cast<int*>(tab + (size_t)kc * D);                // [kc]           (unweighted)
    double* wtab = reinterpret_cast<double*>(tab + (size_t)kc * D);         // [kc] fp64      (weighted)
    int* lab = WEIGHTED ? reinterpret_cast<int*>(wtab + kc) : cnt + ((kc + 3) & ~3);   // [2][KM_CH]
    float* wst = reinterpret_cast<float*>(lab + 2 * KM_CH);                 // [2][KM_CH]     (weighted)
    uint64_t* full = reinterpret_cast<uint64_t*>(WEIGHTED ? reinterpret_cast<int*>(wst + 2 * KM_CH) : lab + 2 * KM_CH);  // [2]
    const int tid = threadIdx.x, lane = tid & 31;
    const bool helper = tid >= 256;

    for (int i = tid; i < kc * D; i += KM_THREADS) tab[i] = 0.0f;
    if constexpr (WEIGHTED) {
        for (int i = tid; i < kc; i += KM_THREADS) wtab[i] = 0.0;
    } else {
        for (int i = tid; i < kc; i += KM_THREADS) cnt[i] = 0;
    }
    if (tid == 0) {
        mbar_init(&full[0], 1);
        mbar_init(&full[1], 1);
        mbar_fence_init();
    }
    __syncthreads();

    int64_t per = (n + nranges - 1) / nranges;
    per = (per + KM_CH - 1) / KM_CH * KM_CH;
    const int64_t i0 = per * range;
    const int64_t i1 = (i0 + per) < n ? (i0 + per) : n;
    const int nchunks = i0 < i1 ? (int)((i1 - i0 + KM_CH - 1) / KM_CH) : 0;

    auto issue = [&](int c) {   // helper warp only
        if (c < nchunks) {
            const int64_t p0 = i0 + (int64_t)c * KM_CH;
            const int cc = (int)((i1 - p0) < KM_CH ? (i1 - p0) : KM_CH);
            if constexpr (SPLIT) {
                const int l = lane < cc ? labels[p0 + lane] - c0 : -1;
                lab[(c & 1) * KM_CH + lane] = l < kc ? l : -1;
            } else {
                lab[(c & 1) * KM_CH + lane] = lane < cc ? labels[p0 + lane] : 0;
            }
            if constexpr (WEIGHTED) wst[(c & 1) * KM_CH + lane] = lane < cc ? weights[p0 + lane] : 0.0f;
            if (lane == 0) {
                const uint32_t bytes = (uint32_t)cc * (uint32_t)D * 4u;
                mbar_arrive_expect_tx(&full[c & 1], bytes);
                tma_load_1d(stg + (size_t)(c & 1) * KM_CH * D, X + p0 * D, bytes, &full[c & 1]);
            }
        }
    };
    if (helper) {
        issue(0);
        issue(1);
    }
    __syncthreads();

    for (int c = 0; c < nchunks; ++c) {
        const int64_t p0 = i0 + (int64_t)c * KM_CH;
        const int cc = (int)((i1 - p0) < KM_CH ? (i1 - p0) : KM_CH);
        const int* L = lab + (c & 1) * KM_CH;
        mbar_wait(&full[c & 1], (c >> 1) & 1);
        if (!helper) {
            const int d = tid;
            if (d < D) {
                const float* S = stg + (size_t)(c & 1) * KM_CH * D + d;
                if constexpr (WEIGHTED) {
                    const float* W = wst + (c & 1) * KM_CH;
                    int j = 0;
                    for (; j + 1 < cc; j += 2) {  // the same pairwise order as the unweighted instance
                        const int l0 = L[j], l1 = L[j + 1];
                        const float v0 = __fmul_rn(S[j * D], W[j]), v1 = __fmul_rn(S[(j + 1) * D], W[j + 1]);
                        if (SPLIT && (l0 < 0 || l1 < 0)) {
                            if (l0 >= 0) tab[l0 * D + d] = __fadd_rn(tab[l0 * D + d], v0);
                            if (l1 >= 0) tab[l1 * D + d] = __fadd_rn(tab[l1 * D + d], v1);
                        } else if (l0 != l1) {
                            const float a = tab[l0 * D + d], b = tab[l1 * D + d];
                            tab[l0 * D + d] = __fadd_rn(a, v0);
                            tab[l1 * D + d] = __fadd_rn(b, v1);
                        } else {
                            tab[l0 * D + d] = __fadd_rn(__fadd_rn(tab[l0 * D + d], v0), v1);
                        }
                    }
                    if (j < cc && (!SPLIT || L[j] >= 0)) tab[L[j] * D + d] = __fadd_rn(tab[L[j] * D + d], __fmul_rn(S[j * D], W[j]));
                } else {
                    int j = 0;
                    for (; j + 1 < cc; j += 2) {      // ascending point order; two independent read-modify-writes when labels differ
                        const int l0 = L[j], l1 = L[j + 1];
                        const float v0 = S[j * D], v1 = S[(j + 1) * D];
                        if (SPLIT && (l0 < 0 || l1 < 0)) {
                            if (l0 >= 0) tab[l0 * D + d] += v0;
                            if (l1 >= 0) tab[l1 * D + d] += v1;
                        } else if (l0 != l1) {
                            const float a = tab[l0 * D + d], b = tab[l1 * D + d];
                            tab[l0 * D + d] = a + v0;
                            tab[l1 * D + d] = b + v1;
                        } else {
                            tab[l0 * D + d] = (tab[l0 * D + d] + v0) + v1;
                        }
                    }
                    if (j < cc && (!SPLIT || L[j] >= 0)) tab[L[j] * D + d] += S[j * D];
                }
            }
        } else if constexpr (WEIGHTED) {
            if (lane == 0) {                      // fp64, ascending point order: no floating-point atomics
                const float* W = wst + (c & 1) * KM_CH;
                for (int j = 0; j < cc; ++j)
                    if (!SPLIT || L[j] >= 0) wtab[L[j]] += (double)W[j];
            }
        } else if (lane < cc && (!SPLIT || L[lane] >= 0)) {
            atomicAdd(&cnt[L[lane]], 1);
        }
        __syncthreads();                          // chunk buffer and its labels are free again
        if (helper) issue(c + 2);
    }
    __syncthreads();
    float* o = partial + ((size_t)range * K + c0) * D;
    for (int i = tid; i < kc * D; i += KM_THREADS) o[i] = tab[i];
    if constexpr (WEIGHTED) {
        for (int i = tid; i < kc; i += KM_THREADS) pweight[(size_t)range * K + c0 + i] = wtab[i];
    } else {
        for (int i = tid; i < kc; i += KM_THREADS) pcount[(size_t)range * K + c0 + i] = cnt[i];
    }
}

template <bool WEIGHTED>
__global__ void __launch_bounds__(KM_THREADS, 1)
kmeans_partial_kernel(const float* __restrict__ X, int64_t n, int D, const int32_t* __restrict__ labels,
                      const float* __restrict__ weights, int K, float* __restrict__ partial, int32_t* __restrict__ pcount,
                      double* __restrict__ pweight) {
    kmeans_partial_body<WEIGHTED, false>(X, n, D, labels, weights, K, 1, K, partial, pcount, pweight);
}

template <bool WEIGHTED>
__global__ void __launch_bounds__(KM_THREADS, 1)
kmeans_partial_split_kernel(const float* __restrict__ X, int64_t n, int D, const int32_t* __restrict__ labels,
                            const float* __restrict__ weights, int K, int slices, int kslice, float* __restrict__ partial,
                            int32_t* __restrict__ pcount, double* __restrict__ pweight) {
    kmeans_partial_body<WEIGHTED, true>(X, n, D, labels, weights, K, slices, kslice, partial, pcount, pweight);
}

// shared memory of a table of kc centres, its counts or fp64 weight sums and the staging
static size_t km_smem(int kc, int D, bool weighted) {
    return weighted ? (size_t)(2 * KM_CH + kc) * D * sizeof(float) + (size_t)kc * sizeof(double) + 2 * KM_CH * (sizeof(int) + sizeof(float)) + 64
                    : (size_t)(2 * KM_CH + kc) * D * sizeof(float) + (size_t)((kc + 3) & ~3) * sizeof(int) + 2 * KM_CH * sizeof(int) + 64;
}
constexpr size_t KM_SMEM = 220 * 1024;

// centre slices per point range: 1 while the whole table fits (the single-table kernel), else the fewest that fit; the split
// is built for the k-means shapes beyond 192 centres, K <= 512 with D <= 192 (0: not built)
static int km_slices(int K, int D, bool weighted) {
    if (km_smem(K, D, weighted) <= KM_SMEM) return 1;
    if (K > 512 || D > 192) return 0;
    for (int g = 2; g <= K; ++g)
        if (km_smem((K + g - 1) / g, D, weighted) <= KM_SMEM) return g;
    return 0;
}

// CTA-order reduction of the per-CTA tables: sums in fp64; int32 counts into int64, or fp64 weight sums into fp64
template <typename PartialCount, typename Count>
__global__ void kmeans_reduce_kernel(const float* __restrict__ partial, const PartialCount* __restrict__ pcount, int P, int KD, int K,
                                     double* __restrict__ sums, Count* __restrict__ counts) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < KD) {
        double acc = 0.0;
        for (int p = 0; p < P; ++p) acc += (double)partial[(size_t)p * KD + i];
        sums[i] = acc;
    }
    if (i < K) {
        Count c = 0;
        for (int p = 0; p < P; ++p) c += pcount[(size_t)p * K + i];
        counts[i] = c;
    }
}

}  // namespace gfs

extern "C" int gfs_kmeans_partials(void) { return gfs::sm_count(); }

extern "C" int gfs_kmeans_accumulate_ranges(int K, int D, int weighted) {
    const int g = gfs::km_slices(K, D, weighted != 0);
    return g > 0 ? gfs::sm_count() / g : 0;
}

namespace gfs {
// One resident CTA per SM: the single-table kernel over sm_count() point ranges when the K x D table fits, else
// kmeans_partial_split_kernel with `slices` CTAs per range (sm_count() / slices ranges); then the range-order fp64 reduction.
template <bool WEIGHTED, typename PartialCount, typename Count>
static int km_accumulate(const char* who, const float* X, int64_t n, int D, const int32_t* labels, const float* weights, int K,
                         float* partial, int32_t* pcount, double* pweight, PartialCount* preduce, double* sums, Count* counts,
                         cudaStream_t st) {
    const int slices = km_slices(K, D, WEIGHTED);
    GFS_REQUIRE(slices > 0, GFS_ERR_UNSUPPORTED, "%s: K*D=%d does not fit shared memory", who, K * D);
    const int sms = sm_count();
    GFS_REQUIRE(sms > 0, GFS_ERR_CUDA, "%s: cannot query the device", who);
    const int P = sms / slices;
    GFS_REQUIRE(P > 0, GFS_ERR_UNSUPPORTED, "%s: K=%d needs %d CTAs per point range, the device has %d SMs", who, K, slices, sms);
    if (slices == 1) {
        GFS_CUDA_OK(allow_smem(reinterpret_cast<const void*>(kmeans_partial_kernel<WEIGHTED>), KM_SMEM));
        kmeans_partial_kernel<WEIGHTED><<<P, KM_THREADS, km_smem(K, D, WEIGHTED), st>>>(X, n, D, labels, weights, K, partial, pcount, pweight);
    } else {
        const int kslice = (K + slices - 1) / slices;
        GFS_CUDA_OK(allow_smem(reinterpret_cast<const void*>(kmeans_partial_split_kernel<WEIGHTED>), KM_SMEM));
        kmeans_partial_split_kernel<WEIGHTED><<<P * slices, KM_THREADS, km_smem(kslice, D, WEIGHTED), st>>>(
            X, n, D, labels, weights, K, slices, kslice, partial, pcount, pweight);
    }
    GFS_LAUNCH_OK("kmeans_partial_kernel");
    kmeans_reduce_kernel<PartialCount, Count><<<(K * D + 255) / 256, 256, 0, st>>>(partial, preduce, P, K * D, K, sums, counts);
    GFS_LAUNCH_OK("kmeans_reduce_kernel");
    return GFS_OK;
}
}  // namespace gfs

extern "C" int gfs_kmeans_accumulate(const float* X, int64_t n, int D, const int32_t* labels, int K, float* partial,
                                     int32_t* pcount, double* sums, int64_t* counts, void* stream) {
    using namespace gfs;
    GFS_REQUIRE(X && labels && partial && pcount && sums && counts, GFS_ERR_BAD_ARG, "gfs_kmeans_accumulate: null pointer");
    GFS_REQUIRE(n > 0 && D > 0 && K > 0, GFS_ERR_BAD_ARG, "gfs_kmeans_accumulate: non-positive size");
    GFS_REQUIRE(D <= 256 && D % 4 == 0, GFS_ERR_UNSUPPORTED, "gfs_kmeans_accumulate: D=%d must be a multiple of 4, <= 256", D);
    GFS_REQUIRE((reinterpret_cast<uintptr_t>(X) & 15) == 0, GFS_ERR_BAD_ARG, "gfs_kmeans_accumulate: X must be 16-byte aligned");
    return km_accumulate<false>("gfs_kmeans_accumulate", X, n, D, labels, nullptr, K, partial, pcount, nullptr, pcount, sums, counts,
                                static_cast<cudaStream_t>(stream));
}

extern "C" int gfs_kmeans_accumulate_weighted(const float* X, int64_t n, int D, const int32_t* labels, const float* weights, int K,
                                              float* partial, double* pweight, double* sums, double* wsums, void* stream) {
    using namespace gfs;
    GFS_REQUIRE(X && labels && weights && partial && pweight && sums && wsums, GFS_ERR_BAD_ARG,
                "gfs_kmeans_accumulate_weighted: null pointer");
    GFS_REQUIRE(n > 0 && D > 0 && K > 0, GFS_ERR_BAD_ARG, "gfs_kmeans_accumulate_weighted: non-positive size");
    GFS_REQUIRE(D <= 256 && D % 4 == 0, GFS_ERR_UNSUPPORTED, "gfs_kmeans_accumulate_weighted: D=%d must be a multiple of 4, <= 256", D);
    GFS_REQUIRE((reinterpret_cast<uintptr_t>(X) & 15) == 0, GFS_ERR_BAD_ARG, "gfs_kmeans_accumulate_weighted: X must be 16-byte aligned");
    return km_accumulate<true>("gfs_kmeans_accumulate_weighted", X, n, D, labels, weights, K, partial, nullptr, pweight, pweight, sums,
                               wsums, static_cast<cudaStream_t>(stream));
}

namespace gfs {

// ---------------------------------------------------------------------------------------------------------------
// The rest of a Lloyd iteration as two launches (it used to be ~25 elementwise / reduction launches of the host library:
// at the sharded size of BASELINE.json configs[3], 500 k points per GPU, those fixed costs were half of the iteration).
//
//   kmeans_pack_kernel    packed = [sums (K*D, written by the reduce kernel) | weight sums as fp64 (K) | #labels changed (1)]
//                         -- the ONE buffer the sharded version all-reduces (get_basis.py:210; SURVEY 8e).  The weight sums
//                         are the counts (copied here; exact integers, so the all-reduce keeps them exact) or, when counts
//                         is NULL, the fp64 sums the weighted reduce kernel already wrote into the slot.
//   kmeans_update_kernel  sklearn _k_means_common.pyx:_average_centers + the convergence quantities of _kmeans.py:_kmeans_single_lloyd:
//                         new = wsum > 0 ? sums / wsum : 0 (an empty cluster keeps the zero sum; the rare relocation is the
//                         caller's), shift = sum (new - old)^2 (fp64, fixed order), #empty; also the transposed (D, Kp) copy of
//                         the new centres that the next E-step reads.  result = [changed, shift, empty] (fp64) = one D2H read.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
kmeans_pack_kernel(const int32_t* __restrict__ labels, const int32_t* __restrict__ labels_old, int64_t n, const int64_t* __restrict__ counts,
                   int K, int KD, double* __restrict__ packed, unsigned long long* __restrict__ scratch) {
    // scratch[0]: mismatch counter, scratch[1]: ticket; both are left at zero for the next call
    unsigned long long mine = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        mine += labels[i] != labels_old[i];
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(&scratch[0], mine);          // integer sum: order does not matter
    __threadfence();
    __syncthreads();
    __shared__ bool last;
    if (threadIdx.x == 0) last = atomicAdd(&scratch[1], 1ull) == (unsigned long long)gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    if (counts)
        for (int c = threadIdx.x; c < K; c += blockDim.x) packed[KD + c] = (double)counts[c];
    if (threadIdx.x == 0) {
        packed[KD + K] = (double)atomicAdd(&scratch[0], 0ull);
        scratch[0] = 0ull;
        scratch[1] = 0ull;
    }
}

__global__ void __launch_bounds__(1024)
kmeans_update_kernel(const double* __restrict__ packed, const float* __restrict__ centers_old, int K, int D, int Kp,
                     float* __restrict__ centers_new, float* __restrict__ ct, double* __restrict__ result) {
    __shared__ double red[32];
    const int KD = K * D;
    double shift = 0.0;
    for (int i = threadIdx.x; i < KD; i += 1024) {
        const int c = i / D, d = i - c * D;
        const double wsum = packed[KD + c];
        const float nw = wsum > 0.0 ? (float)(packed[i] / wsum) : 0.0f;
        const double df = (double)(nw - centers_old[i]);
        shift += df * df;
        centers_new[i] = nw;
        ct[(int64_t)d * Kp + c] = nw;
    }
    double empty = 0.0;
    for (int c = threadIdx.x; c < K; c += 1024) empty += packed[KD + c] > 0.0 ? 0.0 : 1.0;
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
        shift += __shfl_xor_sync(0xffffffffu, shift, o);
        empty += __shfl_xor_sync(0xffffffffu, empty, o);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) red[warp] = shift;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 32; ++w) t += red[w];       // fixed order: deterministic
        result[1] = t;
        result[0] = packed[KD + K];
    }
    __syncthreads();
    if (lane == 0) red[warp] = empty;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 32; ++w) t += red[w];
        result[2] = t;
    }
}

}  // namespace gfs

extern "C" int gfs_kmeans_pack(const int32_t* labels, const int32_t* labels_old, int64_t n, const int64_t* counts, int K, int D,
                               double* packed, void* scratch16, void* stream) {
    using namespace gfs;
    GFS_REQUIRE(labels && labels_old && packed && scratch16, GFS_ERR_BAD_ARG, "gfs_kmeans_pack: null pointer");
    GFS_REQUIRE(n > 0 && K > 0 && D > 0, GFS_ERR_BAD_ARG, "gfs_kmeans_pack: non-positive size");
    const int64_t want = (n + 256 * 8 - 1) / (256 * 8);
    const unsigned grid = (unsigned)(want < 1 ? 1 : want > 592 ? 592 : want);
    kmeans_pack_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(labels, labels_old, n, counts, K, K * D, packed,
                                                                           static_cast<unsigned long long*>(scratch16));
    GFS_LAUNCH_OK("kmeans_pack_kernel");
    return GFS_OK;
}

extern "C" int gfs_kmeans_update(const double* packed, const float* centers_old, int K, int D, int Kp, float* centers_new, float* centers_t,
                                 double* result3, void* stream) {
    using namespace gfs;
    GFS_REQUIRE(packed && centers_old && centers_new && centers_t && result3, GFS_ERR_BAD_ARG, "gfs_kmeans_update: null pointer");
    GFS_REQUIRE(K > 0 && D > 0 && Kp >= K, GFS_ERR_BAD_ARG, "gfs_kmeans_update: bad size");
    kmeans_update_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(packed, centers_old, K, D, Kp, centers_new, centers_t, result3);
    GFS_LAUNCH_OK("kmeans_update_kernel");
    return GFS_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// k-means++ seeding step (sklearn _kmeans.py:_kmeans_plusplus, as get_basis.py:210 reaches it through KMeans(init=
// 'k-means++')): for T <= 8 candidate centres at once,
//     m[t][i] = min( max(float(|x_i|^2 - 2 x_i.c_t + |c_t|^2), 0), closest[i] ),      pot[t] = sum_i m[t][i]   (fp64)
// sklearn evaluates these distances on float64 upcasts of the float32 data and rounds the result to float32
// (metrics/pairwise.py:_euclidean_distances_upcast); the kernel does the same -- fp64 fma chains, one rounding to fp32 --
// so the values agree with sklearn's bit for bit except where an fp64 summation-order difference straddles an fp32
// rounding boundary (~1e-9 of the values).  One thread per point over the channel-major copy the E-step already keeps
// resident: every channel is ONE coalesced load feeding T DFMAs against the candidates in shared memory, a single pass
// over X (HBM bound: n*D*4 bytes; 8 DFMA per 4 bytes stay below the B200's fp64 rate).
// ---------------------------------------------------------------------------------------------------------------
namespace gfs {

constexpr int PP_T = 8;
constexpr int PP_THREADS = 256;

// WEIGHTED (sklearn's `distance_to_candidates @ sample_weight`): pots[t] += sum_i w_i * m[t][i] in fp64 -- the product of two
// fp32 values is exact in fp64, so with all weights 1 the sums are those of the unweighted instance.
template <bool WEIGHTED>
__global__ void __launch_bounds__(PP_THREADS)
kmeans_pp_trial_kernel(const float* __restrict__ xt, int64_t npad, int64_t n, int D, const double* __restrict__ xsq,
                       const float* __restrict__ cand, int T, const float* __restrict__ closest, const float* __restrict__ weights,
                       float* __restrict__ m_out, double* __restrict__ pots) {
    extern __shared__ __align__(16) double csd[];   // [D][8] candidate coordinates, then [8] squared norms
    double* csq = csd + D * PP_T;
    for (int i = threadIdx.x; i < D * PP_T; i += PP_THREADS) {
        const int c = i / PP_T, t = i - c * PP_T;
        csd[i] = t < T ? (double)cand[(int64_t)t * D + c] : 0.0;
    }
    __syncthreads();
    if (threadIdx.x < PP_T) {
        double s = 0.0;
        for (int c = 0; c < D; ++c) s = fma(csd[c * PP_T + threadIdx.x], csd[c * PP_T + threadIdx.x], s);
        csq[threadIdx.x] = s;
    }
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * PP_THREADS + threadIdx.x;
    const bool on = i < n;
    const int64_t ii = on ? i : 0;
    double dot[PP_T];
#pragma unroll
    for (int t = 0; t < PP_T; ++t) dot[t] = 0.0;
    const float* xp = xt + ii;
#pragma unroll 4
    for (int c = 0; c < D; ++c) {
        const double x = (double)__ldg(xp + (int64_t)c * npad);
        const double2 w0 = *reinterpret_cast<const double2*>(csd + c * PP_T), w1 = *reinterpret_cast<const double2*>(csd + c * PP_T + 2);
        const double2 w2 = *reinterpret_cast<const double2*>(csd + c * PP_T + 4), w3 = *reinterpret_cast<const double2*>(csd + c * PP_T + 6);
        dot[0] = fma(x, w0.x, dot[0]);
        dot[1] = fma(x, w0.y, dot[1]);
        dot[2] = fma(x, w1.x, dot[2]);
        dot[3] = fma(x, w1.y, dot[3]);
        dot[4] = fma(x, w2.x, dot[4]);
        dot[5] = fma(x, w2.y, dot[5]);
        dot[6] = fma(x, w3.x, dot[6]);
        dot[7] = fma(x, w3.y, dot[7]);
    }
    const double xs = xsq[ii];
    const float cl = closest ? closest[ii] : INFINITY;
    double wi = 1.0;
    if constexpr (WEIGHTED) wi = (double)weights[ii];
    __shared__ double red[PP_T][PP_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int t = 0; t < PP_T; ++t) {
        if (t < T) {                                  // warp-uniform
            const float d = fmaxf((float)((xs - 2.0 * dot[t]) + csq[t]), 0.0f);
            const float m = fminf(d, cl);
            if (on) m_out[(int64_t)t * npad + i] = m;
            double s;
            if constexpr (WEIGHTED) s = on ? (double)m * wi : 0.0;
            else s = on ? (double)m : 0.0;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) red[t][warp] = s;
        }
    }
    __syncthreads();
    if (threadIdx.x < T) {
        double s = 0.0;
        for (int w = 0; w < PP_THREADS / 32; ++w) s += red[threadIdx.x][w];
        atomicAdd(pots + threadIdx.x, s);
    }
}

}  // namespace gfs

extern "C" int gfs_kmeans_pp_trial(const float* xt, int64_t npad, int64_t n, int D, const double* xsq, const float* cand, int T,
                                   const float* closest, const float* weights, float* m_out, double* pots, void* stream) {
    using namespace gfs;
    GFS_REQUIRE(xt && xsq && cand && m_out && pots, GFS_ERR_BAD_ARG, "gfs_kmeans_pp_trial: null pointer");
    GFS_REQUIRE(n > 0 && npad >= n && D > 0 && T > 0, GFS_ERR_BAD_ARG, "gfs_kmeans_pp_trial: non-positive size");
    GFS_REQUIRE(T <= PP_T, GFS_ERR_UNSUPPORTED, "gfs_kmeans_pp_trial: T=%d candidates > %d is not built", T, PP_T);
    GFS_REQUIRE(D <= 512, GFS_ERR_UNSUPPORTED, "gfs_kmeans_pp_trial: D=%d > 512 is not built", D);
    const size_t smem = (size_t)(D * PP_T + PP_T) * sizeof(double);
    const int64_t grid = (n + PP_THREADS - 1) / PP_THREADS;
    GFS_REQUIRE(grid < ((int64_t)1 << 31), GFS_ERR_UNSUPPORTED, "gfs_kmeans_pp_trial: n too large");
    // unit weights run the instance without the weight load and product
    const auto kernel = weights ? kmeans_pp_trial_kernel<true> : kmeans_pp_trial_kernel<false>;
    kernel<<<(unsigned)grid, PP_THREADS, smem, static_cast<cudaStream_t>(stream)>>>(xt, npad, n, D, xsq, cand, T, closest, weights,
                                                                                    m_out, pots);
    GFS_LAUNCH_OK("kmeans_pp_trial_kernel");
    return GFS_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// inertia (sklearn _k_means_common.pyx:_inertia_dense):  sum_i w_i * |x_i - c_{label_i}|^2
// The per-point squared distance is sklearn's fp32 chain (_euclidean_dense_dense): result += ((d0^2 + d1^2) + d2^2) + d3^2 over
// groups of 4 features, every product and add rounded separately.  One warp per point: lane l loads feature groups l and l + 32
// (one coalesced row read), the chain then runs in group order through shuffles.  Each CTA owns a contiguous range of points,
// its warps take the points in a fixed interleave and add w_i * d_i (exact in fp64) in order; the per-CTA fp64 partials are
// reduced in CTA order, so the result depends on n alone, not on scheduling.
// ---------------------------------------------------------------------------------------------------------------
namespace gfs {

constexpr int KI_THREADS = 256;
constexpr int KI_MAX_CTAS = 1024;   // the partial workspace holds this many doubles
constexpr int KI_PTS = 4;           // points per warp step (independent loads in flight)

__device__ __forceinline__ float ki_group(const float4 a, const float4 b) {
    const float d0 = __fsub_rn(a.x, b.x), d1 = __fsub_rn(a.y, b.y), d2 = __fsub_rn(a.z, b.z), d3 = __fsub_rn(a.w, b.w);
    return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(d0, d0), __fmul_rn(d1, d1)), __fmul_rn(d2, d2)), __fmul_rn(d3, d3));
}

__global__ void __launch_bounds__(KI_THREADS)
kmeans_inertia_kernel(const float* __restrict__ X, int64_t n, int D, const int32_t* __restrict__ labels,
                      const float* __restrict__ centers, const float* __restrict__ weights, double* __restrict__ partial) {
    __shared__ double red[KI_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int G = D >> 2;                                     // feature groups of 4 (<= 64)
    const int64_t per = (n + gridDim.x - 1) / gridDim.x;
    const int64_t i0 = per * blockIdx.x;
    const int64_t i1 = (i0 + per) < n ? (i0 + per) : n;
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    double acc = 0.0;
    for (int64_t base = i0 + (int64_t)warp * KI_PTS; base < i1; base += (int64_t)KI_PTS * (KI_THREADS / 32)) {
        float t0[KI_PTS], t1[KI_PTS], w[KI_PTS];
#pragma unroll
        for (int q = 0; q < KI_PTS; ++q) {
            const int64_t i = base + q;
            const bool on = i < i1;
            const int64_t ii = on ? i : i0;
            const int l = labels[ii];
            w[q] = weights ? weights[ii] : 1.0f;
            const float4* xr = reinterpret_cast<const float4*>(X + ii * D);
            const float4* cr = reinterpret_cast<const float4*>(centers + (int64_t)l * D);
            t0[q] = lane < G ? ki_group(__ldg(xr + lane), __ldg(cr + lane)) : ki_group(zero4, zero4);
            t1[q] = lane + 32 < G ? ki_group(__ldg(xr + lane + 32), __ldg(cr + lane + 32)) : ki_group(zero4, zero4);
        }
        float r[KI_PTS];
#pragma unroll
        for (int q = 0; q < KI_PTS; ++q) r[q] = 0.0f;
        for (int g = 0; g < G; ++g) {                        // warp-uniform: sklearn's group order
#pragma unroll
            for (int q = 0; q < KI_PTS; ++q) r[q] = __fadd_rn(r[q], __shfl_sync(0xffffffffu, g < 32 ? t0[q] : t1[q], g & 31));
        }
#pragma unroll
        for (int q = 0; q < KI_PTS; ++q)
            if (base + q < i1) acc += (double)r[q] * (double)w[q];
    }
    if (lane == 0) red[warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int k = 0; k < KI_THREADS / 32; ++k) s += red[k];
        partial[blockIdx.x] = s;
    }
}

__global__ void kmeans_inertia_reduce_kernel(const double* __restrict__ partial, int P, double* __restrict__ out) {
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int p = 0; p < P; ++p) s += partial[p];
        out[0] = s;
    }
}

}  // namespace gfs

extern "C" int gfs_kmeans_inertia_partials(void) { return gfs::KI_MAX_CTAS; }

extern "C" int gfs_kmeans_inertia(const float* X, int64_t n, int D, const int32_t* labels, const float* centers, int K,
                                  const float* weights, double* partial, double* out, void* stream) {
    using namespace gfs;
    GFS_REQUIRE(X && labels && centers && partial && out, GFS_ERR_BAD_ARG, "gfs_kmeans_inertia: null pointer");
    GFS_REQUIRE(n > 0 && D > 0 && K > 0, GFS_ERR_BAD_ARG, "gfs_kmeans_inertia: non-positive size");
    GFS_REQUIRE(D <= 256 && D % 4 == 0, GFS_ERR_UNSUPPORTED, "gfs_kmeans_inertia: D=%d must be a multiple of 4, <= 256", D);
    GFS_REQUIRE((reinterpret_cast<uintptr_t>(X) & 15) == 0 && (reinterpret_cast<uintptr_t>(centers) & 15) == 0, GFS_ERR_BAD_ARG,
                "gfs_kmeans_inertia: X and centers must be 16-byte aligned");
    const int64_t want = (n + 63) / 64;
    const int P = (int)(want < KI_MAX_CTAS ? want : KI_MAX_CTAS);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    kmeans_inertia_kernel<<<P, KI_THREADS, 0, st>>>(X, n, D, labels, centers, weights, partial);
    GFS_LAUNCH_OK("kmeans_inertia_kernel");
    kmeans_inertia_reduce_kernel<<<1, 32, 0, st>>>(partial, P, out);
    GFS_LAUNCH_OK("kmeans_inertia_reduce_kernel");
    return GFS_OK;
}
