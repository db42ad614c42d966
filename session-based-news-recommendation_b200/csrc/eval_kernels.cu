// Full-catalog top-20 evaluation without materialising the [B,N] score matrix.
// Reference: model_combine.py:283-306 (scores -> argsort()[::-1][:20]) and util.py:8-18 (rank = #(S > S[label]) + 1).
//
// The scoring kernel (eval mode) leaves chunkmax[b, j] = max of the bf16-GEMM scores of items 8j..8j+7.  Every item
// of the true top-20 lives in one of the 20 chunks with the largest chunk maxima, so we take the 32 best chunks
// (12 chunks of slack for bf16 rounding), re-score their 256 items exactly in fp32 and sort those by
// (score desc, id asc).  Ties therefore resolve to the lower item id (north_star), which agrees with the
// reference on tie-free inputs.
//
// The slack is then CERTIFIED per query: with eps_b a rigorous bound on |bf16-GEMM score - exact fp32 score| (from the
// query's own rounding error and the catalog's largest row norm / rounding-error norm, tcar_catalog_stats), an item
// outside the re-scored chunks can only belong to the top-20 if its chunk maximum reaches s20 - eps_b (s20 = the 20th
// exact score found).  Queries whose best unselected chunk stays below that bound are done; the others are flagged and
// tcar_eval_topk_widen re-scores EVERY chunk at or above the bound (streaming, any number of them), so the result is
// the exact top-20 either way.
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <math.h>
#include <stdint.h>
#include "tcar_b200.h"
#include "launch.cuh"

namespace tcar {

constexpr int H = TCAR_H, HP = TCAR_HP, XW = TCAR_XW, NB = TCAR_NBINS, TOPK = TCAR_TOPK;
constexpr int NCH = TCAR_NCAND_CHUNKS, CH = TCAR_CHUNK, NCAND = NCH * CH;  // 32 chunks x 8 = 256 candidates
__device__ __constant__ int kBinOffE[6] = {0, 13, 45, 53, 78, 139};

__device__ __forceinline__ float warp_sum_e(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// order-preserving map float -> uint32 (larger float <=> larger key); -inf is the smallest finite-comparable key
__device__ __forceinline__ uint32_t fkey(float f) {
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// same arithmetic as exact_score() in session_kernels.cu (kept identical so label and candidates compare exactly)
__device__ __forceinline__ float exact_score_e(const float* s_aic, const float* s_tq, const float* __restrict__ item,
                                               const float* __restrict__ content,
                                               const int32_t* __restrict__ mwdhm, int n, int lane) {
    const float4* ir = reinterpret_cast<const float4*>(item + ((size_t)n + 1) * HP);
    const float4* cr = reinterpret_cast<const float4*>(content + ((size_t)n + 1) * HP);
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const int c = j * 128 + lane * 4;
        const float4 iv = __ldg(ir + j * 32 + lane), cv = __ldg(cr + j * 32 + lane);
        if (c + 0 < H) { acc = fmaf(iv.x, s_aic[c + 0], acc); acc = fmaf(cv.x, s_aic[H + c + 0], acc); }
        if (c + 1 < H) { acc = fmaf(iv.y, s_aic[c + 1], acc); acc = fmaf(cv.y, s_aic[H + c + 1], acc); }
        if (c + 2 < H) { acc = fmaf(iv.z, s_aic[c + 2], acc); acc = fmaf(cv.z, s_aic[H + c + 2], acc); }
        if (c + 3 < H) { acc = fmaf(iv.w, s_aic[c + 3], acc); acc = fmaf(cv.w, s_aic[H + c + 3], acc); }
    }
    acc = warp_sum_e(acc);
    float tsum = 0.f;
#pragma unroll
    for (int k = 0; k < 5; ++k) tsum += s_tq[kBinOffE[k] + mwdhm[(size_t)n * 5 + k]];
    return acc + tsum;
}

// (score desc, id asc) "a ranks before b"
__device__ __forceinline__ bool before(float sa, int ia, float sb, int ib) {
    return sa > sb || (sa == sb && ia < ib);
}

// Block-wide selection of the NCH largest of vals[0..n) (n > NCH) by (value desc, index asc): 4 x 8-bit radix passes
// on the order-preserving key find the NCH-th largest key, then strictly-greater entries are taken in any order and
// equal-key entries lowest index first.  256 threads; s_sel receives NCH indices.
__device__ __forceinline__ void select_top(const float* __restrict__ vals, int n, int* s_sel, int* s_hist, int* s_warp,
                                           int* s_misc /* [4]: cnt, need, digit, above */) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    uint32_t prefix = 0, mask = 0;
    int kth = NCH;
    if (tid == 0) s_misc[0] = 0;
    for (int shift = 24; shift >= 0; shift -= 8) {
        s_hist[tid] = 0;
        __syncthreads();
        for (int i = tid; i < n; i += 256) {
            const uint32_t k = fkey(vals[i]);
            if ((k & mask) == prefix) atomicAdd(&s_hist[(k >> shift) & 255u], 1);
        }
        __syncthreads();
        if (tid == 0) {
            int above = 0, d = 255;
            for (; d > 0; --d) {
                if (above + s_hist[d] >= kth) break;
                above += s_hist[d];
            }
            s_misc[2] = d;
            s_misc[3] = above;
        }
        __syncthreads();
        prefix |= (uint32_t)s_misc[2] << shift;
        mask |= 255u << shift;
        kth -= s_misc[3];
        __syncthreads();
    }
    // prefix = key of the NCH-th largest; kth = how many keys equal to it are still needed
    for (int i = tid; i < n; i += 256)
        if (fkey(vals[i]) > prefix) s_sel[atomicAdd(&s_misc[0], 1)] = i;
    __syncthreads();
    int base = s_misc[0];
    __syncthreads();
    for (int i0 = 0; i0 < n && base < NCH; i0 += 256) {
        const int i = i0 + tid;
        const bool eq = i < n && fkey(vals[i]) == prefix;
        const uint32_t bal = __ballot_sync(0xffffffffu, eq);
        if (lane == 0) s_warp[w] = __popc(bal);
        __syncthreads();
        int off = base;
        for (int j = 0; j < w; ++j) off += s_warp[j];
        int tot = 0;
        for (int j = 0; j < 8; ++j) tot += s_warp[j];
        const int pos = off + __popc(bal & ((1u << lane) - 1u));
        if (eq && pos < NCH) s_sel[pos] = i;
        base += tot;
        __syncthreads();
    }
    __syncthreads();
}

__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16(x)); }

// eps_b >= |S_gemm[b,n] - S_exact[b,n]| for every item n of the catalog the statistics were taken over:
//   S_gemm = bf(q) . bf(i) + sum_k bf(Tq[k, idx_k])   (exact products, fp32 accumulation on the tensor cores)
//   S_exact = q . i + sum_k Tq[k, idx_k]              (fp32 FMA chain, exact_score_e)
//   q . i - bf(q) . bf(i) = dq . i + bf(q) . di  ->  <= ||dq|| max||i|| + ||bf(q)|| max||di||   (Cauchy-Schwarz)
// plus the rounding of the five time terms and 2e-4 of the magnitudes for the two fp32 accumulations.
// Block-wide (256 threads); `red` = 32 floats of scratch.  One pass over the session vector, one over the 139 bins.
__device__ __forceinline__ float score_error_bound(const float* s_aic, const float* s_tq, const float* cat_stats,
                                                   float* red) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    float dq2 = 0.f, q2 = 0.f, f2 = 0.f;
    for (int c = tid; c < XW; c += 256) {
        const float v = s_aic[c], r = bf16_round(v);
        dq2 = fmaf(v - r, v - r, dq2);
        q2 = fmaf(r, r, q2);
        f2 = fmaf(v, v, f2);
    }
    dq2 = warp_sum_e(dq2);
    q2 = warp_sum_e(q2);
    f2 = warp_sum_e(f2);
    // time bins: thread r < 139 owns one bin; per-table maxima of |rounding error| and |value| by warp 0 afterwards
    __syncthreads();
    if (lane == 0) { red[w] = dq2; red[8 + w] = q2; red[16 + w] = f2; }
    __shared__ float s_te[NB + 1], s_tm[NB + 1];
    if (tid < NB) {
        const float v = s_tq[tid];
        s_te[tid] = fabsf(v - bf16_round(v));
        s_tm[tid] = fabsf(v);
    }
    __syncthreads();
    dq2 = q2 = f2 = 0.f;
    for (int i = 0; i < 8; ++i) { dq2 += red[i]; q2 += red[8 + i]; f2 += red[16 + i]; }
    float terr = 0.f, tmag = 0.f;
    if (w == 0) {
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            float e = 0.f, m = 0.f;
            for (int r = kBinOffE[k] + lane; r < kBinOffE[k + 1]; r += 32) { e = fmaxf(e, s_te[r]); m = fmaxf(m, s_tm[r]); }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                e = fmaxf(e, __shfl_xor_sync(0xffffffffu, e, o));
                m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
            }
            terr += e;
            tmag += m;
        }
    }
    const float imax = cat_stats[0], dimax = cat_stats[1];
    const float eps = sqrtf(dq2) * imax + sqrtf(q2) * dimax + terr + 2e-4f * (sqrtf(f2) * imax + tmag);
    return eps * 1.0001f + 1e-30f;          // valid in warp 0 (thread 0 consumes it)
}

constexpr int TILE_CH = 128 / CH;          // 16 chunks per 128-item tile
constexpr int NCC = NCH * TILE_CH;         // 512 candidate chunks after the tile-level selection

constexpr int NSEL = TCAR_EVAL_NSEL;       // 33 entries per (query, shard) list: 32 candidate chunks + 1 bound carrier

// The two halves of the kernel can run on different GPUs (catalog-sharded evaluation, Seq2SeqAttNN.eval_round):
//   select-only  (out_vals != NULL): the item range's 32 best chunks of every query as (bf16-GEMM chunk maximum, GLOBAL
//                chunk id) + a 33rd entry whose value bounds every chunk NOT listed (33rd chunk of the selected tiles /
//                best unselected tile) -- no re-scoring;
//   re-score     (in_vals != NULL): `in_lists` such lists per query (one per item range, `in_stride` words apart) are
//                merged: the 32 best entries overall are re-scored exactly from the (replicated) fp32 tables; the 33rd
//                best value bounds everything that is not (a range's 33rd entry can never be among the 32 best overall:
//                its own 32 predecessors would all be, too).
struct SelIO {
    float* out_vals;
    int32_t* out_ids;
    int chunk_base;
    const float* in_vals;
    const int32_t* in_ids;
    int in_lists;
    long long in_stride;
    // select-only over several session groups in one launch (blockIdx.y = group): group g has gn[g] queries, its chunk /
    // tile maxima lie cm_gs / tm_gs floats apart and its output lists out_gs words apart
    int groups;
    int gn[TCAR_MAX_PEERS];
    long long cm_gs, tm_gs, out_gs;
};

// bitonic sort of the NCC (value, chunk id) candidates by (value desc, id asc); ends with a barrier
__device__ __forceinline__ void sort_chunk_candidates(float* s_cv, int* s_ci) {
    const int tid = threadIdx.x;
    for (int k = 2; k <= NCC; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            __syncthreads();
            for (int i = tid; i < NCC; i += 256) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const float sa = s_cv[i], sb = s_cv[ixj];
                    const int ia = s_ci[i], ib = s_ci[ixj];
                    const bool up = (i & k) == 0;
                    const bool swap = up ? before(sb, ib, sa, ia) : before(sa, ia, sb, ib);
                    if (swap) { s_cv[i] = sb; s_cv[ixj] = sa; s_ci[i] = ib; s_ci[ixj] = ia; }
                }
            }
        }
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------ warp-per-query selection
// The selection half (32 best chunks of a query by bf16 chunk maximum + a bound on the rest) needs no block-wide
// cooperation: a CTA of 256 threads spends it in ~75 barriers.  Here ONE WARP owns a query: a 4-pass radix select over
// the tile maxima (warp-private 256-bin histogram in shared memory, bins scanned with shuffles) finds the 32 best tiles,
// lane l then holds tile l's 16 chunk maxima in registers, chunks below the 32nd tile maximum are pruned (they cannot
// be among the 32 best chunks), and the 32 best survivors are extracted with 32 warp arg-max steps.  8 queries per CTA,
// >= 32 queries in flight per SM instead of 3-4.
struct SelGroups {
    int groups;                          // 0: one group of B queries
    int n[TCAR_MAX_PEERS];
    long long cm_gs, tm_gs, out_gs;
};

__global__ void __launch_bounds__(256)
eval_select_warp_kernel(const float* chunkmax, const float* tilemax, float* sel_vals, int32_t* sel_ids, int B, int N,
                        int n_pad, int chunk_base, const __grid_constant__ SelGroups sg) {
    PDL_ENTER();
    __shared__ int s_hist[8][256];
    __shared__ int s_tile[8][NCH];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int b = blockIdx.x * 8 + w;
    if (sg.groups > 0) {
        const int g = blockIdx.y;
        B = sg.n[g];
        chunkmax += (size_t)g * sg.cm_gs;
        tilemax += (size_t)g * sg.tm_gs;
        sel_vals += (size_t)g * sg.out_gs;
        sel_ids += (size_t)g * sg.out_gs;
    }
    if (b >= B) return;                  // warp-uniform; no block-wide barrier below
    const int nchunks = (N + CH - 1) / CH;
    const int ntiles = (N + 127) / 128;
    const float* cm = chunkmax + (size_t)b * (n_pad / CH);
    const float* tm = tilemax + (size_t)b * (n_pad / 128);
    int* hist = s_hist[w];
    int* tiles = s_tile[w];
    float thr = -INFINITY;               // 32nd largest tile maximum: chunks below it are not candidates
    float rest_tile_max = -INFINITY;     // best tile NOT taken
    int ntake = ntiles < NCH ? ntiles : NCH;
    if (ntiles <= NCH) {
        if (lane < ntiles) tiles[lane] = lane;
    } else {
        uint32_t prefix = 0, mask = 0;
        int kth = NCH;
        for (int shift = 24; shift >= 0; shift -= 8) {
#pragma unroll
            for (int j = 0; j < 8; ++j) hist[lane * 8 + j] = 0;
            __syncwarp();
            for (int base = 0; base < ntiles; base += 32 * 8) {      // warp-uniform trip count (match_any below)
                const int i0 = base + lane;
                // eight independent loads in flight per lane (one warp per query: nothing else hides the latency)
                float t[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) t[u] = i0 + 32 * u < ntiles ? tm[i0 + 32 * u] : 0.f;
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    // scores of one query sit in a narrow range: most lanes hit the SAME bin, and a shared-memory
                    // atomic would serialise them (47 us per launch).  Lanes with equal bins are matched instead and
                    // one of them adds their count: the leaders of one step have distinct bins.
                    const uint32_t k = fkey(t[u]);
                    const bool act = i0 + 32 * u < ntiles && (k & mask) == prefix;
                    const uint32_t bin = act ? ((k >> shift) & 255u) : 256u;
                    const uint32_t peers = __match_any_sync(0xffffffffu, bin);
                    if (act && lane == __ffs(peers) - 1) hist[bin] += __popc(peers);
                    __syncwarp();
                }
            }
            __syncwarp();
            int cnt[8], tot = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) { cnt[j] = hist[lane * 8 + j]; tot += cnt[j]; }
            int suf = tot;               // inclusive suffix sum over the lanes (bins of higher lanes are larger digits)
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_down_sync(0xffffffffu, suf, o);
                if (lane + o < 32) suf += v;
            }
            const int above_lane = suf - tot;
            const bool mine = above_lane < kth && kth <= suf;
            int d = 0, above = 0;
            if (mine) {
                int a = above_lane;
                for (int j = 7; j >= 0; --j) {
                    if (a + cnt[j] >= kth) { d = lane * 8 + j; above = a; break; }
                    a += cnt[j];
                }
            }
            const uint32_t who = __ballot_sync(0xffffffffu, mine);
            const int src = __ffs(who) - 1;
            d = __shfl_sync(0xffffffffu, d, src);
            above = __shfl_sync(0xffffffffu, above, src);
            prefix |= (uint32_t)d << shift;
            mask |= 255u << shift;
            kth -= above;
            __syncwarp();
        }
        // prefix = key of the 32nd largest tile maximum; kth = how many tiles equal to it are still needed
        int taken = 0, eq_left = kth;
        float below = -INFINITY;
        bool eq_rest = false;
        for (int i00 = 0; i00 < ntiles; i00 += 32 * 4) {
          float t4[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) t4[u] = i00 + 32 * u + lane < ntiles ? tm[i00 + 32 * u + lane] : -INFINITY;
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int i = i00 + 32 * u + lane;
            if (i00 + 32 * u >= ntiles) break;                      // warp-uniform
            const float v = t4[u];
            const uint32_t k = i < ntiles ? fkey(v) : 0u;
            const bool gt = i < ntiles && k > prefix, eq = i < ntiles && k == prefix;
            const uint32_t bg = __ballot_sync(0xffffffffu, gt), be = __ballot_sync(0xffffffffu, eq);
            if (gt) tiles[taken + __popc(bg & ((1u << lane) - 1u))] = i;
            taken += __popc(bg);
            const int rank_eq = __popc(be & ((1u << lane) - 1u));
            if (eq && rank_eq < eq_left) tiles[taken + rank_eq] = i;
            const int take_eq = min(__popc(be), eq_left);
            if (__popc(be) > eq_left) eq_rest = true;
            taken += take_eq;
            eq_left -= take_eq;
            if (i < ntiles && k < prefix) below = fmaxf(below, v);
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) below = fmaxf(below, __shfl_xor_sync(0xffffffffu, below, o));
        // value of the prefix key (the 32nd largest tile maximum)
        const uint32_t pu = (prefix & 0x80000000u) ? (prefix & 0x7fffffffu) : ~prefix;
        thr = __uint_as_float(pu);
        rest_tile_max = eq_rest ? thr : below;
        __syncwarp();
    }
    // ---- lane l <- tile l: its 16 chunk maxima, pruned by thr
    float v[TILE_CH];
    uint32_t alive = 0;
    float pruned = -INFINITY;
    const int tile = lane < ntake ? tiles[lane] : -1;
    if (tile >= 0) {
        const float4* src = reinterpret_cast<const float4*>(cm + (size_t)tile * TILE_CH);
#pragma unroll
        for (int c = 0; c < TILE_CH / 4; ++c) {
            const float4 q = src[c];
            v[4 * c] = q.x; v[4 * c + 1] = q.y; v[4 * c + 2] = q.z; v[4 * c + 3] = q.w;
        }
#pragma unroll
        for (int c = 0; c < TILE_CH; ++c) {
            const bool ok = tile * TILE_CH + c < nchunks;
            if (ok && v[c] >= thr) alive |= 1u << c;
            else if (ok) pruned = fmaxf(pruned, v[c]);
        }
    }
    // ---- 32 arg-max extractions by (value desc, chunk id asc)
    float* out_v = sel_vals + (size_t)b * NSEL;
    int32_t* out_i = sel_ids + (size_t)b * NSEL;
    float my_v = -INFINITY;
    int my_c = 0x7fffffff;
    auto refresh = [&]() {
        my_v = -INFINITY;
        my_c = 0x7fffffff;
#pragma unroll
        for (int c = 0; c < TILE_CH; ++c)
            if (((alive >> c) & 1u) && before(v[c], tile * TILE_CH + c, my_v, my_c)) { my_v = v[c]; my_c = tile * TILE_CH + c; }
    };
    refresh();
    for (int r = 0; r < NCH; ++r) {
        float bv = my_v;
        int bc = my_c;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oc = __shfl_xor_sync(0xffffffffu, bc, o);
            if (before(ov, oc, bv, bc)) { bv = ov; bc = oc; }
        }
        if (lane == 0) {
            out_v[r] = bc == 0x7fffffff ? -INFINITY : bv;
            out_i[r] = bc == 0x7fffffff ? -1 : bc + chunk_base;
        }
        if (bc != 0x7fffffff && bc == my_c) {           // the winner retires its entry
            alive &= ~(1u << (bc - tile * TILE_CH));
            refresh();
        }
    }
    // ---- bound on every chunk that is not listed: best survivor left, best pruned chunk, best tile not taken
    float rest = fmaxf(my_v, pruned);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rest = fmaxf(rest, __shfl_xor_sync(0xffffffffu, rest, o));
    rest = fmaxf(rest, rest_tile_max);
    if (lane == 0) {
        out_v[NCH] = rest;
        out_i[NCH] = -2;
    }
}

// one CTA (256 threads) per query.  Two-level selection: the 32 best 128-item tiles by tile max (every one of the 32
// best chunks lives in one of them: the 32 largest tile maxima are 32 distinct chunk values, so the 32nd largest chunk
// is >= the 32nd largest tile max), then the 32 best of their 512 chunks, then the exact fp32 re-scoring.
__global__ void __launch_bounds__(256)
eval_topk_kernel(const float* chunkmax, const float* tilemax, const float* __restrict__ a_ic,
                 const float* __restrict__ Tq, const float* __restrict__ item, const float* __restrict__ content,
                 const int32_t* __restrict__ mwdhm, const int32_t* __restrict__ label, int32_t* __restrict__ top_ids,
                 float* __restrict__ top_scores, int32_t* __restrict__ n_greater, int N, int n_pad, int item_offset,
                 const float* __restrict__ cat_stats, int32_t* __restrict__ uncertain, float* __restrict__ tau,
                 const __grid_constant__ SelIO io) {
    PDL_ENTER();
    __shared__ float s_aic[XW], s_tq[NB + 1];
    __shared__ float s_red[32];
    __shared__ uint32_t s_tilebits[(TCAR_MAX_EVAL_TILES + 31) / 32];
    float unsel_max = -INFINITY;         // largest bf16 score an item outside the re-scored chunks can have
    __shared__ int s_hist[256];
    __shared__ int s_sel[NCH];
    __shared__ int s_misc[4];
    __shared__ float s_cv[NCC];
    __shared__ int s_ci[NCC];
    __shared__ float s_sc[NCAND];
    __shared__ int s_id[NCAND];
    __shared__ int s_warp[8];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int nchunks = (N + CH - 1) / CH;
    const int ntiles = (N + 127) / 128;
    const bool sel_only = io.out_vals != nullptr, from_lists = io.in_vals != nullptr;
    float* sel_vals = io.out_vals;
    int32_t* sel_ids = io.out_ids;
    if (io.groups > 0) {
        const int g = blockIdx.y;
        if (b >= io.gn[g]) return;
        chunkmax += (size_t)g * io.cm_gs;
        tilemax += (size_t)g * io.tm_gs;
        sel_vals += (size_t)g * io.out_gs;
        sel_ids += (size_t)g * io.out_gs;
    }
    const float* cm = chunkmax + (size_t)b * (n_pad / CH);
    const float* tm = tilemax + (size_t)b * (n_pad / 128);
    if (!sel_only) {
        for (int c = tid; c < XW; c += 256) s_aic[c] = a_ic[(size_t)b * XW + c];
        for (int c = tid; c < NB; c += 256) s_tq[c] = Tq[(size_t)b * NB + c];
    }
    for (int i = tid; i < NCH; i += 256) s_sel[i] = -1;
    __syncthreads();

    if (from_lists && io.in_lists == 1) {
        // ---- one list (single GPU): its 32 entries are the candidates, the 33rd is the bound
        const size_t at = (size_t)b * NSEL + tid;
        if (tid < NCH) {
            const int cid = io.in_ids[at];
            s_sel[tid] = cid >= 0 ? cid : -1;
        }
        unsel_max = io.in_vals[(size_t)b * NSEL + NCH];
    } else if (from_lists) {
        // ---- the item ranges' candidate lists (global chunk ids): the 32 best overall, the 33rd as the bound
        const int n_in = io.in_lists * NSEL;
        for (int i = tid; i < NCC; i += 256) {
            float v = -INFINITY;
            int id = 0x7fffffff;
            if (i < n_in) {
                const size_t at = (size_t)(i / NSEL) * io.in_stride + (size_t)b * NSEL + (i % NSEL);
                const int cid = io.in_ids[at];
                if (cid >= 0) { v = io.in_vals[at]; id = cid; }
                else if (cid == -2) { v = io.in_vals[at]; }       // bound carrier without a chunk
            }
            s_cv[i] = v;
            s_ci[i] = id;
        }
        sort_chunk_candidates(s_cv, s_ci);
        unsel_max = s_cv[NCH];
        if (tid < NCH) s_sel[tid] = s_ci[tid] == 0x7fffffff ? -1 : s_ci[tid];
    } else if (nchunks > NCH) {
        // ---- level 1: tiles
        if (ntiles <= NCH) {
            for (int i = tid; i < ntiles; i += 256) s_sel[i] = i;
            __syncthreads();
        } else {
            select_top(tm, ntiles, s_sel, s_hist, s_warp, s_misc);
            if (cat_stats || sel_only) {
                // best tile NOT selected: bitmap of the selected ones, then a max over the rest
                for (int i = tid; i < (ntiles + 31) / 32; i += 256) s_tilebits[i] = 0u;
                __syncthreads();
                if (tid < NCH && s_sel[tid] >= 0) atomicOr(&s_tilebits[s_sel[tid] >> 5], 1u << (s_sel[tid] & 31));
                __syncthreads();
                float m = -INFINITY;
                for (int i = tid; i < ntiles; i += 256)
                    if (!((s_tilebits[i >> 5] >> (i & 31)) & 1u)) m = fmaxf(m, tm[i]);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
                if (lane == 0) s_red[w] = m;
                __syncthreads();
                for (int i = 0; i < 8; ++i) unsel_max = fmaxf(unsel_max, s_red[i]);
                __syncthreads();
            }
        }
        // ---- level 2: the 16 chunks of every selected tile, sorted by (max desc, chunk index asc)
        for (int i = tid; i < NCC; i += 256) {
            const int tile = s_sel[i / TILE_CH];
            const int chunk = tile * TILE_CH + (i % TILE_CH);
            const bool ok = tile >= 0 && chunk < nchunks;
            s_cv[i] = ok ? cm[chunk] : -INFINITY;
            s_ci[i] = ok ? chunk : 0x7fffffff;
        }
        sort_chunk_candidates(s_cv, s_ci);
        unsel_max = fmaxf(unsel_max, s_cv[NCH]);        // best chunk of the selected tiles that is NOT re-scored
        if (tid < NCH) s_sel[tid] = s_ci[tid] == 0x7fffffff ? -1 : s_ci[tid];
    } else {
        for (int i = tid; i < NCC; i += 256) {           // tiny item range: every chunk is a candidate
            s_cv[i] = i < nchunks ? cm[i] : -INFINITY;
            s_ci[i] = i < nchunks ? i : 0x7fffffff;
        }
        for (int i = tid; i < nchunks; i += 256) s_sel[i] = i;
    }
    __syncthreads();
    if (sel_only) {
        // 32 candidates (value, GLOBAL chunk id; -1 = none) + the bound on everything not listed (id -2)
        if (tid < NSEL) {
            const size_t at = (size_t)b * NSEL + tid;
            if (tid < NCH) {
                const bool ok = s_ci[tid] != 0x7fffffff;
                sel_vals[at] = ok ? s_cv[tid] : -INFINITY;
                sel_ids[at] = ok ? s_ci[tid] + io.chunk_base : -1;
            } else {
                sel_vals[at] = nchunks > NCH ? unsel_max : -INFINITY;
                sel_ids[at] = -2;
            }
        }
        return;
    }

    // exact re-scoring: warp w handles candidates w*32 .. w*32+31
    const int lab = label[b];
    float lab_score = 0.f;
    {
        const float ls = exact_score_e(s_aic, s_tq, item, content, mwdhm, lab, lane);
        lab_score = ls;
    }
    for (int j = 0; j < 32; ++j) {
        // one candidate per warp iteration: 3-4 CTAs per SM x 8 warps keep ~50 KB of row loads in flight per SM, which
        // already saturates L2/HBM for these 2 KB random rows (a 4-way unrolled variant needed 110 registers, fell to
        // 2 CTAs per SM and was slower: 151 vs 121 us)
        const int ci = w * 32 + j;
        const int chunk = s_sel[ci / CH];
        const int n = chunk < 0 ? -1 : chunk * CH + (ci % CH);          // local item id
        const bool ok = n >= 0 && n < N;
        float sc = -INFINITY;
        if (ok) sc = exact_score_e(s_aic, s_tq, item, content, mwdhm, n + item_offset, lane);
        if (lane == 0) {
            s_sc[ci] = sc;
            s_id[ci] = ok ? n + item_offset : 0x7fffffff;
        }
    }
    __syncthreads();
    // n_greater: strict, never counts the label itself                       (util.py:14)
    {
        const bool gt = s_id[tid] != 0x7fffffff && s_id[tid] != lab && s_sc[tid] > lab_score;
        const uint32_t bal = __ballot_sync(0xffffffffu, gt);
        if (lane == 0) s_warp[w] = __popc(bal);
    }
    __syncthreads();
    if (tid == 0) {
        int t = 0;
        for (int j = 0; j < 8; ++j) t += s_warp[j];
        n_greater[b] = t;
    }
    // bitonic sort of 256 (score, id) pairs, ascending in "before" order
    for (int k = 2; k <= NCAND; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            __syncthreads();
            const int ixj = tid ^ j;
            if (ixj > tid) {
                const float sa = s_sc[tid], sb = s_sc[ixj];
                const int ia = s_id[tid], ib = s_id[ixj];
                const bool up = (tid & k) == 0;
                const bool swap = up ? before(sb, ib, sa, ia) : before(sa, ia, sb, ib);
                if (swap) { s_sc[tid] = sb; s_sc[ixj] = sa; s_id[tid] = ib; s_id[ixj] = ia; }
            }
        }
    }
    __syncthreads();
    if (tid < TOPK) {
        top_ids[(size_t)b * TOPK + tid] = s_id[tid] == 0x7fffffff ? -1 : s_id[tid];
        top_scores[(size_t)b * TOPK + tid] = s_sc[tid];
    }
    if (cat_stats) {
        // certification: nothing outside the re-scored chunks can reach the 20th exact score
        const float s20 = s_sc[TOPK - 1];
        const float eps = score_error_bound(s_aic, s_tq, cat_stats, s_red);
        if (tid == 0) {
            const float bound = s20 - eps;
            // s20 == -inf: fewer than 20 candidates re-scored, i.e. every chunk of a tiny catalog was taken
            uncertain[b] = ((nchunks > NCH || from_lists) && unsel_max > -INFINITY && !(unsel_max < bound)) ? 1 : 0;
            tau[b] = bound;
        }
    }
}

// Second stage for the queries tcar_eval_topk could not certify: every chunk whose maximum reaches tau[b] = s20 - eps_b
// is re-scored exactly (tiles below tau are skipped by their tile maximum), 32 chunks at a time, and merged into a
// running top-20 by (score desc, id asc); n_greater is counted over the same exact scores.  The result is the exact
// top-20 of the whole catalog (items below tau cannot reach the 20th score already found).  Cost grows with the number
// of near-ties (in the limit a full exact scan), so a flagged query is spread over TCAR_WIDEN_SPLITS CTAs, each taking
// a contiguous range of tiles and leaving a partial list in the workspace; the merge kernel behind it combines them.
// A certified query costs nothing (its CTAs return at once).
constexpr int WQ_CAP = 4096;        // chunk queue: one sweep of 256 tiles x 16 chunks
constexpr int WSPLIT = TCAR_WIDEN_SPLITS;
// workspace per group: partial lists [S][512][20] ids | scores, counts [S][512], then one ticket per query (zero between
// launches: the split CTA that arrives last merges the query's partial lists and resets it)
constexpr size_t W_LIST_WORDS = (size_t)TCAR_WIDEN_SPLITS * TCAR_QROWS * (2 * TCAR_TOPK + 1);
constexpr size_t W_GROUP_WORDS = W_LIST_WORDS + TCAR_QROWS;

// several session groups in one launch of the widening pass / its merge (blockIdx.z resp. blockIdx.y = group)
struct WidenGroups {
    int groups;
    int n[TCAR_MAX_PEERS];
    long long cm_gs, tm_gs;      // floats between the groups' chunk / tile maxima
    long long q_gs;              // words between the groups' a_ic / Tq / label planes (one exchange block per group)
    long long flag_gs;           // words between the groups' uncertain / tau vectors
    long long out_gs;            // words between the groups' result planes (top_ids / top_scores / n_greater)
};
constexpr int WIDEN_SLOTS = 37;     // x 16 splits = 592 CTAs = 4 per SM: one wave

__device__ __forceinline__ void warp_merge_lists(const int32_t* ids, const float* scores, int G, int B, long long gstride,
                                                 int b, int lane, int32_t* out_ids, float* out_scores);

// The WSPLIT CTAs of a flagged query each scan their share of the item range; the one that finishes last (ticket
// counter behind the partial lists) merges the WSPLIT partial lists into the query's result -- no second launch.
__global__ void __launch_bounds__(256)
eval_topk_widen_kernel(const float* chunkmax, const float* tilemax, const float* a_ic, const float* Tq,
                       const float* __restrict__ item, const float* __restrict__ content,
                       const int32_t* __restrict__ mwdhm, const int32_t* label, const int32_t* uncertain,
                       const float* tau, int32_t* wspace, int32_t* out_ids, float* out_scores, int32_t* out_ngt, int N,
                       int n_pad, int item_offset, int B, const __grid_constant__ WidenGroups wg) {
    PDL_ENTER();
    const int split = blockIdx.y, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (wg.groups > 0) {
        const int g = blockIdx.z;
        B = wg.n[g];
        if (B <= 0) return;
        chunkmax += (size_t)g * wg.cm_gs;
        tilemax += (size_t)g * wg.tm_gs;
        a_ic += (size_t)g * wg.q_gs;
        Tq += (size_t)g * wg.q_gs;
        label += (size_t)g * wg.q_gs;
        uncertain += (size_t)g * wg.flag_gs;
        tau += (size_t)g * wg.flag_gs;
        wspace += (size_t)g * W_GROUP_WORDS;
        out_ids += (size_t)g * wg.out_gs;
        out_scores += (size_t)g * wg.out_gs;
        out_ngt += (size_t)g * wg.out_gs;
    }
    // partial lists of this launch: ids [S][B][20] | scores [S][B][20] | counts [S][B]
    int32_t* top_ids = wspace;
    float* top_scores = reinterpret_cast<float*>(wspace + (size_t)WSPLIT * TCAR_QROWS * TOPK);
    int32_t* n_greater = wspace + 2 * (size_t)WSPLIT * TCAR_QROWS * TOPK;
    int32_t* ticket = wspace + W_LIST_WORDS;
    __shared__ int s_last;
    // compact list of the flagged queries (ascending, built identically by every CTA): the grid is WIDEN_SLOTS x
    // WSPLIT CTAs whatever B is, CTA (i, s) takes the flagged queries i, i + WIDEN_SLOTS, ...
    __shared__ int s_flag[TCAR_QROWS];
    __shared__ int s_unc[TCAR_QROWS];
    __shared__ int s_nflag;
    for (int i = tid; i < TCAR_QROWS; i += 256) s_unc[i] = i < B ? uncertain[i] : 0;    // two loads in flight per thread
    __syncthreads();
    if (w == 0) {
        int cnt = 0;
        for (int base = 0; base < B; base += 32) {
            const bool f = s_unc[base + lane] != 0;
            const uint32_t bal = __ballot_sync(0xffffffffu, f);
            if (f) s_flag[cnt + __popc(bal & ((1u << lane) - 1u))] = base + lane;
            cnt += __popc(bal);
        }
        if (lane == 0) s_nflag = cnt;
    }
    __syncthreads();
    if ((int)blockIdx.x >= s_nflag) return;
    __shared__ float s_aic[XW], s_tq[NB + 1];
    __shared__ int s_q[WQ_CAP];
    __shared__ int s_qn, s_ngt;
    __shared__ float s_sc[NCAND];
    __shared__ int s_id[NCAND];
    __shared__ float s_top_sc[TOPK], s_new_sc[TOPK];
    __shared__ int s_top_id[TOPK], s_new_id[TOPK];
    __shared__ int s_warp[8];
    const int nchunks = (N + CH - 1) / CH;
    const int ntiles = (N + 127) / 128;
  for (int fi = blockIdx.x; fi < s_nflag; fi += gridDim.x) {
    const int b = s_flag[fi];
    const float* cm = chunkmax + (size_t)b * (n_pad / CH);
    const float* tm = tilemax + (size_t)b * (n_pad / 128);
    const float bound = tau[b];
    __syncthreads();                     // previous query's shared state fully consumed
    for (int c = tid; c < XW; c += 256) s_aic[c] = a_ic[(size_t)b * XW + c];
    for (int c = tid; c < NB; c += 256) s_tq[c] = Tq[(size_t)b * NB + c];
    if (tid < TOPK) { s_top_sc[tid] = -INFINITY; s_top_id[tid] = 0x7fffffff; }
    if (tid == 0) { s_qn = 0; s_ngt = 0; }
    __syncthreads();
    const int lab = label[b];
    const float lab_score = exact_score_e(s_aic, s_tq, item, content, mwdhm, lab, lane);
    const int per = (ntiles + WSPLIT - 1) / WSPLIT;
    const int t_lo = split * per, t_hi = min(t_lo + per, ntiles);
    for (int t0 = t_lo; t0 < t_hi; t0 += 256) {
        const int tile = t0 + tid;
        if (tile < t_hi && tm[tile] >= bound) {
            // the tile's 16 chunk maxima: four 16-byte loads issued together (cm rows are 16-byte aligned: n_pad % 256 == 0)
            float4 v[TILE_CH / 4];
#pragma unroll
            for (int c = 0; c < TILE_CH / 4; ++c) v[c] = reinterpret_cast<const float4*>(cm + (size_t)tile * TILE_CH)[c];
#pragma unroll
            for (int c = 0; c < TILE_CH; ++c) {
                const int chunk = tile * TILE_CH + c;
                const float cv = c % 4 == 0 ? v[c / 4].x : c % 4 == 1 ? v[c / 4].y : c % 4 == 2 ? v[c / 4].z : v[c / 4].w;
                if (chunk < nchunks && cv >= bound) s_q[atomicAdd(&s_qn, 1)] = chunk;
            }
        }
        __syncthreads();
        const int qn = s_qn;
        for (int q0 = 0; q0 < qn; q0 += NCH) {
            // exact scores of up to 32 queued chunks
            const int ncand = min(qn - q0, NCH) * CH;            // candidates of this batch
            int P = 32;                                           // sort size: power of two >= max(ncand, 20)
            while (P < ncand) P <<= 1;
            if (tid < P) { s_sc[tid] = -INFINITY; s_id[tid] = 0x7fffffff; }
            __syncthreads();
            for (int ci = w; ci < ncand; ci += 32) {              // interleaved: few candidates -> few iterations
                // four candidates per warp and iteration, branch-free, so that the 16 row loads of a lane are all in
                // flight before the first dot product (a candidate costs one DRAM round trip otherwise)
                int nn[4];
                float sc[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int cu = ci + 8 * u;
                    const int n = cu < ncand ? s_q[q0 + cu / CH] * CH + (cu % CH) : N;
                    nn[u] = n < N ? n + item_offset : -1;
                }
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    sc[u] = exact_score_e(s_aic, s_tq, item, content, mwdhm, nn[u] >= 0 ? nn[u] : 0, lane);
                if (lane == 0) {
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (nn[u] >= 0) { s_sc[ci + 8 * u] = sc[u]; s_id[ci + 8 * u] = nn[u]; }
                }
            }
            __syncthreads();
            {
                const bool gt = tid < P && s_id[tid] != 0x7fffffff && s_id[tid] != lab && s_sc[tid] > lab_score;
                const uint32_t bal = __ballot_sync(0xffffffffu, gt);
                if (lane == 0) s_warp[w] = __popc(bal);
            }
            for (int k = 2; k <= P; k <<= 1) {
                for (int j = k >> 1; j > 0; j >>= 1) {
                    __syncthreads();
                    const int ixj = tid ^ j;
                    if (tid < P && ixj > tid) {
                        const float sa = s_sc[tid], sb = s_sc[ixj];
                        const int ia = s_id[tid], ib = s_id[ixj];
                        const bool up = (tid & k) == 0;
                        const bool swap = up ? before(sb, ib, sa, ia) : before(sa, ia, sb, ib);
                        if (swap) { s_sc[tid] = sb; s_sc[ixj] = sa; s_id[tid] = ib; s_id[ixj] = ia; }
                    }
                }
            }
            __syncthreads();
            if (tid == 0) {
                for (int j = 0; j < 8; ++j) s_ngt += s_warp[j];
                // merge the running list with the 20 best of this batch (both sorted)
                int ia = 0, ib = 0;
                for (int r = 0; r < TOPK; ++r) {
                    if (before(s_top_sc[ia], s_top_id[ia], s_sc[ib], s_id[ib])) {
                        s_new_sc[r] = s_top_sc[ia]; s_new_id[r] = s_top_id[ia]; ++ia;
                    } else {
                        s_new_sc[r] = s_sc[ib]; s_new_id[r] = s_id[ib]; ++ib;
                    }
                }
                for (int r = 0; r < TOPK; ++r) { s_top_sc[r] = s_new_sc[r]; s_top_id[r] = s_new_id[r]; }
            }
            __syncthreads();
        }
        if (tid == 0) s_qn = 0;
        __syncthreads();
    }
    // partial lists [WSPLIT][B][20] / counts [WSPLIT][B] in the workspace
    const size_t slot = (size_t)split * B + b;
    if (tid < TOPK) {
        top_ids[slot * TOPK + tid] = s_top_id[tid] == 0x7fffffff ? -1 : s_top_id[tid];
        top_scores[slot * TOPK + tid] = s_top_sc[tid];
    }
    if (tid == 0) n_greater[slot] = s_ngt;
    // last split CTA of this query: merge the WSPLIT partial lists (written by other CTAs: fence, ticket, fence)
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(&ticket[b], 1) == WSPLIT - 1;
    __syncthreads();
    if (s_last) {
        __threadfence();
        if (w == 0) {
            if (lane == 0) {
                int cnt = 0;
                for (int g = 0; g < WSPLIT; ++g) cnt += n_greater[(size_t)g * B + b];
                out_ngt[b] = cnt;
                ticket[b] = 0;
            }
            warp_merge_lists(top_ids, top_scores, WSPLIT, B, 0LL, b, lane, out_ids, out_scores);
        }
    }
  }
}

// Catalog statistics behind eps_b: out[0] = max_n ||[item | content] row n||_2, out[1] = max_n ||row n - bf16(row n)||_2
// over table rows [row_lo, row_hi).  One warp per row; non-negative floats order like their bit patterns (atomicMax).
__global__ void __launch_bounds__(256)
catalog_stats_kernel(const float* __restrict__ item, const float* __restrict__ content, int row_lo, int row_hi,
                     float* __restrict__ out) {
    PDL_ENTER();
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    float mx = 0.f, dmx = 0.f;
    for (int row = row_lo + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5); row < row_hi; row += warps) {
        float n2 = 0.f, d2 = 0.f;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const float4 iv = __ldg(reinterpret_cast<const float4*>(item + (size_t)row * HP) + j * 32 + lane);
            const float4 cv = __ldg(reinterpret_cast<const float4*>(content + (size_t)row * HP) + j * 32 + lane);
            const float v[8] = {iv.x, iv.y, iv.z, iv.w, cv.x, cv.y, cv.z, cv.w};
            const int c = j * 128 + lane * 4;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                if (c + (u & 3) < H) {
                    const float d = v[u] - bf16_round(v[u]);
                    n2 = fmaf(v[u], v[u], n2);
                    d2 = fmaf(d, d, d2);
                }
            }
        }
        n2 = warp_sum_e(n2);
        d2 = warp_sum_e(d2);
        mx = fmaxf(mx, n2);
        dmx = fmaxf(dmx, d2);
    }
    if (lane == 0) {
        atomicMax(reinterpret_cast<int*>(out), __float_as_int(sqrtf(mx) * 1.000001f));
        atomicMax(reinterpret_cast<int*>(out) + 1, __float_as_int(sqrtf(dmx) * 1.000001f));
    }
}

// One warp merges the G sorted lists of query b (G * 20 <= 32 * 32 entries) into the 20 best by (score desc, id asc).
// Lists: [G][B][20] back to back (gstride == 0) or one block of `gstride` words per list owner.
__device__ __forceinline__ void warp_merge_lists(const int32_t* ids, const float* scores, int G, int B, long long gstride,
                                                 int b, int lane, int32_t* out_ids, float* out_scores) {
    const int n = G * TOPK;
    uint32_t taken = 0;           // each lane owns entries lane, lane + 32, ...: one `taken` bit per owned entry
    for (int r = 0; r < TOPK; ++r) {
        float bs = -INFINITY; int bi = 0x7fffffff, bslot = -1;
        for (int e = lane, s = 0; e < n; e += 32, ++s) {
            if (taken & (1u << s)) continue;
            const int g = e / TOPK, j = e % TOPK;
            const size_t at = gstride ? (size_t)g * gstride + (size_t)b * TOPK + j : ((size_t)g * B + b) * TOPK + j;
            const float sc = scores[at];
            int id = ids[at];
            if (id < 0) id = 0x7fffffff;
            if (before(sc, id, bs, bi)) { bs = sc; bi = id; bslot = s; }
        }
        float ws = bs; int wi = bi;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float os = __shfl_xor_sync(0xffffffffu, ws, o);
            const int oi = __shfl_xor_sync(0xffffffffu, wi, o);
            if (before(os, oi, ws, wi)) { ws = os; wi = oi; }
        }
        if (bslot >= 0 && bs == ws && bi == wi && wi != 0x7fffffff) taken |= 1u << bslot;
        if (lane == 0) {
            out_ids[(size_t)b * TOPK + r] = wi == 0x7fffffff ? -1 : wi;
            out_scores[(size_t)b * TOPK + r] = ws;
        }
    }
}

// merge G shard lists: one warp per query, serial selection (G*20 <= 160 entries)
__global__ void __launch_bounds__(256)
topk_merge_kernel(const int32_t* ids, const float* scores, int32_t* out_ids, float* out_scores, int G, int B,
                  long long gstride, const int32_t* ngt, const float* __restrict__ sumexp,
                  const float* __restrict__ rowmax, int32_t* out_ngt, float* __restrict__ out_ce,
                  const int32_t* only_if,
                  const __grid_constant__ WidenGroups wg) {
    PDL_ENTER();
    const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (wg.groups > 0) {
        // the widening pass's own merge, one group per blockIdx.y: inputs in the group's workspace, outputs and flags
        // in the group's result block
        const int g = blockIdx.y;
        B = wg.n[g];
        ids += (size_t)g * W_GROUP_WORDS;
        scores += (size_t)g * W_GROUP_WORDS;
        ngt += (size_t)g * W_GROUP_WORDS;
        out_ids += (size_t)g * wg.out_gs;
        out_scores += (size_t)g * wg.out_gs;
        out_ngt += (size_t)g * wg.out_gs;
        only_if += (size_t)g * wg.flag_gs;
    }
    if (b >= B) return;
    if (only_if && !only_if[b]) return;      // widening pass: certified queries keep their result
    if (ngt && !sumexp && lane == 0) {
        // partial rank counts of the widening pass ([G][B], like the lists)
        int cnt = 0;
        for (int g = 0; g < G; ++g) cnt += ngt[gstride ? (size_t)g * gstride + b : (size_t)g * B + b];
        out_ngt[b] = cnt;
    }
    if (ngt && sumexp && lane == 0) {
        // rank counts add up; the shards' softmax sums are relative to their own exponent shifts (overflow guard):
        // sum_g sumexp_g 2^(shift_g - M) with M the largest shift, CE = log(sum) + M ln 2 = logsumexp(S_b) - S_b[label]
        int cnt = 0;
        float M = 0.f;
        for (int g = 0; g < G; ++g) {
            cnt += ngt[g * gstride + b];
            const float r = rowmax ? rowmax[g * gstride + b] : 0.f;
            M = fmaxf(M, r > TCAR_EXP_LIMIT2 ? r : 0.f);
        }
        float tot = 0.f;
        for (int g = 0; g < G; ++g) {
            const float r = rowmax ? rowmax[g * gstride + b] : 0.f;
            tot += sumexp[g * gstride + b] * exp2f((r > TCAR_EXP_LIMIT2 ? r : 0.f) - M);
        }
        out_ngt[b] = cnt;
        out_ce[b] = fmaf(M, 0.6931471805599453f, logf(tot));
    }
    warp_merge_lists(ids, scores, G, B, gstride, b, lane, out_ids, out_scores);
}

// ------------------------------------------------------------------------------------------------ candidate re-ranking
// One CTA per session.  Warp w scores the list entries w, w + 8, w + 16, w + 24, then the next 32, with exact_score_e
// (the re-scoring arithmetic of the full-catalog top-20): four candidates per warp and iteration, branch-free, so that
// a lane's 16 row loads are in flight before the first dot product, as in the widening pass.  Every candidate row is
// used once per session, so this is a gather plus a GEMV: no tensor cores.  The order is found by counting -- entry i
// goes to position #{j : key_j < key_i, or key_j == key_i and j < i} -- with no sort network and no atomics, so
// repeated runs are bit-identical.
constexpr int RMAXL = TCAR_RERANK_MAXL;

// ascending key = (score desc, id asc).  +0 and -0 are equal scores and share a key; NaN gets a place in the order
// (fkey is total on bit patterns), so the positions always form a permutation.
__device__ __forceinline__ unsigned long long rerank_key(float s, int id) {
    const uint32_t k = fkey(s == 0.f ? 0.f : s);
    return ((unsigned long long)(~k) << 32) | (uint32_t)id;
}

__global__ void __launch_bounds__(256)
rerank_kernel(const float* __restrict__ a_ic, const float* __restrict__ Tq, const float* __restrict__ item,
              const float* __restrict__ content, const int32_t* __restrict__ mwdhm,
              const int32_t* __restrict__ cand_off, const int32_t* __restrict__ cand_ids,
              const int32_t* __restrict__ label, int N, int max_len, float* __restrict__ scores,
              int32_t* __restrict__ ranked, int32_t* __restrict__ label_rank, float* __restrict__ auc) {
    PDL_ENTER();
    __shared__ float s_aic[XW], s_tq[NB + 1];
    __shared__ float s_sc[RMAXL];
    __shared__ unsigned long long s_key[RMAXL];
    __shared__ float s_lab;
    __shared__ int s_cnt[3][8];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int off = cand_off[b], L = cand_off[b + 1] - off;
    if (L < 0 || L > max_len) return;               // block-uniform; the shared arrays hold max_len entries
    for (int c = tid; c < XW; c += 256) s_aic[c] = a_ic[(size_t)b * XW + c];
    for (int c = tid; c < NB; c += 256) s_tq[c] = Tq[(size_t)b * NB + c];
    __syncthreads();
    const int lab = label ? label[b] : -1;
    const bool lab_ok = lab >= 0 && lab < N;
    if (label && w == 0) {
        const float ls = exact_score_e(s_aic, s_tq, item, content, mwdhm, lab_ok ? lab : 0, lane);
        if (lane == 0) s_lab = lab_ok ? ls : NAN;
    }
    const int32_t* ids = cand_ids + off;
    for (int c0 = w; c0 < L; c0 += 32) {
        int raw[4];
        bool ok[4];
        float sc[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int c = c0 + 8 * u;
            raw[u] = c < L ? ids[c] : -1;
            ok[u] = raw[u] >= 0 && raw[u] < N;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) sc[u] = exact_score_e(s_aic, s_tq, item, content, mwdhm, ok[u] ? raw[u] : 0, lane);
        if (lane == 0) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int c = c0 + 8 * u;
                if (c < L) {
                    const float s = ok[u] ? sc[u] : NAN;
                    s_sc[c] = s;
                    s_key[c] = rerank_key(s, raw[u]);
                    scores[off + c] = s;
                }
            }
        }
    }
    __syncthreads();
    const float sl = label ? s_lab : 0.f;
    int gt = 0, eq = 0, nneg = 0;
    for (int i = tid; i < L; i += 256) {
        const unsigned long long ki = s_key[i];
        int pos = 0;
#pragma unroll 4
        for (int j = 0; j < L; ++j) {               // every lane reads the same s_key[j]: a broadcast
            const unsigned long long kj = s_key[j];
            pos += (kj < ki) | ((kj == ki) & (j < i));
        }
        const int id = (int)(uint32_t)ki;
        ranked[off + pos] = id;
        if (label && id != lab) {
            const float s = s_sc[i];
            ++nneg;
            gt += s > sl;
            eq += s == sl;
        }
    }
    if (!label) return;
    gt = __reduce_add_sync(0xffffffffu, gt);
    eq = __reduce_add_sync(0xffffffffu, eq);
    nneg = __reduce_add_sync(0xffffffffu, nneg);
    if (lane == 0) { s_cnt[0][w] = gt; s_cnt[1][w] = eq; s_cnt[2][w] = nneg; }
    __syncthreads();
    if (tid == 0) {
        int g = 0, e = 0, n = 0;
        for (int k = 0; k < 8; ++k) { g += s_cnt[0][k]; e += s_cnt[1][k]; n += s_cnt[2][k]; }
        label_rank[b] = lab_ok ? 1 + g : 0;                                               // util.py:14
        auc[b] = lab_ok && n > 0 ? ((float)(n - g - e) + 0.5f * (float)e) / (float)n : NAN;
    }
}

// ------------------------------------------------------------------------------------------------ top-K recommendation
// The exact top-K of the whole catalog per session, K <= 256, with up to 1024 excluded ids per session, in two launches
// behind the eval-mode scoring GEMM (chunk / tile maxima of the bf16 scores):
//   select  one CTA per query: K' = K + x_b (x_b = the session's exclusion entries, duplicates counted),
//           tau_hi = the K'-th largest chunk maximum, tau_b = tau_hi - 2 eps_b (eps_b = score_error_bound);
//           tau_b = -inf (a full exact scan) when K' >= the number of chunks.
//   scan    TCAR_WIDEN_SPLITS CTAs per query over contiguous tile ranges: tiles whose maximum is below tau_b are
//           skipped, chunks whose maximum reaches tau_b are re-scored exactly (exact_score_e) except for excluded
//           ids (sorted list in shared memory, tested before the row loads) and ids >= N, and merged into a running
//           top-K; the split CTA that finishes last (ticket counter) merges the partial lists.
// Why the result is exact: the K' chunks with the largest maxima hold K' distinct valid items (chunk maxima mask items
// >= N to -inf) whose bf16 scores are >= tau_hi.  At most x_b of them are excluded, so at least K eligible items score
// >= tau_hi - eps_b exactly, i.e. the exact K-th best eligible score s_K >= tau_hi - eps_b.  Every member of the exact
// top-K (ties included) scores >= s_K exactly, so its bf16 score is >= s_K - eps_b >= tau_b: its chunk is re-scored.
// The order is the total order of rerank_key (score desc, id asc) and every item is re-scored by exactly one CTA, so
// the order in which chunks are queued (shared-memory atomics) cannot change the result: reruns are bit-identical.
constexpr int RK = TCAR_RECOMMEND_MAXK;
constexpr int RX = TCAR_RECOMMEND_MAXX;
constexpr int TL_CAP = 4096;                     // tiles listed for the chunk-level selection (more: scan every tile)
constexpr unsigned long long KEY_NONE = ~0ull;   // empty slot: after every real key

__device__ __forceinline__ float key_value(uint32_t k) {                     // inverse of fkey
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// fkey of the k-th largest of get(0 .. n) (1 <= k <= n) by four 8-bit radix passes.  256 threads, s_hist [256],
// s_misc [2].  The values of one query sit in a narrow range, so lanes with equal bins are combined (match_any) before
// the shared-memory atomic.
template <class Get>
__device__ __forceinline__ uint32_t block_kth_key(int n, int k, Get get, int* s_hist, int* s_misc) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    uint32_t prefix = 0, mask = 0;
    for (int shift = 24; shift >= 0; shift -= 8) {
        s_hist[tid] = 0;
        __syncthreads();
        for (int i0 = 0; i0 < n; i0 += 256) {                         // block-uniform trip count (match_any below)
            const int i = i0 + tid;
            const uint32_t key = i < n ? fkey(get(i)) : 0u;
            const bool act = i < n && (key & mask) == prefix;
            const uint32_t bin = act ? ((key >> shift) & 255u) : 256u;
            const uint32_t peers = __match_any_sync(0xffffffffu, bin);
            if (act && lane == __ffs(peers) - 1) atomicAdd(&s_hist[bin], __popc(peers));
        }
        __syncthreads();
        if (w == 0) {                                                 // lane l owns bins 8l .. 8l+7
            int cnt[8], tot = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) { cnt[j] = s_hist[lane * 8 + j]; tot += cnt[j]; }
            int suf = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_down_sync(0xffffffffu, suf, o);
                if (lane + o < 32) suf += v;
            }
            const int above_lane = suf - tot;
            const bool mine = above_lane < k && k <= suf;
            if (mine) {
                int a = above_lane;
                for (int j = 7; j >= 0; --j) {
                    if (a + cnt[j] >= k) { s_misc[0] = lane * 8 + j; s_misc[1] = a; break; }
                    a += cnt[j];
                }
            }
        }
        __syncthreads();
        prefix |= (uint32_t)s_misc[0] << shift;
        mask |= 255u << shift;
        k -= s_misc[1];
    }
    __syncthreads();
    return prefix;
}

__global__ void __launch_bounds__(256)
recommend_select_kernel(const float* chunkmax, const float* tilemax, const float* __restrict__ a_ic,
                        const float* __restrict__ Tq, const float* __restrict__ cat_stats,
                        const int32_t* __restrict__ x_off, int n_clicks, int K, int N, int n_pad,
                        float* __restrict__ tau) {
    PDL_ENTER();
    __shared__ float s_aic[XW], s_tq[NB + 1];
    __shared__ float s_red[32];
    __shared__ int s_hist[256], s_misc[2];
    __shared__ int s_tl[TL_CAP];
    __shared__ int s_ntl;
    const int b = blockIdx.x, tid = threadIdx.x;
    const int nchunks = (N + CH - 1) / CH, ntiles = (N + 127) / 128;
    const int kp = K + (x_off ? x_off[b + 1] - x_off[b] : 0) + n_clicks;
    if (kp >= nchunks) {                                              // block-uniform
        if (tid == 0) tau[b] = -INFINITY;
        return;
    }
    const float* cm = chunkmax + (size_t)b * (n_pad / CH);
    const float* tm = tilemax + (size_t)b * (n_pad / 128);
    for (int c = tid; c < XW; c += 256) s_aic[c] = a_ic[(size_t)b * XW + c];
    for (int c = tid; c < NB; c += 256) s_tq[c] = Tq[(size_t)b * NB + c];
    if (tid == 0) s_ntl = 0;
    __syncthreads();
    // The K' largest tile maxima are K' distinct chunk values, so the K'-th largest chunk is >= the K'-th largest tile
    // maximum: tiles below it cannot hold one of the K' best chunks.
    float thr = -INFINITY;
    if (ntiles > kp) thr = key_value(block_kth_key(ntiles, kp, [&](int i) { return tm[i]; }, s_hist, s_misc));
    for (int i = tid; i < ntiles; i += 256)
        if (tm[i] >= thr) {
            const int at = atomicAdd(&s_ntl, 1);
            if (at < TL_CAP) s_tl[at] = i;
        }
    __syncthreads();
    const bool listed = s_ntl <= TL_CAP;                              // else ties: every tile
    const int n = (listed ? s_ntl : ntiles) * TILE_CH;
    const uint32_t kk = block_kth_key(n, kp, [&](int i) {
        const int c = (listed ? s_tl[i / TILE_CH] : i / TILE_CH) * TILE_CH + i % TILE_CH;
        return c < nchunks ? cm[c] : -INFINITY;
    }, s_hist, s_misc);
    const float eps = score_error_bound(s_aic, s_tq, cat_stats, s_red);
    if (tid == 0) tau[b] = key_value(kk) - 2.f * eps;
}

// number of entries of a sorted list below x
__device__ __forceinline__ int rank_in(const unsigned long long* a, int n, unsigned long long x) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a[mid] < x) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// out[0 .. K) = the K smallest keys of the ascending lists a[0 .. K) and c[0 .. nc), by merge path: an entry's place is
// its index plus its rank in the other list (real keys are distinct; KEY_NONE slots write KEY_NONE wherever they
// collide).  Ends with a barrier.
__device__ __forceinline__ void merge_topk(const unsigned long long* a, int K, const unsigned long long* c, int nc,
                                           unsigned long long* out) {
    for (int i = threadIdx.x; i < K; i += 256) {
        const unsigned long long v = a[i];
        const int pos = i + rank_in(c, nc, v);
        if (pos < K) out[pos] = v;
    }
    for (int j = threadIdx.x; j < nc && j < K; j += 256) {
        const unsigned long long v = c[j];
        const int pos = j + rank_in(a, K, v);
        if (pos < K) out[pos] = v;
    }
    __syncthreads();
}

// workspace: tickets [512] (zero between calls; at fixed places, whatever B a call has) | tau [B] |
// re-scored counts [S][B] | partial lists [S][B][256] keys
__host__ __device__ constexpr size_t rec_keys_offset(int B) {
    return ((size_t)(TCAR_QROWS + (1 + WSPLIT) * B) * 4 + 7) / 8 * 8;
}

__global__ void __launch_bounds__(256, 2)
recommend_scan_kernel(const float* chunkmax, const float* tilemax, const float* __restrict__ a_ic,
                      const float* __restrict__ Tq, const float* __restrict__ item, const float* __restrict__ content,
                      const int32_t* __restrict__ mwdhm, const int32_t* __restrict__ x_off,
                      const int32_t* __restrict__ x_ids, const int32_t* __restrict__ clicks, int n_clicks, int K, int N,
                      int n_pad, int B, char* wspace, int32_t* __restrict__ out_ids, float* __restrict__ out_scores,
                      int32_t* __restrict__ rescored) {
    PDL_ENTER();
    __shared__ float s_aic[XW], s_tq[NB + 1];
    __shared__ int s_x[RX];
    __shared__ int s_q[WQ_CAP];
    __shared__ unsigned long long s_top[2][RK];
    __shared__ unsigned long long s_new[NCAND];
    __shared__ int s_qn, s_cnt, s_last;
    const int b = blockIdx.x, split = blockIdx.y, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    int32_t* ticket = reinterpret_cast<int32_t*>(wspace);
    const float* tau = reinterpret_cast<const float*>(wspace) + TCAR_QROWS;
    int32_t* part_cnt = reinterpret_cast<int32_t*>(wspace) + TCAR_QROWS + B;
    unsigned long long* part = reinterpret_cast<unsigned long long*>(wspace + rec_keys_offset(B));
    const int xo = x_off ? x_off[b] : 0;
    const int nl = x_off ? x_off[b + 1] - xo : 0, nx = nl + n_clicks;
    if (nl < 0 || nx > RX) return;                                   // block-uniform, and the same for every split
    // the exclusion list, sorted ascending (padded with INT_MAX to a power of two)
    int P = 1;
    while (P < nx) P <<= 1;
    for (int i = tid; i < P; i += 256)
        s_x[i] = i < nl ? x_ids[xo + i] : i < nx ? clicks[(size_t)b * n_clicks + (i - nl)] - 1 : 0x7fffffff;
    for (int c = tid; c < XW; c += 256) s_aic[c] = a_ic[(size_t)b * XW + c];
    for (int c = tid; c < NB; c += 256) s_tq[c] = Tq[(size_t)b * NB + c];
    for (int i = tid; i < RK; i += 256) s_top[0][i] = KEY_NONE;
    if (tid == 0) { s_qn = 0; s_cnt = 0; }
    __syncthreads();
    for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < P; i += 256) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const int a = s_x[i], c = s_x[ixj];
                    if (((i & k) == 0) ? a > c : a < c) { s_x[i] = c; s_x[ixj] = a; }
                }
            }
            __syncthreads();
        }
    }
    auto excluded = [&](int n) {
        int lo = 0, hi = nx;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (s_x[mid] < n) lo = mid + 1; else hi = mid;
        }
        return lo < nx && s_x[lo] == n;
    };
    const int nchunks = (N + CH - 1) / CH, ntiles = (N + 127) / 128;
    const float* cm = chunkmax + (size_t)b * (n_pad / CH);
    const float* tm = tilemax + (size_t)b * (n_pad / 128);
    const float bound = tau[b];
    const int per = (ntiles + WSPLIT - 1) / WSPLIT;
    const int t_lo = split * per, t_hi = min(t_lo + per, ntiles);
    int cur = 0, my_cnt = 0;
    for (int t0 = t_lo; t0 < t_hi; t0 += 256) {
        const int tile = t0 + tid;
        if (tile < t_hi && tm[tile] >= bound) {
            float4 v[TILE_CH / 4];
#pragma unroll
            for (int c = 0; c < TILE_CH / 4; ++c) v[c] = reinterpret_cast<const float4*>(cm + (size_t)tile * TILE_CH)[c];
#pragma unroll
            for (int c = 0; c < TILE_CH; ++c) {
                const int chunk = tile * TILE_CH + c;
                const float cv = c % 4 == 0 ? v[c / 4].x : c % 4 == 1 ? v[c / 4].y : c % 4 == 2 ? v[c / 4].z : v[c / 4].w;
                if (chunk < nchunks && cv >= bound) s_q[atomicAdd(&s_qn, 1)] = chunk;
            }
        }
        __syncthreads();
        const int qn = s_qn;
        for (int q0 = 0; q0 < qn; q0 += NCH) {
            const int ncand = min(qn - q0, NCH) * CH;
            int P2 = 32;                                              // sort size: power of two >= ncand
            while (P2 < ncand) P2 <<= 1;
            if (tid < P2) s_new[tid] = KEY_NONE;
            __syncthreads();
            for (int ci = w; ci < ncand; ci += 32) {
                // four candidates per warp and iteration, branch-free, as in the widening pass; an excluded id or one
                // >= N reads row 0 instead of its own
                int nn[4];
                float sc[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int cu = ci + 8 * u;
                    const int n = cu < ncand ? s_q[q0 + cu / CH] * CH + (cu % CH) : N;
                    nn[u] = n < N && !excluded(n) ? n : -1;
                }
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    sc[u] = exact_score_e(s_aic, s_tq, item, content, mwdhm, nn[u] >= 0 ? nn[u] : 0, lane);
                if (lane == 0) {
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (nn[u] >= 0) { s_new[ci + 8 * u] = rerank_key(sc[u], nn[u]); ++my_cnt; }
                }
            }
            for (int k = 2; k <= P2; k <<= 1) {
                for (int j = k >> 1; j > 0; j >>= 1) {
                    __syncthreads();
                    const int ixj = tid ^ j;
                    if (tid < P2 && ixj > tid) {
                        const unsigned long long a = s_new[tid], c = s_new[ixj];
                        if (((tid & k) == 0) ? a > c : a < c) { s_new[tid] = c; s_new[ixj] = a; }
                    }
                }
            }
            __syncthreads();
            merge_topk(s_top[cur], K, s_new, P2, s_top[cur ^ 1]);
            cur ^= 1;
        }
        if (tid == 0) s_qn = 0;
        __syncthreads();
    }
    // partial list and count of this split, then the ticket: the last split CTA of the query merges all of them
    if (lane == 0 && my_cnt) atomicAdd(&s_cnt, my_cnt);
    unsigned long long* mine = part + ((size_t)split * B + b) * RK;
    for (int i = tid; i < K; i += 256) mine[i] = s_top[cur][i];
    __syncthreads();
    if (tid == 0) part_cnt[(size_t)split * B + b] = s_cnt;
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(&ticket[b], 1) == WSPLIT - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (int s = 0; s < WSPLIT; ++s) {
        if (s == split) continue;
        const unsigned long long* other = part + ((size_t)s * B + b) * RK;
        for (int i = tid; i < K; i += 256) s_new[i] = __ldcg(other + i);
        __syncthreads();
        merge_topk(s_top[cur], K, s_new, K, s_top[cur ^ 1]);
        cur ^= 1;
    }
    for (int r = tid; r < K; r += 256) {
        const unsigned long long key = s_top[cur][r];
        out_ids[(size_t)b * K + r] = key == KEY_NONE ? -1 : (int)(uint32_t)key;
        out_scores[(size_t)b * K + r] = key == KEY_NONE ? -INFINITY : key_value(~(uint32_t)(key >> 32));
    }
    if (tid == 0) {
        if (rescored) {
            int t = 0;
            for (int s = 0; s < WSPLIT; ++s) t += __ldcg(part_cnt + (size_t)s * B + b);
            rescored[b] = t;
        }
        ticket[b] = 0;
    }
}

}  // namespace tcar

using namespace tcar;
#define STREAM static_cast<cudaStream_t>(stream)

extern "C" int tcar_eval_topk(const float* chunkmax, const float* tilemax, const float* a_ic, const float* Tq,
                              const float* item,
                              const float* content, const int32_t* mwdhm, const int32_t* label, int32_t* top_ids,
                              float* top_scores, int32_t* n_greater, int B, int N, int n_pad, int item_offset,
                              void* stream) {
    return tcar_eval_topk_certified(chunkmax, tilemax, a_ic, Tq, item, content, mwdhm, label, top_ids, top_scores,
                                    n_greater, B, N, n_pad, item_offset, nullptr, nullptr, nullptr, stream);
}

extern "C" int tcar_eval_topk_certified(const float* chunkmax, const float* tilemax, const float* a_ic, const float* Tq,
                                        const float* item, const float* content, const int32_t* mwdhm,
                                        const int32_t* label, int32_t* top_ids, float* top_scores, int32_t* n_greater,
                                        int B, int N, int n_pad, int item_offset, const float* cat_stats,
                                        int32_t* uncertain, float* tau, void* stream) {
    if (B < 1 || B > TCAR_QROWS || N < 1 || n_pad < N || !tilemax) return TCAR_ERR_ARG;
    if (cat_stats && (!uncertain || !tau || (N + 127) / 128 > TCAR_MAX_EVAL_TILES)) return TCAR_ERR_ARG;
    launch_pdl(eval_topk_kernel, dim3(B), dim3(256), 0, STREAM, chunkmax, tilemax, a_ic, Tq, item, content, mwdhm,
               label, top_ids, top_scores, n_greater, N, n_pad, item_offset, cat_stats, uncertain, tau, SelIO{});
    return (int)cudaGetLastError();
}

extern "C" int tcar_eval_select(const float* chunkmax, const float* tilemax, float* sel_vals, int32_t* sel_ids, int B,
                                int N, int n_pad, int item_offset, void* stream) {
    if (B < 1 || B > TCAR_QROWS || N < 1 || n_pad < N || !chunkmax || !tilemax || !sel_vals || !sel_ids ||
        item_offset % CH)
        return TCAR_ERR_ARG;
    launch_pdl(eval_select_warp_kernel, dim3((B + 7) / 8), dim3(256), 0, STREAM, chunkmax, tilemax, sel_vals, sel_ids,
               B, N, n_pad, item_offset / CH, SelGroups{});
    return (int)cudaGetLastError();
}

extern "C" int tcar_eval_rescore(const float* sel_vals, const int32_t* sel_ids, int lists, long long list_stride,
                                 const float* a_ic, const float* Tq, const float* item, const float* content,
                                 const int32_t* mwdhm, const int32_t* label, int32_t* top_ids, float* top_scores,
                                 int32_t* n_greater, int B, int N_total, const float* cat_stats, int32_t* uncertain,
                                 float* tau, void* stream) {
    if (B < 1 || B > TCAR_QROWS || N_total < 1 || !sel_vals || !sel_ids || lists < 1 || lists * NSEL > NCC ||
        list_stride < (long long)B * NSEL || !cat_stats || !uncertain || !tau)
        return TCAR_ERR_ARG;
    SelIO io = {};
    io.in_vals = sel_vals;
    io.in_ids = sel_ids;
    io.in_lists = lists;
    io.in_stride = list_stride;
    launch_pdl(eval_topk_kernel, dim3(B), dim3(256), 0, STREAM, static_cast<const float*>(nullptr),
               static_cast<const float*>(nullptr), a_ic, Tq, item, content, mwdhm, label, top_ids, top_scores,
               n_greater, N_total, 0, 0, cat_stats, uncertain, tau, io);
    return (int)cudaGetLastError();
}

static int launch_widen(const float* chunkmax, const float* tilemax, const float* a_ic, const float* Tq,
                        const float* item, const float* content, const int32_t* mwdhm, const int32_t* label,
                        const int32_t* uncertain, const float* tau, int32_t* top_ids, float* top_scores,
                        int32_t* n_greater, int B, int N, int n_pad, int item_offset, void* workspace,
                        const WidenGroups& wg, void* stream) {
    // workspace per group: ids [S][512][20] | scores [S][512][20] | counts [S][512] (rows of a launch use its own B)
    int32_t* w = static_cast<int32_t*>(workspace);
    const int groups = wg.groups > 0 ? wg.groups : 1;
    launch_pdl(eval_topk_widen_kernel, dim3(B < WIDEN_SLOTS ? B : WIDEN_SLOTS, WSPLIT, groups), dim3(256), 0, STREAM,
               chunkmax, tilemax, a_ic, Tq, item, content, mwdhm, label, uncertain, tau, w, top_ids, top_scores,
               n_greater, N, n_pad, item_offset, B, wg);
    return (int)cudaGetLastError();
}

extern "C" long long tcar_eval_topk_widen_ws_bytes(int groups) {
    return (long long)(groups > 0 ? groups : 1) * W_GROUP_WORDS * 4;
}

extern "C" int tcar_eval_topk_widen(const float* chunkmax, const float* tilemax, const float* a_ic, const float* Tq,
                                    const float* item, const float* content, const int32_t* mwdhm,
                                    const int32_t* label, const int32_t* uncertain, const float* tau,
                                    int32_t* top_ids, float* top_scores, int32_t* n_greater, int B, int N, int n_pad,
                                    int item_offset, void* workspace, void* stream) {
    if (B < 1 || B > TCAR_QROWS || N < 1 || n_pad < N || !tilemax || !uncertain || !tau || !workspace)
        return TCAR_ERR_ARG;
    return launch_widen(chunkmax, tilemax, a_ic, Tq, item, content, mwdhm, label, uncertain, tau, top_ids, top_scores,
                        n_greater, B, N, n_pad, item_offset, workspace, WidenGroups{}, stream);
}

// The widening pass for the session groups of a catalog-sharded evaluation round in one launch pair: group g (n_rows[g]
// queries) has its chunk / tile maxima cm_stride / tm_stride floats apart, its a_ic / Tq / label planes q_stride words
// apart (one exchange block per group), its (uncertain, tau) vectors flag_stride words apart and its result planes
// (top_ids / top_scores / n_greater) out_stride words apart.  workspace: tcar_eval_topk_widen_ws_bytes(groups).
extern "C" int tcar_eval_topk_widen_groups(const float* chunkmax, long long cm_stride, const float* tilemax,
                                           long long tm_stride, const float* a_ic, const float* Tq,
                                           const int32_t* label, long long q_stride, const float* item,
                                           const float* content, const int32_t* mwdhm, const int32_t* uncertain,
                                           const float* tau, long long flag_stride, int32_t* top_ids,
                                           float* top_scores, int32_t* n_greater, long long out_stride,
                                           const int* n_rows, int groups, int N, int n_pad, int item_offset,
                                           void* workspace, void* stream) {
    if (!n_rows || groups < 1 || groups > TCAR_MAX_PEERS || N < 1 || n_pad < N || !tilemax || !uncertain || !tau ||
        !workspace)
        return TCAR_ERR_ARG;
    WidenGroups wg = {};
    wg.groups = groups;
    int bmax = 0;
    for (int g = 0; g < groups; ++g) {
        if (n_rows[g] > TCAR_QROWS) return TCAR_ERR_ARG;
        wg.n[g] = n_rows[g] > 0 ? n_rows[g] : 0;
        if (wg.n[g] > bmax) bmax = wg.n[g];
    }
    if (bmax == 0) return 0;
    wg.cm_gs = cm_stride;
    wg.tm_gs = tm_stride;
    wg.q_gs = q_stride;
    wg.flag_gs = flag_stride;
    wg.out_gs = out_stride;
    return launch_widen(chunkmax, tilemax, a_ic, Tq, item, content, mwdhm, label, uncertain, tau, top_ids, top_scores,
                        n_greater, bmax, N, n_pad, item_offset, workspace, wg, stream);
}

// tcar_eval_select for several session groups in one launch (see tcar_eval_topk_widen_groups for the strides).
extern "C" int tcar_eval_select_groups(const float* chunkmax, long long cm_stride, const float* tilemax,
                                       long long tm_stride, float* sel_vals, int32_t* sel_ids, long long out_stride,
                                       const int* n_rows, int groups, int N, int n_pad, int item_offset, void* stream) {
    if (!n_rows || groups < 1 || groups > TCAR_MAX_PEERS || N < 1 || n_pad < N || !chunkmax || !tilemax || !sel_vals ||
        !sel_ids || item_offset % CH)
        return TCAR_ERR_ARG;
    SelGroups sg = {};
    sg.groups = groups;
    int bmax = 0;
    for (int g = 0; g < groups; ++g) {
        if (n_rows[g] > TCAR_QROWS) return TCAR_ERR_ARG;
        sg.n[g] = n_rows[g] > 0 ? n_rows[g] : 0;
        if (sg.n[g] > bmax) bmax = sg.n[g];
    }
    if (bmax == 0) return 0;
    sg.cm_gs = cm_stride;
    sg.tm_gs = tm_stride;
    sg.out_gs = out_stride;
    launch_pdl(eval_select_warp_kernel, dim3((bmax + 7) / 8, groups), dim3(256), 0, STREAM, chunkmax, tilemax, sel_vals,
               sel_ids, bmax, N, n_pad, item_offset / CH, sg);
    return (int)cudaGetLastError();
}

extern "C" int tcar_catalog_stats(const float* item, const float* content, int row_lo, int row_hi, float* out2,
                                  void* stream) {
    if (row_lo < 0 || row_hi <= row_lo || !out2) return TCAR_ERR_ARG;
    cudaError_t e = cudaMemsetAsync(out2, 0, 2 * sizeof(float), STREAM);
    if (e != cudaSuccess) return (int)e;
    launch_pdl(catalog_stats_kernel, dim3(148 * 8), dim3(256), 0, STREAM, item, content, row_lo, row_hi, out2);
    return (int)cudaGetLastError();
}

extern "C" int tcar_topk_merge(const int32_t* ids, const float* scores, int32_t* out_ids, float* out_scores, int G,
                               int B, void* stream) {
    if (G < 1 || G > TCAR_MAX_PEERS || B < 1) return TCAR_ERR_ARG;
    launch_pdl(topk_merge_kernel, dim3((B + 7) / 8), dim3(256), 0, STREAM, ids, scores, out_ids, out_scores, G, B,
               0LL, static_cast<const int32_t*>(nullptr), static_cast<const float*>(nullptr),
               static_cast<const float*>(nullptr), static_cast<int32_t*>(nullptr), static_cast<float*>(nullptr),
               static_cast<const int32_t*>(nullptr), WidenGroups{});
    return (int)cudaGetLastError();
}

// cross loss of B queries from G item ranges' softmax partial sums, each relative to its own exponent shift
__global__ void __launch_bounds__(256)
ce_combine_kernel(const float* __restrict__ sumexp, const float* __restrict__ rowmax, long long gstride,
                  float* __restrict__ out_ce, int G, int B) {
    PDL_ENTER();
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    float M = 0.f;
    for (int g = 0; g < G; ++g) {
        const float r = rowmax[g * gstride + b];
        M = fmaxf(M, r > TCAR_EXP_LIMIT2 ? r : 0.f);
    }
    float tot = 0.f;
    for (int g = 0; g < G; ++g) {
        const float r = rowmax[g * gstride + b];
        tot += sumexp[g * gstride + b] * exp2f((r > TCAR_EXP_LIMIT2 ? r : 0.f) - M);
    }
    out_ce[b] = fmaf(M, 0.6931471805599453f, logf(tot));
}

extern "C" int tcar_eval_ce_combine(const float* sumexp, const float* rowmax, long long gstride, float* out_ce, int G,
                                    int B, void* stream) {
    if (G < 1 || G > TCAR_MAX_PEERS || B < 1 || !sumexp || !rowmax || !out_ce) return TCAR_ERR_ARG;
    launch_pdl(ce_combine_kernel, dim3((B + 255) / 256), dim3(256), 0, STREAM, sumexp, rowmax, gstride, out_ce, G, B);
    return (int)cudaGetLastError();
}

extern "C" int tcar_eval_merge_flagged(const void* blocks, long long block_words, const int32_t* only_if,
                                       int32_t* out_ids, float* out_scores, int32_t* out_ngt, int G, int B,
                                       void* stream) {
    if (G < 1 || G > TCAR_MAX_PEERS || B < 1 || B > TCAR_QROWS || block_words < TCAR_EVAL_BLOCK_WORDS || !blocks ||
        !only_if)
        return TCAR_ERR_ARG;
    const float* f = static_cast<const float*>(blocks);
    const int32_t* i = static_cast<const int32_t*>(blocks);
    launch_pdl(topk_merge_kernel, dim3((B + 7) / 8), dim3(256), 0, STREAM, i + TCAR_EVAL_OFF_IDS, f + TCAR_EVAL_OFF_SCORES,
               out_ids, out_scores, G, B, block_words, i + TCAR_EVAL_OFF_NGT, static_cast<const float*>(nullptr),
               static_cast<const float*>(nullptr), out_ngt, static_cast<float*>(nullptr), only_if, WidenGroups{});
    return (int)cudaGetLastError();
}

extern "C" int tcar_rerank(const float* a_ic, const float* Tq, const float* item, const float* content,
                           const int32_t* mwdhm, const int32_t* cand_off, const int32_t* cand_ids, const int32_t* label,
                           int B, int N, int max_len, float* scores, int32_t* ranked, int32_t* label_rank, float* auc,
                           void* stream) {
    if (B < 0 || B > TCAR_QROWS || N <= 0 || max_len < 0 || max_len > TCAR_RERANK_MAXL || !a_ic || !Tq || !item ||
        !content || !mwdhm || !cand_off || (label && (!label_rank || !auc)))
        return TCAR_ERR_ARG;
    if (B == 0) return 0;
    launch_pdl(rerank_kernel, dim3(B), dim3(256), 0, STREAM, a_ic, Tq, item, content, mwdhm, cand_off, cand_ids, label,
               N, max_len, scores, ranked, label_rank, auc);
    return (int)cudaGetLastError();
}

extern "C" long long tcar_recommend_ws_bytes(int B) {
    if (B < 0 || B > TCAR_QROWS) return TCAR_ERR_ARG;
    return (long long)(rec_keys_offset(B) + (size_t)WSPLIT * B * RK * 8);
}

extern "C" int tcar_recommend(const float* chunkmax, const float* tilemax, const float* a_ic, const float* Tq,
                              const float* item, const float* content, const int32_t* mwdhm, const float* cat_stats,
                              const int32_t* x_off, const int32_t* x_ids, const int32_t* clicks, int T, int B, int N,
                              int n_pad, int K, void* workspace, int32_t* ids, float* scores, int32_t* rescored,
                              void* stream) {
    if (B < 0 || B > TCAR_QROWS || N < 1 || n_pad < N || n_pad % 128 || K < 1 || K > RK ||
        (clicks && (T < 1 || T > RX)) || !chunkmax || !tilemax || !a_ic || !Tq || !item || !content || !mwdhm ||
        !cat_stats || (x_off && !x_ids) || !workspace || !ids || !scores)
        return TCAR_ERR_ARG;
    if (B == 0) return 0;
    const int n_clicks = clicks ? T : 0;
    char* ws = static_cast<char*>(workspace);
    cudaError_t e = launch_pdl(recommend_select_kernel, dim3(B), dim3(256), 0, STREAM, chunkmax, tilemax, a_ic, Tq,
                               cat_stats, x_off, n_clicks, K, N, n_pad, reinterpret_cast<float*>(ws) + TCAR_QROWS);
    if (e != cudaSuccess) return (int)e;
    launch_pdl(recommend_scan_kernel, dim3(B, WSPLIT), dim3(256), 0, STREAM, chunkmax, tilemax, a_ic, Tq, item,
               content, mwdhm, x_off, x_ids, clicks, n_clicks, K, N, n_pad, B, ws, ids, scores, rescored);
    return (int)cudaGetLastError();
}

extern "C" int tcar_eval_merge(const void* blocks, long long block_words, int32_t* out_ids, float* out_scores,
                               int32_t* out_ngt, float* out_ce, int G, int B, void* stream) {
    if (G < 1 || G > TCAR_MAX_PEERS || B < 1 || B > TCAR_QROWS || block_words < TCAR_EVAL_BLOCK_WORDS || !blocks)
        return TCAR_ERR_ARG;
    const float* f = static_cast<const float*>(blocks);
    const int32_t* i = static_cast<const int32_t*>(blocks);
    launch_pdl(topk_merge_kernel, dim3((B + 7) / 8), dim3(256), 0, STREAM, i + TCAR_EVAL_OFF_IDS, f + TCAR_EVAL_OFF_SCORES,
               out_ids, out_scores, G, B, block_words, i + TCAR_EVAL_OFF_NGT, f + TCAR_EVAL_OFF_SUMEXP,
               f + TCAR_EVAL_OFF_ROWMAX, out_ngt, out_ce, static_cast<const int32_t*>(nullptr), WidenGroups{});
    return (int)cudaGetLastError();
}
