// Full-catalog scoring on 5th-gen tensor cores (tcgen05 + TMEM + TMA), sm_100a only.
//
// Replaces the reference's k9/k10/k13 call sites (model_combine.py:132-138 scoring matmul, :145 softmax CE,
// :283-301 eval scores) and the two scoring-matmul gradients TF derives from them (model_combine.py:156).
//
// Data layout (see DESIGN.md §3):
//   Q    [512, 640]  bf16  session operand  [a_ic(500) | T(139) | 0]      (T = a_pt . clip(time tables)^T)
//   Iext [Npad, 640] bf16  item operand     [item(250) | content(250) | onehot(139) | 0], rows >= N are zero
//   E    [Npad/8][512][8] bf16  exp(S - c_b), written by the forward kernel in train mode, read by both backward
//        GEMMs.  Logically E[b, n]; stored in blocks of 8 items so that the forward epilogue (thread <-> session
//        row, 8 items = one 16-byte store) writes 512 contiguous bytes per warp instruction instead of 32 scattered
//        16-byte pieces (23 M single-sector L2 write requests per call with the row-major layout).  The backward
//        kernels read it through a 3-D tensor map (8 items | session | item block) WITHOUT swizzle: a box lands in
//        shared memory as [item block][session][8 items], which is exactly UMMA's no-swizzle canonical layout
//        (8 x 16-byte core matrices) -- K-major for dQ (K = items), MN-major for dItem (K = sessions).
//
//   score_fwd   : S = Q . Iext^T, 128 sessions (TMEM lanes) x 128 items per tile, K = 640 resident in smem for Q,
//                 item tiles TMA-multicast across a cluster of CL CTAs (CL session tiles share every item tile).
//                 epilogue TRAIN: E = exp(S - c_b) -> bf16 store, per-(tile,row) partial sums of E
//                 epilogue EVAL : partial sums of E (for the CE "avg loss") + max over each 8 consecutive items
//   score_bwd_q : dQ[b,c]   = sum_n E[b,n] Iext[n,c]      (split over n, partials reduced by a second kernel)
//   score_bwd_i : dItem[n,c] = sum_b E[b,n] Qs[b,c]       (Qs = a_ic / sumexp_b in bf16, c < 256)
#include "sm100_ptx.cuh"
#include "tcar_b200.h"
#include "launch.cuh"
#include "decay.cuh"

namespace tcar {

constexpr int kThreads = 256;  // warp0 TMA, warp1 MMA, warp2 TMEM alloc, warp3 idle, warps4-7 epilogue
constexpr int BM = 128;
constexpr int BK = 64;
constexpr int KEXT = TCAR_KEXT;  // 640
constexpr int NKB = KEXT / BK;   // 10
constexpr int QROWS = TCAR_QROWS;  // 512
constexpr float kLog2e = 1.4426950408889634f;

// ------------------------------------------------------------------------------------------------ forward
constexpr int F_BN = 128;
constexpr int F_STAGES = 4;
constexpr int F_NACC = 4;
constexpr int F_A_BYTES = BM * KEXT * 2;        // 163840
constexpr int F_B_STAGE = F_BN * BK * 2;        // 16384
constexpr int F_SMEM = F_A_BYTES + F_STAGES * F_B_STAGE + 1024 /*align*/ + 256 /*barriers*/;

struct FwdParams {
    __nv_bfloat16* E;       // [512, e_pitch] (train) or nullptr
    float* rowsum_part;     // [n_tiles, 512]
    float* chunkmax;        // [512, e_pitch/8] (eval) or nullptr
    float* tilemax;         // [512, e_pitch/128] (eval, nullable): max of S over each 128 consecutive items
    const float* c_ref;     // [512] reference score per row (exp argument shift)
    float* rowmax_part;     // [n_tiles, 512] (nullable) max over the tile's valid items of the exponent argument
                            // (S - c_ref) * log2(e): pass 1 of the overflow guard (tcar_ce_finish reduces it)
    const float* rowmax;    // [512] (nullable) pass 2: per-row maxima found by pass 1.  Rows above TCAR_EXP_LIMIT2 are
                            // shifted by their maximum (TF's max-subtracted softmax, model_combine.py:145); CTAs none
                            // of whose rows need it exit at once, the others rewrite identical values for quiet rows
    int n_items;            // valid items N
    int n_tiles;            // ceil(Npad / F_BN)
    int n_rows;             // valid sessions B
    int e_pitch;            // Npad
    int groups;             // number of session groups (ceil(ceil(B/128)/CL))
    int mode;               // 0 = train, 1 = eval, 2 = eval with a publish-time window per row, 3 = eval with a
                            // freshness decay per row (2 and 3: pair kernel only)
    int prefetch;           // pair kernel: L2 prefetch distance of the streamed item operand in stages (0 = off)
    const int32_t* item_time;   // MODE 2: [e_pitch] time of every item
    const int32_t* win_lo;      // MODE 2: [512] window of every row: item n is in row b's window when
    const int32_t* win_hi;      //         win_lo[b] <= item_time[n] <= win_hi[b]; the others count as -inf
                                // MODE 3: item_time as MODE 2, win_lo / win_hi both null (no window) or as MODE 2
    const int32_t* t_ref;       // MODE 3: [512] request time of every row
    const float* rate;          // MODE 3: [512] decay rate of every row (decay.cuh)
};

// exponent shift of one session row in log2 units: the label score, plus -- in pass 2 of the overflow guard -- the
// row maximum found by pass 1 when that exceeded TCAR_EXP_LIMIT2
__device__ __forceinline__ float exp_shift(const FwdParams& p, uint32_t row) {
    float sh = p.c_ref[row] * kLog2e;
    if (p.rowmax) {
        const float m = p.rowmax[row];
        if (m > TCAR_EXP_LIMIT2) sh += m;
    }
    return sh;
}

// pass 2 of the overflow guard: does any of the `rows` session rows starting at row0 need the extra shift?  Called
// by every thread of the CTA (and with the same arguments by every CTA of a cluster, so that they agree).
__device__ __forceinline__ bool guard_pass_needed(const FwdParams& p, uint32_t row0, uint32_t rows) {
    bool need = false;
    for (uint32_t r = row0 + threadIdx.x; r < row0 + rows && r < (uint32_t)p.n_rows; r += blockDim.x)
        need |= p.rowmax[r] > TCAR_EXP_LIMIT2;
    return __syncthreads_or(need) != 0;
}

template <int CL>
__global__ void __launch_bounds__(kThreads, 1)
score_fwd_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_i,
                 const FwdParams p) {
    PDL_ENTER();
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + F_A_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_b + F_STAGES * F_B_STAGE);
    uint64_t* full = bars;                      // [F_STAGES]
    uint64_t* empty = bars + F_STAGES;          // [F_STAGES]
    uint64_t* acc_full = bars + 2 * F_STAGES;   // [F_NACC]
    uint64_t* acc_empty = acc_full + F_NACC;    // [F_NACC]
    uint64_t* a_full = acc_empty + F_NACC;      // [1]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_full + 1);

    const uint32_t warp = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    const uint32_t rank = (CL > 1) ? cluster_ctarank() : 0u;
    const uint32_t cluster_id = blockIdx.x / CL;
    const uint32_t n_clusters = gridDim.x / CL;
    // static schedule: cluster -> (session group, strided item tiles) so that Q stays resident
    const uint32_t grp = cluster_id % p.groups;
    const uint32_t tile0 = cluster_id / p.groups;
    const uint32_t tile_step = n_clusters / p.groups;
    const uint32_t mtile = grp * CL + rank;
    const uint32_t my_tiles =
        tile0 < (uint32_t)p.n_tiles ? ((uint32_t)p.n_tiles - tile0 + tile_step - 1) / tile_step : 0u;
    if (p.rowmax && !guard_pass_needed(p, grp * CL * BM, CL * BM)) return;

    if (warp == 0 && elect_one()) {
        tma_prefetch_desc(&map_q);
        tma_prefetch_desc(&map_i);
    }
    if (warp == 1 && elect_one()) {
        for (int i = 0; i < F_STAGES; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], CL);
        }
        for (int i = 0; i < F_NACC; ++i) {
            mbar_init(&acc_full[i], 1);
            mbar_init(&acc_empty[i], 4);
        }
        mbar_init(a_full, 1);
        fence_mbar_init();
    }
    if (warp == 2) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    if (CL > 1) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= TMA producer =================
        if (elect_one()) {
            mbar_expect_tx(a_full, F_A_BYTES);
            for (int kb = 0; kb < NKB; ++kb)
                tma_load_2d(smem_a + kb * (BM * BK * 2), &map_q, a_full, kb * BK, mtile * BM);
            uint32_t stage = 0, phase = 0;
            for (uint32_t it = 0; it < my_tiles; ++it) {
                const int n0 = (tile0 + it * tile_step) * F_BN;
                for (int kb = 0; kb < NKB; ++kb) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    mbar_expect_tx(&full[stage], F_B_STAGE);
                    uint8_t* dst = smem_b + stage * F_B_STAGE + rank * (F_B_STAGE / CL);
                    if (CL > 1)
                        tma_load_2d_mcast(dst, &map_i, &full[stage], kb * BK, n0 + rank * (F_BN / CL),
                                          (uint16_t)((1u << CL) - 1));
                    else
                        tma_load_2d(dst, &map_i, &full[stage], kb * BK, n0);
                    if (++stage == F_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        constexpr uint32_t idesc = make_idesc_bf16(BM, F_BN, 0, 0);
        mbar_wait(a_full, 0);
        tc_fence_after();
        uint32_t stage = 0, phase = 0;
        for (uint32_t it = 0; it < my_tiles; ++it) {
            const uint32_t acc = it % F_NACC;
            const uint32_t acc_phase = (it / F_NACC) & 1;
            mbar_wait(&acc_empty[acc], acc_phase ^ 1);
            tc_fence_after();
            for (int kb = 0; kb < NKB; ++kb) {
                mbar_wait(&full[stage], phase);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t a_addr = smem_u32(smem_a + kb * (BM * BK * 2));
                    const uint32_t b_addr = smem_u32(smem_b + stage * F_B_STAGE);
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k)
                        umma_bf16(tmem_base + acc * F_BN, sdesc_kmajor(a_addr + k * 32), sdesc_kmajor(b_addr + k * 32),
                                  idesc, (kb | k) != 0);
                    if (CL > 1) umma_commit_mcast(&empty[stage], (uint16_t)((1u << CL) - 1));
                    else umma_commit(&empty[stage]);
                    if (kb == NKB - 1) umma_commit(&acc_full[acc]);
                }
                __syncwarp();
                if (++stage == F_STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp >= 4) {
        // ================= epilogue: thread <-> session row =================
        const uint32_t q = warp - 4;
        const uint32_t row = mtile * BM + q * 32 + lane;
        const bool row_ok = row < (uint32_t)p.n_rows;
        // rows in [B, round_up(B,64)) are stored as zeros: they are K-padding of the dItem GEMM
        const bool store_ok = row < (((uint32_t)p.n_rows + 63u) & ~63u);
        const float cshift = row_ok ? exp_shift(p, row) : 0.f;
        for (uint32_t it = 0; it < my_tiles; ++it) {
            const uint32_t acc = it % F_NACC;
            const uint32_t acc_phase = (it / F_NACC) & 1;
            const uint32_t tile = tile0 + it * tile_step;
            const int n0 = tile * F_BN;
            mbar_wait(&acc_full[acc], acc_phase);
            tc_fence_after();
            float psum = 0.f, tmax = -INFINITY, amax = -INFINITY;
            const bool tail = n0 + F_BN > p.n_items;
#pragma unroll 1
            for (int ch = 0; ch < F_BN / 32; ++ch) {
                uint32_t v[32];
                tmem_ld32(tmem_base + ((q * 32) << 16) + acc * F_BN + ch * 32, v);
                tmem_ld_wait();
                const int nb = n0 + ch * 32;
                float e[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float s = __uint_as_float(v[j]);
                    const float arg = fmaf(s, kLog2e, -cshift);
                    float ex = exp2f(arg);
                    if (!row_ok || (tail && nb + j >= p.n_items)) ex = 0.f;
                    else amax = fmaxf(amax, arg);
                    e[j] = ex;
                    psum += ex;
                }
                if (p.mode == 0) {
                  if (store_ok) {
                    uint4* dst = reinterpret_cast<uint4*>(p.E) + (size_t)(nb >> 3) * QROWS + row;
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        uint4 o;
                        o.x = pack_bf16(e[g * 8 + 0], e[g * 8 + 1]);
                        o.y = pack_bf16(e[g * 8 + 2], e[g * 8 + 3]);
                        o.z = pack_bf16(e[g * 8 + 4], e[g * 8 + 5]);
                        o.w = pack_bf16(e[g * 8 + 6], e[g * 8 + 7]);
                        dst[(size_t)g * QROWS] = o;
                    }
                  }
                } else {
                    float4 m;
                    float* mm = reinterpret_cast<float*>(&m);
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        float mx = -INFINITY;
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float s = __uint_as_float(v[g * 8 + j]);
                            const bool ok = !(tail && nb + g * 8 + j >= p.n_items);
                            mx = ok ? fmaxf(mx, s) : mx;
                        }
                        mm[g] = mx;
                        tmax = fmaxf(tmax, mx);
                    }
                    if (row_ok)
                        *reinterpret_cast<float4*>(p.chunkmax + (size_t)row * (p.e_pitch / 8) + nb / 8) = m;
                }
            }
            // all TMEM reads of this accumulator are complete -> hand it back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[acc]);
            if (row_ok) p.rowsum_part[(size_t)tile * QROWS + row] = psum;
            if (row_ok && p.rowmax_part) p.rowmax_part[(size_t)tile * QROWS + row] = amax;
            if (row_ok && p.mode == 1 && p.tilemax) p.tilemax[(size_t)row * (p.e_pitch / 128) + tile] = tmax;
        }
    }

    tc_fence_before();
    if (CL > 1) cluster_sync_all(); else __syncthreads();
    if (warp == 2) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------ forward, CTA pair
// Same contract as score_fwd_kernel, restructured for pipeline depth: the 160 KB resident session operand leaves
// only 64 KB of shared memory for the streamed item operand, which is ~0.5 us of MMA work per SM with 128-item
// tiles -- less than the TMA round trip under load.  Here two CTAs (one TPC) issue tcgen05.mma.cta_group::2 with
// M = 256 sessions x N = 256 items: each CTA keeps its own 128 session rows resident and streams only HALF of every
// item tile (128 items x 64 k = 16 KB per stage), so the same 64 KB hold 4 x 512 = 2048 clks of MMA work and each
// SM ingests half the bytes per FLOP.  Two 256-column accumulators fill TMEM (double buffered); 8 epilogue warps
// (2 per 32-lane TMEM quarter, 128 columns each) run exp / bf16-pack / partial row sums under the next tile's MMAs.
constexpr int P_THREADS = 384;   // warp0 TMA, warp1 MMA (leader CTA only), warp2 TMEM alloc, warp3 idle, warps4-11 epilogue
constexpr int P_BN = 256;        // items per tile (both CTAs)
constexpr int P_HALF = 128;      // items per CTA per tile
constexpr int P_STAGES = 4;
constexpr int P_NACC = 2;
constexpr int P_B_STAGE = P_HALF * BK * 2;      // 16384
constexpr int P_SMEM = F_A_BYTES + P_STAGES * P_B_STAGE + 1024 /*align*/ + 256 /*barriers*/;

// TAIL = false: every item of the chunk exists (all tiles but the last one or two) -- no per-element bounds logic, which
// was half of the epilogue's instructions (2 ISETP + 2 PLOP3 + FSEL per element beside FFMA / MUFU / FMNMX / FADD).
// MODE 2 (eval with a window): an item outside the row's window gets the score -inf before anything reads it, so it adds
// exp(-inf) = 0 to the partial sum and nothing to the chunk / tile maxima, exactly like an item >= N.  The row's window
// arrives as wlo = win_lo and wspan = win_hi - win_lo (uint32: t is inside iff t - wlo <= wspan, one IADD + one ISETP),
// wempty = win_lo > win_hi.  The chunk's 32 item times are the same for every lane: eight warp-uniform 16-byte loads.
template <int MODE, bool TAIL>
__device__ __forceinline__ void fwd_epilogue_chunk_t(const uint32_t (&v)[32], const FwdParams& p, float cshift,
                                                     bool row_ok, bool store_ok, uint32_t row, int nb,
                                                     float& psum, float& tmax, float& amax, uint32_t wlo = 0,
                                                     uint32_t wspan = 0, bool wempty = false) {
    constexpr bool tail = TAIL;
    float e[32];
    float sm[32];                                            // MODE 2: the masked scores
    if (MODE == 2) {
        const int4* tp = reinterpret_cast<const int4*>(p.item_time + nb);
#pragma unroll
        for (int g = 0; g < 8; ++g) {
            const int4 t = __ldg(tp + g);
            const int tv[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const bool out = wempty || (uint32_t)tv[c] - wlo > wspan;
                sm[g * 4 + c] = out ? -INFINITY : __uint_as_float(v[g * 4 + c]);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        const float arg = fmaf(MODE == 2 ? sm[j] : __uint_as_float(v[j]), kLog2e, -cshift);
        float ex = ex2_approx(arg);
        if (TAIL) {
            if (!row_ok || nb + j >= p.n_items) ex = 0.f;
            else if (MODE == 0) amax = fmaxf(amax, arg);     // eval mode derives it from tmax (monotone map)
        } else {
            ex = row_ok ? ex : 0.f;
            if (MODE == 0) amax = fmaxf(amax, arg);          // rows beyond the batch never store it
        }
        e[j] = ex;
        psum += ex;
    }
    if (MODE == 0) {
        if (store_ok) {
            // block-of-8-items layout: the 32 lanes (consecutive session rows) of one store are contiguous
            uint4* dst = reinterpret_cast<uint4*>(p.E) + (size_t)(nb >> 3) * QROWS + row;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                uint4 o;
                o.x = pack_bf16(e[g * 8 + 0], e[g * 8 + 1]);
                o.y = pack_bf16(e[g * 8 + 2], e[g * 8 + 3]);
                o.z = pack_bf16(e[g * 8 + 4], e[g * 8 + 5]);
                o.w = pack_bf16(e[g * 8 + 6], e[g * 8 + 7]);
                dst[(size_t)g * QROWS] = o;
            }
        }
    } else {
        float4 m;
        float* mm = reinterpret_cast<float*>(&m);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            float mx = -INFINITY;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float sv = MODE == 2 ? sm[g * 8 + j] : __uint_as_float(v[g * 8 + j]);
                const bool ok = !(tail && nb + g * 8 + j >= p.n_items);
                mx = ok ? fmaxf(mx, sv) : mx;
            }
            mm[g] = mx;
            tmax = fmaxf(tmax, mx);
        }
        if (row_ok) *reinterpret_cast<float4*>(p.chunkmax + (size_t)row * (p.e_pitch / 8) + nb / 8) = m;
    }
}

template <int MODE>
__device__ __forceinline__ void fwd_epilogue_chunk(const uint32_t (&v)[32], const FwdParams& p, float cshift,
                                                   bool row_ok, bool store_ok, bool tail, uint32_t row, int nb,
                                                   float& psum, float& tmax, float& amax, uint32_t wlo = 0,
                                                   uint32_t wspan = 0, bool wempty = false) {
    if (tail)
        fwd_epilogue_chunk_t<MODE, true>(v, p, cshift, row_ok, store_ok, row, nb, psum, tmax, amax, wlo, wspan, wempty);
    else
        fwd_epilogue_chunk_t<MODE, false>(v, p, cshift, row_ok, store_ok, row, nb, psum, tmax, amax, wlo, wspan, wempty);
}

// MODE 3 (eval with a freshness decay, DESIGN §4.10): the chunk maxima (and the running tile maximum) of the decayed
// scores r = decayed(s, d, t) of one row's 32 items nb .. nb+31; items >= N and items outside the row's window (wlo /
// wspan / wempty as MODE 2; wspan = ~0 without a window) count as -inf.  No exp and no partial sums.  t = the 32 item
// times, loaded by the caller before the tcgen05.wait::ld of these scores (load_times).
__device__ __forceinline__ void load_times(const FwdParams& p, int nb, int4 (&t)[8]) {
    const int4* tp = reinterpret_cast<const int4*>(p.item_time + nb);
#pragma unroll
    for (int g = 0; g < 8; ++g) t[g] = __ldg(tp + g);
}

template <bool TAIL>
__device__ __forceinline__ void fwd_decay_chunk_t(const uint32_t (&v)[32], const int4 (&t)[8], const FwdParams& p,
                                                  const DecayRow& d, uint32_t wlo, uint32_t wspan, bool wempty,
                                                  bool row_ok, uint32_t row, int nb, float& tmax) {
    float4 m;
    float* mm = reinterpret_cast<float*>(&m);
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        float mx = -INFINITY;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int k = g * 8 + j;
            const int4 tq = t[k / 4];
            const int32_t tv = k % 4 == 0 ? tq.x : k % 4 == 1 ? tq.y : k % 4 == 2 ? tq.z : tq.w;
            const bool ok = !wempty && (uint32_t)tv - wlo <= wspan && !(TAIL && nb + k >= p.n_items);
            mx = ok ? fmaxf(mx, decayed(__uint_as_float(v[k]), d, tv)) : mx;
        }
        mm[g] = mx;
        tmax = fmaxf(tmax, mx);
    }
    if (row_ok) *reinterpret_cast<float4*>(p.chunkmax + (size_t)row * (p.e_pitch / 8) + nb / 8) = m;
}

__device__ __forceinline__ void fwd_decay_chunk(const uint32_t (&v)[32], const int4 (&t)[8], const FwdParams& p,
                                                const DecayRow& d, uint32_t wlo, uint32_t wspan, bool wempty,
                                                bool row_ok, bool tail, uint32_t row, int nb, float& tmax) {
    if (tail) fwd_decay_chunk_t<true>(v, t, p, d, wlo, wspan, wempty, row_ok, row, nb, tmax);
    else fwd_decay_chunk_t<false>(v, t, p, d, wlo, wspan, wempty, row_ok, row, nb, tmax);
}

template <int MODE>
__global__ void __launch_bounds__(P_THREADS, 1)
score_fwd_pair_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_i,
                      const FwdParams p) {
    PDL_ENTER();
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + F_A_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_b + P_STAGES * P_B_STAGE);
    uint64_t* full = bars;                      // [P_STAGES]  used in the leader CTA (tx from both CTAs' loads)
    uint64_t* empty = bars + P_STAGES;          // [P_STAGES]  one per CTA, MMA commit multicast
    uint64_t* acc_full = bars + 2 * P_STAGES;   // [P_NACC]    one per CTA, MMA commit multicast
    uint64_t* acc_empty = acc_full + P_NACC;    // [P_NACC]    used in the leader CTA, 16 epilogue-warp arrivals
    uint64_t* a_full = acc_empty + P_NACC;      // [1]         leader CTA
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_full + 1);

    const uint32_t warp = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    const uint32_t rank = cluster_ctarank();    // 0 = leader
    const uint32_t pair_id = blockIdx.x >> 1;
    const uint32_t n_pairs = gridDim.x >> 1;
    const uint32_t grp = pair_id % p.groups;
    const uint32_t tile0 = pair_id / p.groups;
    const uint32_t tile_step = n_pairs / p.groups;
    const uint32_t mtile = grp * 2 + rank;
    const uint32_t my_tiles =
        tile0 < (uint32_t)p.n_tiles ? ((uint32_t)p.n_tiles - tile0 + tile_step - 1) / tile_step : 0u;
    if (p.rowmax && !guard_pass_needed(p, grp * 2 * BM, 2 * BM)) return;      // both CTAs of the pair decide alike

    if (warp == 0 && elect_one()) {
        tma_prefetch_desc(&map_q);
        tma_prefetch_desc(&map_i);
    }
    if (warp == 1 && elect_one()) {
        for (int i = 0; i < P_STAGES; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], 1);
        }
        for (int i = 0; i < P_NACC; ++i) {
            mbar_init(&acc_full[i], 1);
            mbar_init(&acc_empty[i], 16);
        }
        mbar_init(a_full, 1);
        fence_mbar_init();
    }
    if (warp == 2) tmem_alloc_pair(tmem_slot, 512);
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= TMA producer (both CTAs; completion bytes land on the LEADER's barriers) =================
        if (elect_one()) {
            const uint32_t a_full_l = mapa_u32(a_full, 0);
            if (rank == 0) mbar_expect_tx(a_full, 2 * F_A_BYTES);
            for (int kb = 0; kb < NKB; ++kb)
                tma_load_2d_pair(smem_a + kb * (BM * BK * 2), &map_q, a_full_l, kb * BK, mtile * BM);
            uint32_t stage = 0, phase = 0;
            // L2 prefetch `pf` stages ahead of the loads (same boxes, same order)
            const uint32_t pf = (uint32_t)p.prefetch, total = my_tiles * NKB;
            auto prefetch_stage = [&](uint32_t s) {
                if (s < total) {
                    const uint32_t pit = s / NKB, pkb = s - pit * NKB;
                    tma_prefetch_2d(&map_i, pkb * BK, (tile0 + pit * tile_step) * P_BN + rank * P_HALF);
                }
            };
            for (uint32_t s = 0; s < pf; ++s) prefetch_stage(s);
            uint32_t sidx = 0;
            for (uint32_t it = 0; it < my_tiles; ++it) {
                const int n0 = (tile0 + it * tile_step) * P_BN + rank * P_HALF;
                for (int kb = 0; kb < NKB; ++kb, ++sidx) {
                    if (pf) prefetch_stage(sidx + pf);
                    mbar_wait(&empty[stage], phase ^ 1);
                    if (rank == 0) mbar_expect_tx(&full[stage], 2 * P_B_STAGE);
                    tma_load_2d_pair(smem_b + stage * P_B_STAGE, &map_i, mapa_u32(&full[stage], 0), kb * BK, n0);
                    if (++stage == P_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer (leader CTA only) =================
        if (rank == 0) {
            constexpr uint32_t idesc = make_idesc_bf16(2 * BM, P_BN, 0, 0);
            mbar_wait(a_full, 0);
            tc_fence_after();
            uint32_t stage = 0, phase = 0;
            for (uint32_t it = 0; it < my_tiles; ++it) {
                const uint32_t acc = it % P_NACC;
                const uint32_t acc_phase = (it / P_NACC) & 1;
                mbar_wait(&acc_empty[acc], acc_phase ^ 1);
                tc_fence_after();
                for (int kb = 0; kb < NKB; ++kb) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    if (elect_one()) {
                        const uint32_t a_addr = smem_u32(smem_a + kb * (BM * BK * 2));
                        const uint32_t b_addr = smem_u32(smem_b + stage * P_B_STAGE);
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k)
                            umma_bf16_pair(tmem_base + acc * P_BN, sdesc_kmajor(a_addr + k * 32),
                                           sdesc_kmajor(b_addr + k * 32), idesc, (kb | k) != 0);
                        umma_commit_pair(&empty[stage], 3);
                        if (kb == NKB - 1) umma_commit_pair(&acc_full[acc], 3);
                    }
                    __syncwarp();
                    if (++stage == P_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (MODE == 3 && warp >= 4) {
        // ================= epilogue of the decayed maxima: the TMEM walk of the epilogue below =================
        const uint32_t e = warp - 4;
        const uint32_t q = e & 3, h = e >> 2;
        const uint32_t row = mtile * BM + q * 32 + lane;
        const bool row_ok = row < (uint32_t)p.n_rows;
        DecayRow d = decay_row(0, 0.f);
        uint32_t wlo = 0, wspan = ~0u;
        bool wempty = false;
        if (row_ok) {                               // the row's decay and window, loaded once
            d = decay_row(p.t_ref[row], p.rate[row]);
            if (p.win_lo) {
                const int32_t lo = p.win_lo[row], hi = p.win_hi[row];
                wlo = (uint32_t)lo;
                wspan = (uint32_t)hi - (uint32_t)lo;
                wempty = lo > hi;
            }
        }
        const uint32_t acc_empty_l = mapa_u32(acc_empty, 0);
        for (uint32_t it = 0; it < my_tiles; ++it) {
            const uint32_t acc = it % P_NACC;
            const uint32_t acc_phase = (it / P_NACC) & 1;
            const uint32_t tile = tile0 + it * tile_step;
            const int n0 = tile * P_BN + h * 128;
            mbar_wait(&acc_full[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((q * 32) << 16) + acc * P_BN + h * 128;
            const bool tail = n0 + 128 > p.n_items;
            float tmax = -INFINITY;
            uint32_t va[32], vb[32];
            int4 ta[8], tb[8];
            // each chunk's item times are requested before the wait for its scores
            tmem_ld32(taddr, va);
            load_times(p, n0, ta);
            tmem_ld_wait();
            tmem_ld32(taddr + 32, vb);
            load_times(p, n0 + 32, tb);
            fwd_decay_chunk(va, ta, p, d, wlo, wspan, wempty, row_ok, tail, row, n0, tmax);
            tmem_ld_wait();
            tmem_ld32(taddr + 64, va);
            load_times(p, n0 + 64, ta);
            fwd_decay_chunk(vb, tb, p, d, wlo, wspan, wempty, row_ok, tail, row, n0 + 32, tmax);
            tmem_ld_wait();
            tmem_ld32(taddr + 96, vb);
            load_times(p, n0 + 96, tb);
            fwd_decay_chunk(va, ta, p, d, wlo, wspan, wempty, row_ok, tail, row, n0 + 64, tmax);
            tmem_ld_wait();
            // every TMEM read of this accumulator half is in registers -> hand it back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(acc_empty_l + acc * 8);
            fwd_decay_chunk(vb, tb, p, d, wlo, wspan, wempty, row_ok, tail, row, n0 + 96, tmax);
            if (row_ok && p.tilemax) p.tilemax[(size_t)row * (p.e_pitch / 128) + tile * 2 + h] = tmax;
        }
    } else if (warp >= 4) {
        // ================= epilogue: thread <-> session row, warp <-> (TMEM lane quarter, column half) =================
        const uint32_t e = warp - 4;
        const uint32_t q = e & 3, h = e >> 2;
        const uint32_t row = mtile * BM + q * 32 + lane;
        const bool row_ok = row < (uint32_t)p.n_rows;
        const bool store_ok = row < (((uint32_t)p.n_rows + 63u) & ~63u);
        const float cshift = row_ok ? exp_shift(p, row) : 0.f;
        uint32_t wlo = 0, wspan = 0;
        bool wempty = false;
        if (MODE == 2 && row_ok) {                  // the row's window, loaded once
            const int32_t lo = p.win_lo[row], hi = p.win_hi[row];
            wlo = (uint32_t)lo;
            wspan = (uint32_t)hi - (uint32_t)lo;
            wempty = lo > hi;
        }
        const uint32_t acc_empty_l = mapa_u32(acc_empty, 0);
        for (uint32_t it = 0; it < my_tiles; ++it) {
            const uint32_t acc = it % P_NACC;
            const uint32_t acc_phase = (it / P_NACC) & 1;
            const uint32_t tile = tile0 + it * tile_step;
            const int n0 = tile * P_BN + h * 128;
            mbar_wait(&acc_full[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((q * 32) << 16) + acc * P_BN + h * 128;
            const bool tail = n0 + 128 > p.n_items;
            float psum = 0.f, tmax = -INFINITY, amax = -INFINITY;
            uint32_t va[32], vb[32];
            tmem_ld32(taddr, va);
            tmem_ld_wait();
            tmem_ld32(taddr + 32, vb);
            fwd_epilogue_chunk<MODE>(va, p, cshift, row_ok, store_ok, tail, row, n0, psum, tmax, amax, wlo, wspan,
                                     wempty);
            tmem_ld_wait();
            tmem_ld32(taddr + 64, va);
            fwd_epilogue_chunk<MODE>(vb, p, cshift, row_ok, store_ok, tail, row, n0 + 32, psum, tmax, amax, wlo, wspan,
                                     wempty);
            tmem_ld_wait();
            tmem_ld32(taddr + 96, vb);
            fwd_epilogue_chunk<MODE>(va, p, cshift, row_ok, store_ok, tail, row, n0 + 64, psum, tmax, amax, wlo, wspan,
                                     wempty);
            tmem_ld_wait();
            // every TMEM read of this accumulator half is in registers -> hand it back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(acc_empty_l + acc * 8);
            fwd_epilogue_chunk<MODE>(vb, p, cshift, row_ok, store_ok, tail, row, n0 + 96, psum, tmax, amax, wlo, wspan,
                                     wempty);
            if (row_ok) p.rowsum_part[(size_t)(tile * 2 + h) * QROWS + row] = psum;
            if (row_ok && p.rowmax_part)
                p.rowmax_part[(size_t)(tile * 2 + h) * QROWS + row] = MODE != 0 ? fmaf(tmax, kLog2e, -cshift) : amax;
            if (MODE != 0 && row_ok && p.tilemax) p.tilemax[(size_t)row * (p.e_pitch / 128) + tile * 2 + h] = tmax;
        }
    }

    tc_fence_before();
    cluster_sync_all();
    if (warp == 2) tmem_dealloc_pair(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------ forward, all groups
// The session groups of a catalog-sharded step (group g = rank g's <= 512 sessions, scored against the caller's item
// range) in ONE launch of the CTA-pair kernel.  Work unit = (row block of 256 sessions, item tile of 256); the units are
// numbered row-block major and every pair takes one contiguous run of them, so it changes its resident 2 x 160 KB
// session operand at most a few times (one TMA reload from L2 each, waited for by a `q_empty` barrier the MMA warp
// commits behind the last MMA that reads the old rows).  Replaces one launch per group (R x pipeline ramp, R x resident
// operand load per pair, and pairs left idle when 74 is not a multiple of the row blocks).
// Pass 2 of the overflow guard: row blocks none of whose rows are above the limit are skipped unit by unit.
constexpr int M_MAX_RB = 2 * TCAR_MAX_PEERS;       // row blocks: 16 groups x 2

struct FwdMultiParams {
    float* chunkmax;           // MODE 1: group g at chunkmax + g * cm_stride ([512, e_pitch/8] each)
    float* tilemax;            // MODE 1: group g at tilemax + g * tm_stride ([512, e_pitch/128] each)
    long long cm_stride, tm_stride;
    __nv_bfloat16* E;          // MODE 0: group g at E + g * e_stride
    float* rowsum_part;        // group g at rowsum_part + g * part_stride
    float* rowmax_part;        // same stride (nullable)
    const float* c_ref;        // group g at c_ref + g * c_stride
    const float* rowmax;       // group g at rowmax + g * rm_stride (nullable: pass 1)
    long long e_stride, part_stride, c_stride, rm_stride;
    int n_items, n_tiles, e_pitch, n_rb;
    int prefetch;              // L2 prefetch distance of the streamed item operand in stages (0 = off)
    unsigned char rb_group[M_MAX_RB], rb_block[M_MAX_RB];
    short rb_rows[M_MAX_RB];   // sessions of the row block's GROUP
};

template <int MODE>
__global__ void __launch_bounds__(P_THREADS, 1)
score_fwd_multi_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_i,
                       const __grid_constant__ FwdMultiParams p) {
    PDL_ENTER();
    extern __shared__ uint8_t smem_raw[];
    __shared__ int s_need[M_MAX_RB];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + F_A_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_b + P_STAGES * P_B_STAGE);
    uint64_t* full = bars;                      // [P_STAGES]  leader
    uint64_t* empty = bars + P_STAGES;          // [P_STAGES]  per CTA, MMA commit multicast
    uint64_t* acc_full = bars + 2 * P_STAGES;   // [P_NACC]    per CTA, MMA commit multicast
    uint64_t* acc_empty = acc_full + P_NACC;    // [P_NACC]    leader, 16 epilogue-warp arrivals
    uint64_t* a_full = acc_empty + P_NACC;      // [1]         leader: resident session rows landed
    uint64_t* q_empty = a_full + 1;             // [1]         per CTA, MMA commit multicast: old session rows retired
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(q_empty + 1);

    const uint32_t warp = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    const uint32_t rank = cluster_ctarank();    // 0 = leader
    const uint32_t pair_id = blockIdx.x >> 1;
    const uint32_t n_pairs = gridDim.x >> 1;
    const uint32_t units = (uint32_t)p.n_rb * (uint32_t)p.n_tiles;
    const uint32_t u0 = (uint32_t)(((uint64_t)pair_id * units) / n_pairs);
    const uint32_t u1 = (uint32_t)(((uint64_t)(pair_id + 1) * units) / n_pairs);

    // which row blocks does this pass touch?  (same answer in both CTAs of the pair)
    for (int rb = 0; rb < p.n_rb; ++rb) {
        bool need = p.rowmax == nullptr;
        if (p.rowmax) {
            const int g = p.rb_group[rb], r0 = p.rb_block[rb] * 2 * BM;
            for (int r = r0 + threadIdx.x; r < r0 + 2 * BM && r < p.rb_rows[rb]; r += blockDim.x)
                need |= p.rowmax[(size_t)g * p.rm_stride + r] > TCAR_EXP_LIMIT2;
        }
        const int any = __syncthreads_or(need);
        if (threadIdx.x == 0) s_need[rb] = any;
    }
    __syncthreads();
    bool work = false;
    for (uint32_t u = u0; u < u1; u += (uint32_t)p.n_tiles - (u % (uint32_t)p.n_tiles)) work |= s_need[u / p.n_tiles] != 0;
    if (!work) return;

    if (warp == 0 && elect_one()) {
        tma_prefetch_desc(&map_q);
        tma_prefetch_desc(&map_i);
    }
    if (warp == 1 && elect_one()) {
        for (int i = 0; i < P_STAGES; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], 1);
        }
        for (int i = 0; i < P_NACC; ++i) {
            mbar_init(&acc_full[i], 1);
            mbar_init(&acc_empty[i], 16);
        }
        mbar_init(a_full, 1);
        mbar_init(q_empty, 1);
        fence_mbar_init();
    }
    if (warp == 2) tmem_alloc_pair(tmem_slot, 512);
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= TMA producer (both CTAs; completion bytes land on the LEADER's barriers) =================
        if (elect_one()) {
            const uint32_t a_full_l = mapa_u32(a_full, 0);
            uint32_t stage = 0, phase = 0, qe_par = 0;
            int cur_rb = -1;
            // L2 prefetch `pf` stages ahead over the flattened (unit, K block) sequence of this pair
            const uint32_t pf = (uint32_t)p.prefetch;
            auto prefetch_stage = [&](uint32_t flat) {
                const uint32_t pu = u0 + flat / NKB, pkb = flat % NKB;
                if (pu < u1 && s_need[pu / p.n_tiles])
                    tma_prefetch_2d(&map_i, pkb * BK, (pu % p.n_tiles) * P_BN + rank * P_HALF);
            };
            for (uint32_t f = 0; f < pf; ++f) prefetch_stage(f);
            for (uint32_t u = u0; u < u1; ++u) {
                const int rb = u / p.n_tiles, tile = u % p.n_tiles;
                if (!s_need[rb]) continue;
                if (rb != cur_rb) {
                    if (cur_rb >= 0) {                       // every MMA reading the old rows has retired
                        mbar_wait(q_empty, qe_par);
                        qe_par ^= 1;
                    }
                    if (rank == 0) mbar_expect_tx(a_full, 2 * F_A_BYTES);
                    for (int kb = 0; kb < NKB; ++kb)
                        tma_load_3d_pair(smem_a + kb * (BM * BK * 2), &map_q, a_full_l, kb * BK,
                                         p.rb_block[rb] * 2 * BM + rank * BM, p.rb_group[rb]);
                    cur_rb = rb;
                }
                const int n0 = tile * P_BN + rank * P_HALF;
                for (int kb = 0; kb < NKB; ++kb) {
                    if (pf) prefetch_stage((u - u0) * NKB + kb + pf);
                    mbar_wait(&empty[stage], phase ^ 1);
                    if (rank == 0) mbar_expect_tx(&full[stage], 2 * P_B_STAGE);
                    tma_load_2d_pair(smem_b + stage * P_B_STAGE, &map_i, mapa_u32(&full[stage], 0), kb * BK, n0);
                    if (++stage == P_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer (leader CTA only) =================
        if (rank == 0) {
            constexpr uint32_t idesc = make_idesc_bf16(2 * BM, P_BN, 0, 0);
            uint32_t stage = 0, phase = 0, q_par = 0, it = 0;
            int cur_rb = -1;
            for (uint32_t u = u0; u < u1; ++u) {
                const int rb = u / p.n_tiles;
                if (!s_need[rb]) continue;
                if (rb != cur_rb) {
                    mbar_wait(a_full, q_par);
                    q_par ^= 1;
                    tc_fence_after();
                    cur_rb = rb;
                }
                // does a later unit of this pair use other session rows?  then they may be overwritten once the MMAs
                // of THIS unit have retired, provided this is the last unit of the current row block
                bool last_of_rb = true, more = false;
                for (uint32_t v = u + 1; v < u1; ++v) {
                    const int rv = v / p.n_tiles;
                    if (!s_need[rv]) continue;
                    if (rv == rb) last_of_rb = false; else more = true;
                    break;
                }
                const uint32_t acc = it % P_NACC;
                const uint32_t acc_phase = (it / P_NACC) & 1;
                ++it;
                mbar_wait(&acc_empty[acc], acc_phase ^ 1);
                tc_fence_after();
                for (int kb = 0; kb < NKB; ++kb) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    if (elect_one()) {
                        const uint32_t a_addr = smem_u32(smem_a + kb * (BM * BK * 2));
                        const uint32_t b_addr = smem_u32(smem_b + stage * P_B_STAGE);
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k)
                            umma_bf16_pair(tmem_base + acc * P_BN, sdesc_kmajor(a_addr + k * 32),
                                           sdesc_kmajor(b_addr + k * 32), idesc, (kb | k) != 0);
                        umma_commit_pair(&empty[stage], 3);
                        if (kb == NKB - 1) {
                            umma_commit_pair(&acc_full[acc], 3);
                            if (last_of_rb && more) umma_commit_pair(q_empty, 3);
                        }
                    }
                    __syncwarp();
                    if (++stage == P_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp >= 4) {
        // ================= epilogue: thread <-> session row, warp <-> (TMEM lane quarter, column half) =================
        const uint32_t e = warp - 4;
        const uint32_t q = e & 3, h = e >> 2;
        const uint32_t acc_empty_l = mapa_u32(acc_empty, 0);
        uint32_t it = 0;
        int cur_rb = -1;
        uint32_t row = 0;
        bool row_ok = false, store_ok = false;
        float cshift = 0.f;
        FwdParams pg;                      // the per-group view fwd_epilogue_chunk works on
        pg.n_items = p.n_items;
        pg.e_pitch = p.e_pitch;
        pg.E = p.E;
        pg.chunkmax = p.chunkmax;
        float* tmax_row = nullptr;
        size_t part_off = 0;
        for (uint32_t u = u0; u < u1; ++u) {
            const int rb = u / p.n_tiles;
            const uint32_t tile = u % p.n_tiles;
            if (!s_need[rb]) continue;
            if (rb != cur_rb) {
                cur_rb = rb;
                const int g = p.rb_group[rb];
                const uint32_t n_rows = (uint32_t)p.rb_rows[rb];
                row = p.rb_block[rb] * 2 * BM + rank * BM + q * 32 + lane;
                row_ok = row < n_rows;
                store_ok = row < ((n_rows + 63u) & ~63u);
                cshift = 0.f;
                if (row_ok) {
                    cshift = p.c_ref[(size_t)g * p.c_stride + row] * kLog2e;
                    if (p.rowmax) {
                        const float m = p.rowmax[(size_t)g * p.rm_stride + row];
                        if (m > TCAR_EXP_LIMIT2) cshift += m;
                    }
                }
                if (MODE == 0) pg.E = p.E + (size_t)g * p.e_stride;
                else {
                    pg.chunkmax = p.chunkmax + (size_t)g * p.cm_stride;
                    tmax_row = p.tilemax + (size_t)g * p.tm_stride + (size_t)row * (p.e_pitch / 128);
                }
                part_off = (size_t)g * p.part_stride;
            }
            const uint32_t acc = it % P_NACC;
            const uint32_t acc_phase = (it / P_NACC) & 1;
            ++it;
            const int n0 = tile * P_BN + h * 128;
            mbar_wait(&acc_full[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((q * 32) << 16) + acc * P_BN + h * 128;
            const bool tail = n0 + 128 > p.n_items;
            float psum = 0.f, tmax = -INFINITY, amax = -INFINITY;
            uint32_t va[32], vb[32];
            tmem_ld32(taddr, va);
            tmem_ld_wait();
            tmem_ld32(taddr + 32, vb);
            fwd_epilogue_chunk<MODE>(va, pg, cshift, row_ok, store_ok, tail, row, n0, psum, tmax, amax);
            tmem_ld_wait();
            tmem_ld32(taddr + 64, va);
            fwd_epilogue_chunk<MODE>(vb, pg, cshift, row_ok, store_ok, tail, row, n0 + 32, psum, tmax, amax);
            tmem_ld_wait();
            tmem_ld32(taddr + 96, vb);
            fwd_epilogue_chunk<MODE>(va, pg, cshift, row_ok, store_ok, tail, row, n0 + 64, psum, tmax, amax);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(acc_empty_l + acc * 8);
            fwd_epilogue_chunk<MODE>(vb, pg, cshift, row_ok, store_ok, tail, row, n0 + 96, psum, tmax, amax);
            if (row_ok) {
                p.rowsum_part[part_off + (size_t)(tile * 2 + h) * QROWS + row] = psum;
                if (p.rowmax_part)
                    p.rowmax_part[part_off + (size_t)(tile * 2 + h) * QROWS + row] =
                        MODE == 1 ? fmaf(tmax, kLog2e, -cshift) : amax;
                if (MODE == 1) tmax_row[tile * 2 + h] = tmax;
            }
        }
    }

    tc_fence_before();
    cluster_sync_all();
    if (warp == 2) tmem_dealloc_pair(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------ dQ = E . Iext
constexpr int Q_CH = 320;                 // feature columns per CTA (half of KEXT): one N=256 + one N=64 MMA
constexpr int Q_STAGES = 4;
constexpr int Q_A_STAGE = BM * BK * 2;    // 16384  E tile [128 b x 64 n], K-major
constexpr int Q_B_STAGE = Q_CH * BK * 2;  // 40960  Iext tile [64 n x 320 c], MN-major: 5 boxes of [64 c x 64 n]
constexpr int Q_STAGE = Q_A_STAGE + Q_B_STAGE;
constexpr int Q_SMEM = Q_STAGES * Q_STAGE + 1024 + 256;

constexpr int Q_MAX_MTILES = 64;   // 16 session groups x 4 m-tiles

struct BwdQParams {
    float* part;     // [splits, rows_total, 640]
    int kb_total;    // Npad / 64
    int kb_per;      // K blocks per split
    int splits;
    int mtiles;      // m-tiles of 128 session rows, over all groups
    int rows_total;  // rows of one split's partial: 512 (one group) or groups x 512
    int prefetch;    // L2 prefetch distance of both streamed operands in stages (0 = off)
    unsigned char grp[Q_MAX_MTILES];   // MULTI: session group and m-tile inside the group of every global m-tile
    unsigned char lmt[Q_MAX_MTILES];
};

// MULTI = false: one group of <= 512 sessions, E through a 3-D tensor map (the single-GPU / data-parallel step).
// MULTI = true : the session groups of a catalog-sharded step in ONE launch -- E_g a fixed stride apart behind a 4-D
// tensor map, unit = (split, global m-tile, column half): with R x 4 m-tiles the reduction over the items needs only
// 148 / (2 x 4R) splits, i.e. long K loops and a small split reduction instead of R short launches.
template <bool MULTI>
__global__ void __launch_bounds__(kThreads, 1)
score_bwd_q_kernel(const __grid_constant__ CUtensorMap map_e, const __grid_constant__ CUtensorMap map_i,
                   const BwdQParams p) {
    PDL_ENTER();
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Q_STAGES * Q_STAGE);
    uint64_t* full = bars;
    uint64_t* empty = bars + Q_STAGES;
    uint64_t* acc_full = bars + 2 * Q_STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);

    const uint32_t warp = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    // unit = (split, mtile, chalf)
    const uint32_t unit = blockIdx.x;
    const uint32_t chalf = unit & 1;
    const uint32_t gmt = (unit >> 1) % p.mtiles;
    const uint32_t split = (unit >> 1) / p.mtiles;
    const uint32_t grp = MULTI ? p.grp[gmt] : 0u;
    const uint32_t mtile = MULTI ? p.lmt[gmt] : gmt;
    const int kb0 = split * p.kb_per;
    const int kb1 = min(kb0 + p.kb_per, p.kb_total);
    const int nkb = max(kb1 - kb0, 0);

    if (warp == 0 && elect_one()) {
        tma_prefetch_desc(&map_e);
        tma_prefetch_desc(&map_i);
    }
    if (warp == 1 && elect_one()) {
        for (int i = 0; i < Q_STAGES; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], 1);
        }
        mbar_init(acc_full, 1);
        fence_mbar_init();
    }
    if (warp == 2) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (elect_one()) {
            uint32_t stage = 0, phase = 0;
            const int pf = p.prefetch;
            auto prefetch_stage = [&](int kb) {
                if (kb < kb1) {
                    if (MULTI) tma_prefetch_4d(&map_e, 0, mtile * (BM / 8), kb * (BK / 8), grp);
                    else tma_prefetch_3d(&map_e, 0, mtile * (BM / 8), kb * (BK / 8));
#pragma unroll
                    for (int j = 0; j < Q_CH / 64; ++j) tma_prefetch_2d(&map_i, chalf * Q_CH + j * 64, kb * BK);
                }
            };
            for (int kb = kb0; kb < kb0 + pf; ++kb) prefetch_stage(kb);
            for (int kb = kb0; kb < kb1; ++kb) {
                if (pf) prefetch_stage(kb + pf);
                mbar_wait(&empty[stage], phase ^ 1);
                mbar_expect_tx(&full[stage], Q_STAGE);
                uint8_t* sa = smem + stage * Q_STAGE;
                uint8_t* sb = sa + Q_A_STAGE;
                if (MULTI) tma_load_4d(sa, &map_e, &full[stage], 0, mtile * (BM / 8), kb * (BK / 8), grp);
                else tma_load_3d(sa, &map_e, &full[stage], 0, mtile * (BM / 8), kb * (BK / 8));
#pragma unroll
                for (int j = 0; j < Q_CH / 64; ++j)
                    tma_load_2d(sb + j * 8192, &map_i, &full[stage], chalf * Q_CH + j * 64, kb * BK);
                if (++stage == Q_STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc256 = make_idesc_bf16(BM, 256, 0, 1);
        constexpr uint32_t idesc64 = make_idesc_bf16(BM, 64, 0, 1);
        uint32_t stage = 0, phase = 0;
        for (int kb = kb0; kb < kb1; ++kb) {
            mbar_wait(&full[stage], phase);
            tc_fence_after();
            if (elect_one()) {
                const uint32_t a_addr = smem_u32(smem + stage * Q_STAGE);
                const uint32_t b_addr = a_addr + Q_A_STAGE;
#pragma unroll
                for (int k = 0; k < BK / 16; ++k) {
                    const uint32_t accum = (kb != kb0 || k != 0);
                    // E tile [8 item blocks][128 sessions][8 items]: core matrices 2048 B apart along K, 128 B along M
                    const uint64_t ad = make_sdesc_nosw(a_addr + k * 4096, 2048, 128);
                    umma_bf16(tmem_base, ad, sdesc_mnmajor(b_addr + k * 2048, 8192), idesc256, accum);
                    umma_bf16(tmem_base + 256, ad, sdesc_mnmajor(b_addr + 4 * 8192 + k * 2048, 8192), idesc64, accum);
                }
                umma_commit(&empty[stage]);
                if (kb == kb1 - 1) umma_commit(acc_full);
            }
            __syncwarp();
            if (++stage == Q_STAGES) { stage = 0; phase ^= 1; }
        }
    } else if (warp >= 4) {
        const uint32_t q = warp - 4;
        const uint32_t row = grp * QROWS + mtile * BM + q * 32 + lane;
        float* dst = p.part + ((size_t)split * p.rows_total + row) * KEXT + chalf * Q_CH;
        if (nkb > 0) {
            mbar_wait(acc_full, 0);
            tc_fence_after();
        }
#pragma unroll 1
        for (int ch = 0; ch < Q_CH / 32; ++ch) {
            uint32_t v[32];
            if (nkb > 0) {
                tmem_ld32(tmem_base + ((q * 32) << 16) + ch * 32, v);
                tmem_ld_wait();
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = 0u;
            }
#pragma unroll
            for (int g = 0; g < 8; ++g)
                reinterpret_cast<uint4*>(dst + ch * 32)[g] = make_uint4(v[g * 4], v[g * 4 + 1], v[g * 4 + 2], v[g * 4 + 3]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc(tmem_base, 512);
}

// Fixed-order reduction of the split partials: out[b, c] = sum_s part[s, b, c].
__global__ void reduce_splits_kernel(const float* __restrict__ part, float* __restrict__ out, int splits,
                                     int stride, int n) {
    PDL_ENTER();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float acc = 0.f;
    for (int s = 0; s < splits; ++s) acc += part[(size_t)s * stride + i];
    out[i] = acc;
}

// ------------------------------------------------------------------------------------------------ dItem = E^T . Qs
constexpr int I_BN = 128;                   // feature columns per CTA (half of the 256-pitch item row)
constexpr int I_STAGES = 6;
constexpr int I_A_STAGE = BM * BK * 2;      // 16384  E tile [64 b x 128 n], MN-major: 2 boxes of [64 n x 64 b]
constexpr int I_B_KB = I_BN * BK * 2;       // 16384  Qs tile [64 b x 128 c], MN-major: 2 boxes of [64 c x 64 b]
constexpr int I_NACC = 4;
constexpr int I_SMEM = 8 * I_B_KB + I_STAGES * I_A_STAGE + 1024 + 256;

struct BwdIParams {
    float* sq_partial;  // [gridDim.x] per-CTA sum of squares of the written gradient (nullable)
    float* g_item;   // [N+1, 256] dense item-table gradient (row 0 = pad item)
    int n_items;
    int n_tiles;     // ceil(Npad / 128)
    int nkb;         // ceil(B / 64)
    int accumulate;  // != 0: g_item += result (second and later session groups of a catalog-sharded step)
};

__global__ void __launch_bounds__(kThreads, 1)
score_bwd_i_kernel(const __grid_constant__ CUtensorMap map_e, const __grid_constant__ CUtensorMap map_qs,
                   const BwdIParams p) {
    PDL_ENTER();
    __shared__ float sq_red[4];
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* smem_b = smem;                         // resident Qs half: nkb x 16 KB
    uint8_t* smem_a = smem + 8 * I_B_KB;            // E stages
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_a + I_STAGES * I_A_STAGE);
    uint64_t* full = bars;
    uint64_t* empty = bars + I_STAGES;
    uint64_t* acc_full = bars + 2 * I_STAGES;
    uint64_t* acc_empty = acc_full + I_NACC;
    uint64_t* b_full = acc_empty + I_NACC;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(b_full + 1);

    const uint32_t warp = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    const uint32_t chalf = blockIdx.x & 1;
    const uint32_t tile0 = blockIdx.x >> 1;
    const uint32_t tile_step = gridDim.x >> 1;
    const uint32_t my_tiles =
        tile0 < (uint32_t)p.n_tiles ? ((uint32_t)p.n_tiles - tile0 + tile_step - 1) / tile_step : 0u;
    const int nkb = p.nkb;

    if (warp == 0 && elect_one()) {
        tma_prefetch_desc(&map_e);
        tma_prefetch_desc(&map_qs);
    }
    if (warp == 1 && elect_one()) {
        for (int i = 0; i < I_STAGES; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], 1);
        }
        for (int i = 0; i < I_NACC; ++i) {
            mbar_init(&acc_full[i], 1);
            mbar_init(&acc_empty[i], 4);
        }
        mbar_init(b_full, 1);
        fence_mbar_init();
    }
    if (warp == 2) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (elect_one()) {
            mbar_expect_tx(b_full, nkb * I_B_KB);
            for (int kb = 0; kb < nkb; ++kb)
                for (int j = 0; j < 2; ++j)
                    tma_load_2d(smem_b + kb * I_B_KB + j * 8192, &map_qs, b_full, chalf * I_BN + j * 64, kb * BK);
            uint32_t stage = 0, phase = 0;
            for (uint32_t it = 0; it < my_tiles; ++it) {
                const int n0 = (tile0 + it * tile_step) * BM;
                for (int kb = 0; kb < nkb; ++kb) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    mbar_expect_tx(&full[stage], I_A_STAGE);
                    uint8_t* sa = smem_a + stage * I_A_STAGE;
                    tma_load_3d(sa, &map_e, &full[stage], 0, kb * (BK / 8), n0 / 8);
                    if (++stage == I_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc = make_idesc_bf16(BM, I_BN, 1, 1);
        mbar_wait(b_full, 0);
        tc_fence_after();
        uint32_t stage = 0, phase = 0;
        for (uint32_t it = 0; it < my_tiles; ++it) {
            const uint32_t acc = it % I_NACC;
            const uint32_t acc_phase = (it / I_NACC) & 1;
            mbar_wait(&acc_empty[acc], acc_phase ^ 1);
            tc_fence_after();
            for (int kb = 0; kb < nkb; ++kb) {
                mbar_wait(&full[stage], phase);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t a_addr = smem_u32(smem_a + stage * I_A_STAGE);
                    const uint32_t b_addr = smem_u32(smem_b + kb * I_B_KB);
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k)
                        // E tile [16 item blocks][64 sessions][8 items]: MN-major, core matrices 1024 B apart along
                        // M (items), 128 B apart along K (sessions); one UMMA (K = 16 sessions) advances 256 B
                        umma_bf16(tmem_base + acc * I_BN, make_sdesc_nosw(a_addr + k * 256, 128, 1024),
                                  sdesc_mnmajor(b_addr + k * 2048, 8192), idesc, (kb | k) != 0);
                    umma_commit(&empty[stage]);
                    if (kb == nkb - 1) umma_commit(&acc_full[acc]);
                }
                __syncwarp();
                if (++stage == I_STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp >= 4) {
        // thread <-> item row
        const uint32_t q = warp - 4;
        float sq = 0.f;
        for (uint32_t it = 0; it < my_tiles; ++it) {
            const uint32_t acc = it % I_NACC;
            const uint32_t acc_phase = (it / I_NACC) & 1;
            const int n = (tile0 + it * tile_step) * BM + q * 32 + lane;
            mbar_wait(&acc_full[acc], acc_phase);
            tc_fence_after();
            float* dst = p.g_item + ((size_t)n + 1) * 256 + chalf * I_BN;
#pragma unroll 1
            for (int ch = 0; ch < I_BN / 32; ++ch) {
                uint32_t v[32];
                tmem_ld32(tmem_base + ((q * 32) << 16) + acc * I_BN + ch * 32, v);
                tmem_ld_wait();
                if (n < p.n_items) {
#pragma unroll
                    for (int g = 0; g < 8; ++g) {
                        uint4 o = make_uint4(v[g * 4], v[g * 4 + 1], v[g * 4 + 2], v[g * 4 + 3]);
                        const int c = chalf * I_BN + ch * 32 + g * 4;
                        if (c + 0 >= TCAR_H) o.x = 0u;   // pad columns 250..255 carry no parameter
                        if (c + 1 >= TCAR_H) o.y = 0u;
                        if (c + 2 >= TCAR_H) o.z = 0u;
                        if (c + 3 >= TCAR_H) o.w = 0u;
                        if (p.accumulate) {
                            const float4 old = reinterpret_cast<const float4*>(dst + ch * 32)[g];
                            o.x = __float_as_uint(old.x + __uint_as_float(o.x));
                            o.y = __float_as_uint(old.y + __uint_as_float(o.y));
                            o.z = __float_as_uint(old.z + __uint_as_float(o.z));
                            o.w = __float_as_uint(old.w + __uint_as_float(o.w));
                        }
                        reinterpret_cast<uint4*>(dst + ch * 32)[g] = o;
                        const float f0 = __uint_as_float(o.x), f1 = __uint_as_float(o.y);
                        const float f2 = __uint_as_float(o.z), f3 = __uint_as_float(o.w);
                        sq += (f0 * f0 + f1 * f1) + (f2 * f2 + f3 * f3);
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[acc]);
        }
        // fixed-order reduction of the 128 per-thread sums of squares -> one partial per CTA
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
        if (lane == 0) sq_red[q] = sq;
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (q == 0 && lane == 0 && p.sq_partial)
            p.sq_partial[blockIdx.x] = (sq_red[0] + sq_red[1]) + (sq_red[2] + sq_red[3]);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------ dItem, TMA-store epilogue
// The kernel above writes the gradient with thread <-> item row: every warp store touches 32 rows (32 half-written
// sectors), 4 096 sector requests per 128 x 128 tile against 1.5 us of MMA work -- the L1 store path, not HBM or the
// tensor pipe, set its 171 us (DRAM 50 %, tensor pipe 28 %).  Here the epilogue stages [128 rows x 32 columns] fp32
// blocks in shared memory (128-byte swizzle, conflict-free 16-byte stores) and one thread hands each block to the
// TMA: full 128-byte row segments, no LSU traffic.  MULTI: the session groups of a catalog-sharded step are
// concatenated along K (E and Qs blocks both streamed, 32 KB per stage), so that the gradient of the owned rows is
// accumulated in TMEM and written ONCE instead of overwritten by the first group and re-read + re-written by the others.
constexpr int I2_OUT = 2;
constexpr int I2_OUT_BYTES = BM * 32 * 4;                      // 16384
constexpr int I2_STAGES_ONE = 4;                               // single group: Qs half resident (128 KB) + E stages
constexpr int I2_STAGES_MULTI = 6;                             // several groups: (E | Qs) stages
constexpr int I2_SMEM_ONE = 8 * I_B_KB + I2_STAGES_ONE * I_A_STAGE + I2_OUT * I2_OUT_BYTES + 1024 + 256;
constexpr int I2_SMEM_MULTI = I2_STAGES_MULTI * (I_A_STAGE + I_B_KB) + I2_OUT * I2_OUT_BYTES + 1024 + 256;

struct BwdI2Params {
    float* sq_partial;            // [gridDim.x] per-CTA sum of squares of the written gradient (nullable)
    int n_items;
    int n_tiles;                  // ceil(Npad / 128)
    int groups;
    int prefetch;                 // L2 prefetch distance of the streamed E tiles in stages (0 = off)
    int nkb[TCAR_MAX_PEERS];      // 64-session K blocks of every group (0 = absent group)
};

template <bool MULTI>
__global__ void __launch_bounds__(kThreads, 1)
score_bwd_i_tma_kernel(const __grid_constant__ CUtensorMap map_e, const __grid_constant__ CUtensorMap map_qs,
                       const __grid_constant__ CUtensorMap map_g, const __grid_constant__ BwdI2Params p) {
    PDL_ENTER();
    constexpr int STAGES = MULTI ? I2_STAGES_MULTI : I2_STAGES_ONE;
    constexpr int STAGE_BYTES = MULTI ? I_A_STAGE + I_B_KB : I_A_STAGE;
    __shared__ float sq_red[4];
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* smem_b = smem;                                   // !MULTI: resident Qs half, nkb x 16 KB
    uint8_t* smem_a = smem + (MULTI ? 0 : 8 * I_B_KB);        // stages
    uint8_t* smem_o = smem_a + STAGES * STAGE_BYTES;          // output staging (1024-byte aligned)
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_o + I2_OUT * I2_OUT_BYTES);
    uint64_t* full = bars;
    uint64_t* empty = bars + STAGES;
    uint64_t* acc_full = bars + 2 * STAGES;
    uint64_t* acc_empty = acc_full + I_NACC;
    uint64_t* b_full = acc_empty + I_NACC;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(b_full + 1);

    const uint32_t warp = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    const uint32_t chalf = blockIdx.x & 1;
    const uint32_t tile0 = blockIdx.x >> 1;
    const uint32_t tile_step = gridDim.x >> 1;
    const uint32_t my_tiles =
        tile0 < (uint32_t)p.n_tiles ? ((uint32_t)p.n_tiles - tile0 + tile_step - 1) / tile_step : 0u;
    int kb_total = 0;                 // >= 1 (the host returns early when every group is absent)
    for (int g = 0; g < p.groups; ++g) kb_total += p.nkb[g];

    if (warp == 0 && elect_one()) {
        tma_prefetch_desc(&map_e);
        tma_prefetch_desc(&map_qs);
        tma_prefetch_desc(&map_g);
    }
    if (warp == 1 && elect_one()) {
        for (int i = 0; i < STAGES; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], 1);
        }
        for (int i = 0; i < I_NACC; ++i) {
            mbar_init(&acc_full[i], 1);
            mbar_init(&acc_empty[i], 4);
        }
        mbar_init(b_full, 1);
        fence_mbar_init();
    }
    if (warp == 2) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (elect_one()) {
            if (!MULTI) {
                mbar_expect_tx(b_full, p.nkb[0] * I_B_KB);
                for (int kb = 0; kb < p.nkb[0]; ++kb)
                    for (int j = 0; j < 2; ++j)
                        tma_load_3d(smem_b + kb * I_B_KB + j * 8192, &map_qs, b_full, chalf * I_BN + j * 64, kb * BK, 0);
            }
            uint32_t stage = 0, phase = 0;
            // L2 prefetch of the E boxes `pf` stages ahead: a second cursor (tile, group, K block) runs in front
            const int pf = p.prefetch;
            uint32_t p_it = 0;
            int p_g = 0, p_kb = 0;
            auto prefetch_next = [&]() {
                while (p_it < my_tiles && p_kb >= p.nkb[p_g]) {
                    p_kb = 0;
                    if (++p_g == p.groups) { p_g = 0; ++p_it; }
                }
                if (p_it < my_tiles) {
                    tma_prefetch_4d(&map_e, 0, p_kb * (BK / 8), (int)((tile0 + p_it * tile_step) * BM) / 8, p_g);
                    ++p_kb;
                }
            };
            for (int s = 0; s < pf; ++s) prefetch_next();
            for (uint32_t it = 0; it < my_tiles; ++it) {
                const int n0 = (tile0 + it * tile_step) * BM;
                for (int g = 0; g < p.groups; ++g) {
                    for (int kb = 0; kb < p.nkb[g]; ++kb) {
                        if (pf) prefetch_next();
                        mbar_wait(&empty[stage], phase ^ 1);
                        mbar_expect_tx(&full[stage], STAGE_BYTES);
                        uint8_t* sa = smem_a + stage * STAGE_BYTES;
                        tma_load_4d(sa, &map_e, &full[stage], 0, kb * (BK / 8), n0 / 8, g);
                        if (MULTI) {
                            for (int j = 0; j < 2; ++j)
                                tma_load_3d(sa + I_A_STAGE + j * 8192, &map_qs, &full[stage], chalf * I_BN + j * 64,
                                            kb * BK, g);
                        }
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc = make_idesc_bf16(BM, I_BN, 1, 1);
        if (!MULTI) {
            mbar_wait(b_full, 0);
            tc_fence_after();
        }
        uint32_t stage = 0, phase = 0;
        for (uint32_t it = 0; it < my_tiles; ++it) {
            const uint32_t acc = it % I_NACC;
            const uint32_t acc_phase = (it / I_NACC) & 1;
            mbar_wait(&acc_empty[acc], acc_phase ^ 1);
            tc_fence_after();
            int kidx = 0;
            for (int g = 0; g < p.groups; ++g) {
                const int nkb = p.nkb[g];
                for (int kb = 0; kb < nkb; ++kb, ++kidx) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    if (elect_one()) {
                        const uint32_t a_addr = smem_u32(smem_a + stage * STAGE_BYTES);
                        const uint32_t b_addr = MULTI ? a_addr + I_A_STAGE : smem_u32(smem_b + kb * I_B_KB);
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k)
                            umma_bf16(tmem_base + acc * I_BN, make_sdesc_nosw(a_addr + k * 256, 128, 1024),
                                      sdesc_mnmajor(b_addr + k * 2048, 8192), idesc, (kidx | k) != 0);
                        umma_commit(&empty[stage]);
                        if (kidx == kb_total - 1) umma_commit(&acc_full[acc]);
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp >= 4) {
        // thread <-> item row (TMEM lane); the 128 rows x 128 columns of a tile leave in four staged blocks
        const uint32_t q = warp - 4;
        const uint32_t r = q * 32 + lane;
        const bool issuer = (q == 0 && lane == 0);
        float sq = 0.f;
        uint32_t chunk = 0;
        for (uint32_t it = 0; it < my_tiles; ++it) {
            const uint32_t acc = it % I_NACC;
            const uint32_t acc_phase = (it / I_NACC) & 1;
            const int n0 = (tile0 + it * tile_step) * BM;
            const bool valid = n0 + (int)r < p.n_items;
            mbar_wait(&acc_full[acc], acc_phase);
            tc_fence_after();
#pragma unroll 1
            for (int ch = 0; ch < I_BN / 32; ++ch, ++chunk) {
                uint32_t v[32];
                tmem_ld32(tmem_base + ((q * 32) << 16) + acc * I_BN + ch * 32, v);
                tmem_ld_wait();
                uint8_t* ob = smem_o + (chunk & 1) * I2_OUT_BYTES;
#pragma unroll
                for (int g = 0; g < 8; ++g) {
                    uint4 o = make_uint4(v[g * 4], v[g * 4 + 1], v[g * 4 + 2], v[g * 4 + 3]);
                    const int c = chalf * I_BN + ch * 32 + g * 4;
                    if (c + 0 >= TCAR_H) o.x = 0u;   // pad columns 250..255 carry no parameter
                    if (c + 1 >= TCAR_H) o.y = 0u;
                    if (c + 2 >= TCAR_H) o.z = 0u;
                    if (c + 3 >= TCAR_H) o.w = 0u;
                    // 128-byte swizzle: 16-byte piece g of row r lives at piece g ^ (r & 7)
                    *reinterpret_cast<uint4*>(ob + r * 128 + ((g ^ (r & 7)) << 4)) = o;
                    if (valid) {
                        const float f0 = __uint_as_float(o.x), f1 = __uint_as_float(o.y);
                        const float f2 = __uint_as_float(o.z), f3 = __uint_as_float(o.w);
                        sq += (f0 * f0 + f1 * f1) + (f2 * f2 + f3 * f3);
                    }
                }
                fence_proxy_async();
                // the block staged two chunks ago used the other buffer; the one before this (same parity as the
                // NEXT chunk) must have left shared memory before anybody passes the barrier
                if (issuer) bulk_wait_read0();
                asm volatile("bar.sync 1, 128;" ::: "memory");
                if (issuer) {
                    // rows beyond the table (tail tile) are clipped by the tensor map; row 0 is the pad item
                    tma_store_2d(&map_g, ob, chalf * I_BN + ch * 32, n0 + 1);
                    bulk_commit();
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[acc]);
        }
        if (issuer) bulk_wait0();
        // fixed-order reduction of the 128 per-thread sums of squares -> one partial per CTA
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
        if (lane == 0) sq_red[q] = sq;
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (issuer && p.sq_partial)
            p.sq_partial[blockIdx.x] = (sq_red[0] + sq_red[1]) + (sq_red[2] + sq_red[3]);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
            qres != cudaDriverEntryPointSuccess)
            return nullptr;
        fn = reinterpret_cast<EncodeTiledFn>(ptr);
    }
    return fn;
}

// 2-D bf16 row-major tensor [rows, cols] (cols contiguous, pitch in elements); box = [box_cols, box_rows], SW128.
static int make_map_bf16(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint64_t pitch_elems,
                         uint32_t box_cols, uint32_t box_rows) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return TCAR_ERR_DRIVER;
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {pitch_elems * 2};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = tmap_encode_cached(fn, m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : TCAR_ERR_TENSORMAP;
}

// E in its block-of-8-items layout [n_pad/8][512][8] bf16 as a 3-D tensor (8 sessions x 8 items | session group |
// item block); the box (64, box_rows / 8, box_blocks) lands in shared memory, unswizzled, as
// [box_blocks][box_rows][8 items].
static int make_map_e(CUtensorMap* m, const void* base, uint64_t n_pad, uint32_t box_rows, uint32_t box_blocks) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return TCAR_ERR_DRIVER;
    // 8 consecutive session rows of one item block are 128 contiguous bytes (one UMMA core matrix): use that as the
    // innermost TMA dimension (a 16-byte inner dimension makes the copy engine crawl)
    cuuint64_t dims[3] = {64, (cuuint64_t)QROWS / 8, n_pad / 8};
    cuuint64_t strides[2] = {128, (cuuint64_t)QROWS * 16};
    cuuint32_t box[3] = {64, box_rows / 8, box_blocks};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = tmap_encode_cached(fn, m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : TCAR_ERR_TENSORMAP;
}

// The E blocks of several session groups, `group_stride` elements apart, as a 4-D tensor (group outermost).
static int make_map_e4(CUtensorMap* m, const void* base, uint64_t n_pad, uint32_t box_rows, uint32_t box_blocks,
                       uint32_t groups, uint64_t group_stride) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return TCAR_ERR_DRIVER;
    cuuint64_t dims[4] = {64, (cuuint64_t)QROWS / 8, n_pad / 8, groups};
    cuuint64_t strides[3] = {128, (cuuint64_t)QROWS * 16, group_stride * 2};
    cuuint32_t box[4] = {64, box_rows / 8, box_blocks, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = tmap_encode_cached(fn, m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : TCAR_ERR_TENSORMAP;
}

// Session operands of several groups, `group_stride` bf16 elements apart, as a 3-D tensor (k | row | group), SW128.
static int make_map_q3(CUtensorMap* m, const void* base, uint32_t groups, uint64_t group_stride) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return TCAR_ERR_DRIVER;
    cuuint64_t dims[3] = {KEXT, QROWS, groups};
    cuuint64_t strides[2] = {KEXT * 2, group_stride * 2};
    cuuint32_t box[3] = {BK, BM, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = tmap_encode_cached(fn, m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : TCAR_ERR_TENSORMAP;
}

static int sm_count() {
    static int n = 0;
    if (!n) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    }
    return n;
}

// L2 prefetch distance (stages) of the streamed GEMM operands (DESIGN §4.1): the forward gains equally at distances 4
// to 12 and loses from 16 on; the dQ GEMM is bound by the L2 -> SM fill, where prefetches only add requests
constexpr int PREFETCH_FWD = 12;
constexpr int PREFETCH_BWD_Q = 0;
constexpr int PREFETCH_BWD_I = 8;

template <int CL>
static int launch_fwd(const CUtensorMap& mq, const CUtensorMap& mi, const FwdParams& p, int n_clusters,
                      cudaStream_t stream) {
    TCAR_SET_SMEM_ONCE(score_fwd_kernel<CL>, F_SMEM);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(n_clusters * CL);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = F_SMEM;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
#ifndef TCAR_NO_PDL
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.numAttrs = 2;
#endif
    cudaError_t e = cudaLaunchKernelEx(&cfg, score_fwd_kernel<CL>, mq, mi, p);
    return (int)e;
}

template <int MODE>
static int launch_fwd_pair(const CUtensorMap& mq, const CUtensorMap& mi, const FwdParams& p, int n_pairs,
                           cudaStream_t stream) {
    TCAR_SET_SMEM_ONCE(score_fwd_pair_kernel<MODE>, P_SMEM);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(n_pairs * 2);
    cfg.blockDim = dim3(P_THREADS);
    cfg.dynamicSmemBytes = P_SMEM;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
#ifndef TCAR_NO_PDL
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.numAttrs = 2;
#endif
    return (int)cudaLaunchKernelEx(&cfg, score_fwd_pair_kernel<MODE>, mq, mi, p);
}

}  // namespace tcar

using namespace tcar;

extern "C" int tcar_score_fwd(const void* q_bf16, const void* iext_bf16, const float* c_ref, void* e_out,
                              float* rowsum_part, float* chunkmax, float* tilemax, int n_rows, int n_items, int n_pad,
                              int mode, int cluster, void* stream_) {
    return tcar_score_fwd_guarded(q_bf16, iext_bf16, c_ref, e_out, rowsum_part, chunkmax, tilemax, nullptr, nullptr,
                                  n_rows, n_items, n_pad, mode, cluster, stream_);
}

extern "C" int tcar_score_fwd_guarded(const void* q_bf16, const void* iext_bf16, const float* c_ref, void* e_out,
                                      float* rowsum_part, float* chunkmax, float* tilemax, float* rowmax_part,
                                      const float* rowmax, int n_rows, int n_items, int n_pad, int mode, int cluster,
                                      void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (n_rows < 1 || n_rows > QROWS || n_pad % 256 != 0 || n_items > n_pad) return TCAR_ERR_ARG;
    if (cluster != 1 && cluster != 2 && cluster != 4 && cluster != TCAR_CLUSTER_PAIR) return TCAR_ERR_ARG;
    if ((mode == 0 && !e_out) || (mode == 1 && !chunkmax) || (mode != 0 && mode != 1)) return TCAR_ERR_ARG;
    CUtensorMap mq, mi;
    int rc = make_map_bf16(&mq, q_bf16, QROWS, KEXT, KEXT, BK, BM);
    if (rc) return rc;
    if (cluster == TCAR_CLUSTER_PAIR) {
        rc = make_map_bf16(&mi, iext_bf16, n_pad, KEXT, KEXT, BK, P_HALF);
        if (rc) return rc;
        FwdParams p;
        p.E = static_cast<__nv_bfloat16*>(e_out);
        p.rowsum_part = rowsum_part;
        p.chunkmax = chunkmax;
        p.tilemax = tilemax;
        p.c_ref = c_ref;
        p.rowmax_part = rowmax_part;
        p.rowmax = rowmax;
        p.n_items = n_items;
        p.n_tiles = n_pad / P_BN;
        p.n_rows = n_rows;
        p.e_pitch = n_pad;
        const int mtiles = (n_rows + BM - 1) / BM;
        p.groups = (mtiles + 1) / 2;
        p.mode = mode;
        p.prefetch = PREFETCH_FWD;
        int n_pairs = ((sm_count() / 2) / p.groups) * p.groups;
        if (n_pairs < p.groups) n_pairs = p.groups;
        if (n_pairs / p.groups > p.n_tiles) n_pairs = p.n_tiles * p.groups;
        return mode == 0 ? launch_fwd_pair<0>(mq, mi, p, n_pairs, stream) : launch_fwd_pair<1>(mq, mi, p, n_pairs, stream);
    }
    rc = make_map_bf16(&mi, iext_bf16, n_pad, KEXT, KEXT, BK, F_BN / cluster);
    if (rc) return rc;
    FwdParams p;
    p.E = static_cast<__nv_bfloat16*>(e_out);
    p.rowsum_part = rowsum_part;
    p.chunkmax = chunkmax;
    p.tilemax = tilemax;
    p.c_ref = c_ref;
    p.rowmax_part = rowmax_part;
    p.rowmax = rowmax;
    p.n_items = n_items;
    p.n_tiles = n_pad / F_BN;
    p.n_rows = n_rows;
    p.e_pitch = n_pad;
    const int mtiles = (n_rows + BM - 1) / BM;
    p.groups = (mtiles + cluster - 1) / cluster;
    p.mode = mode;
    p.prefetch = 0;
    // cluster size 4 can only be co-scheduled on 132 of the 148 SMs (GPCs with 18 SMs strand two)
    int max_clusters = sm_count() / cluster;
    if (cluster == 4) max_clusters = (sm_count() * 132 / 148) / 4;
    int n_clusters = (max_clusters / p.groups) * p.groups;
    if (n_clusters < p.groups) n_clusters = p.groups;
    const int per_group = n_clusters / p.groups;
    if (per_group > p.n_tiles) n_clusters = p.n_tiles * p.groups;
    if (cluster == 1) return launch_fwd<1>(mq, mi, p, n_clusters, stream);
    if (cluster == 2) return launch_fwd<2>(mq, mi, p, n_clusters, stream);
    return launch_fwd<4>(mq, mi, p, n_clusters, stream);
}

// Eval mode with a publish-time window per row: score_fwd_pair_kernel<2>, whatever cluster setting the caller's model
// uses for tcar_score_fwd (the pair kernel only needs n_pad % 256 == 0).
extern "C" int tcar_score_fwd_window(const void* q_bf16, const void* iext_bf16, const float* c_ref, float* rowsum_part,
                                     float* chunkmax, float* tilemax, const int32_t* item_time, const int32_t* win_lo,
                                     const int32_t* win_hi, int n_rows, int n_items, int n_pad, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (n_rows < 1 || n_rows > QROWS || n_items < 1 || n_pad % 256 != 0 || n_items > n_pad || !q_bf16 || !iext_bf16 ||
        !c_ref || !rowsum_part || !chunkmax || !item_time || !win_lo || !win_hi)
        return TCAR_ERR_ARG;
    CUtensorMap mq, mi;
    int rc = make_map_bf16(&mq, q_bf16, QROWS, KEXT, KEXT, BK, BM);
    if (rc) return rc;
    rc = make_map_bf16(&mi, iext_bf16, n_pad, KEXT, KEXT, BK, P_HALF);
    if (rc) return rc;
    FwdParams p = {};
    p.rowsum_part = rowsum_part;
    p.chunkmax = chunkmax;
    p.tilemax = tilemax;
    p.c_ref = c_ref;
    p.n_items = n_items;
    p.n_tiles = n_pad / P_BN;
    p.n_rows = n_rows;
    p.e_pitch = n_pad;
    const int mtiles = (n_rows + BM - 1) / BM;
    p.groups = (mtiles + 1) / 2;
    p.mode = 2;
    p.prefetch = PREFETCH_FWD;
    p.item_time = item_time;
    p.win_lo = win_lo;
    p.win_hi = win_hi;
    int n_pairs = ((sm_count() / 2) / p.groups) * p.groups;
    if (n_pairs < p.groups) n_pairs = p.groups;
    if (n_pairs / p.groups > p.n_tiles) n_pairs = p.n_tiles * p.groups;
    return launch_fwd_pair<2>(mq, mi, p, n_pairs, stream);
}

// Eval mode with a freshness decay per row (and an optional window): score_fwd_pair_kernel<3>, the same grid as
// tcar_score_fwd_window
extern "C" int tcar_score_fwd_decay(const void* q_bf16, const void* iext_bf16, float* chunkmax, float* tilemax,
                                    const int32_t* item_time, const int32_t* t_ref, const float* rate,
                                    const int32_t* win_lo, const int32_t* win_hi, int n_rows, int n_items, int n_pad,
                                    void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (n_rows < 1 || n_rows > QROWS || n_items < 1 || n_pad % 256 != 0 || n_items > n_pad || !q_bf16 || !iext_bf16 ||
        !chunkmax || !item_time || !t_ref || !rate || !win_lo != !win_hi)
        return TCAR_ERR_ARG;
    CUtensorMap mq, mi;
    int rc = make_map_bf16(&mq, q_bf16, QROWS, KEXT, KEXT, BK, BM);
    if (rc) return rc;
    rc = make_map_bf16(&mi, iext_bf16, n_pad, KEXT, KEXT, BK, P_HALF);
    if (rc) return rc;
    FwdParams p = {};
    p.chunkmax = chunkmax;
    p.tilemax = tilemax;
    p.n_items = n_items;
    p.n_tiles = n_pad / P_BN;
    p.n_rows = n_rows;
    p.e_pitch = n_pad;
    const int mtiles = (n_rows + BM - 1) / BM;
    p.groups = (mtiles + 1) / 2;
    p.mode = 3;
    p.prefetch = PREFETCH_FWD;
    p.item_time = item_time;
    p.win_lo = win_lo;
    p.win_hi = win_hi;
    p.t_ref = t_ref;
    p.rate = rate;
    int n_pairs = ((sm_count() / 2) / p.groups) * p.groups;
    if (n_pairs < p.groups) n_pairs = p.groups;
    if (n_pairs / p.groups > p.n_tiles) n_pairs = p.n_tiles * p.groups;
    return launch_fwd_pair<3>(mq, mi, p, n_pairs, stream);
}

extern "C" int tcar_score_fwd_tiles(int n_pad) { return n_pad / F_BN; }

static int score_fwd_multi_impl(const void* q_bf16, long long q_stride, const float* c_ref, long long c_stride,
                                const void* iext_bf16, void* e_out, long long e_stride, float* chunkmax,
                                long long cm_stride, float* tilemax, long long tm_stride, float* rowsum_part,
                                long long part_stride, float* rowmax_part, const float* rowmax, long long rm_stride,
                                const int* n_rows, int groups, int n_items, int n_pad, void* stream_);

// All session groups in one launch (score_fwd_multi_kernel): train mode, CTA pairs.  Strides in ELEMENTS of the
// respective arrays; rowmax_part shares part_stride; rowmax is [groups][512].
extern "C" int tcar_score_fwd_multi(const void* q_bf16, long long q_stride, const float* c_ref, long long c_stride,
                                    const void* iext_bf16, void* e_out, long long e_stride, float* rowsum_part,
                                    long long part_stride, float* rowmax_part, const float* rowmax, const int* n_rows,
                                    int groups, int n_items, int n_pad, void* stream_) {
    if (!e_out || e_stride < (long long)QROWS * n_pad) return TCAR_ERR_ARG;
    return score_fwd_multi_impl(q_bf16, q_stride, c_ref, c_stride, iext_bf16, e_out, e_stride, nullptr, 0, nullptr, 0,
                                rowsum_part, part_stride, rowmax_part, rowmax, QROWS, n_rows, groups, n_items, n_pad,
                                stream_);
}

extern "C" int tcar_score_fwd_multi_eval(const void* q_bf16, long long q_stride, const float* c_ref, long long c_stride,
                                         const void* iext_bf16, float* chunkmax, long long cm_stride, float* tilemax,
                                         long long tm_stride, float* rowsum_part, long long part_stride,
                                         float* rowmax_part, const float* rowmax, long long rowmax_stride,
                                         const int* n_rows, int groups, int n_items, int n_pad, void* stream_) {
    if (!chunkmax || !tilemax || cm_stride < (long long)QROWS * (n_pad / 8) || tm_stride < (long long)QROWS * (n_pad / 128))
        return TCAR_ERR_ARG;
    return score_fwd_multi_impl(q_bf16, q_stride, c_ref, c_stride, iext_bf16, nullptr, 0, chunkmax, cm_stride, tilemax,
                                tm_stride, rowsum_part, part_stride, rowmax_part, rowmax, rowmax_stride, n_rows, groups,
                                n_items, n_pad, stream_);
}

static int score_fwd_multi_impl(const void* q_bf16, long long q_stride, const float* c_ref, long long c_stride,
                                const void* iext_bf16, void* e_out, long long e_stride, float* chunkmax,
                                long long cm_stride, float* tilemax, long long tm_stride, float* rowsum_part,
                                long long part_stride, float* rowmax_part, const float* rowmax, long long rm_stride,
                                const int* n_rows, int groups, int n_items, int n_pad, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (!n_rows || groups < 1 || groups > TCAR_MAX_PEERS || n_pad % 256 != 0 || n_items > n_pad ||
        !rowsum_part || q_stride < (long long)QROWS * KEXT || (q_stride & 7))
        return TCAR_ERR_ARG;
    FwdMultiParams p = {};
    int nrb = 0;
    for (int g = 0; g < groups; ++g) {
        if (n_rows[g] > QROWS) return TCAR_ERR_ARG;
        if (n_rows[g] <= 0) continue;
        for (int b = 0; b * 2 * BM < n_rows[g]; ++b, ++nrb) {
            p.rb_group[nrb] = (unsigned char)g;
            p.rb_block[nrb] = (unsigned char)b;
            p.rb_rows[nrb] = (short)n_rows[g];
        }
    }
    if (nrb == 0) return 0;
    CUtensorMap mq, mi;
    int rc = make_map_q3(&mq, q_bf16, (uint32_t)groups, (uint64_t)q_stride);
    if (rc) return rc;
    rc = make_map_bf16(&mi, iext_bf16, n_pad, KEXT, KEXT, BK, P_HALF);
    if (rc) return rc;
    p.E = static_cast<__nv_bfloat16*>(e_out);
    p.chunkmax = chunkmax;
    p.tilemax = tilemax;
    p.cm_stride = cm_stride;
    p.tm_stride = tm_stride;
    p.rowsum_part = rowsum_part;
    p.rowmax_part = rowmax_part;
    p.c_ref = c_ref;
    p.rowmax = rowmax;
    p.e_stride = e_stride;
    p.part_stride = part_stride;
    p.rm_stride = rm_stride;
    p.c_stride = c_stride;
    p.n_items = n_items;
    p.n_tiles = n_pad / P_BN;
    p.e_pitch = n_pad;
    p.n_rb = nrb;
    p.prefetch = PREFETCH_FWD;
    int n_pairs = sm_count() / 2;
    if ((long long)n_pairs > (long long)nrb * p.n_tiles) n_pairs = nrb * p.n_tiles;
    const bool eval_mode = e_out == nullptr;
    if (eval_mode) TCAR_SET_SMEM_ONCE(score_fwd_multi_kernel<1>, P_SMEM);
    else TCAR_SET_SMEM_ONCE(score_fwd_multi_kernel<0>, P_SMEM);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(n_pairs * 2);
    cfg.blockDim = dim3(P_THREADS);
    cfg.dynamicSmemBytes = P_SMEM;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
#ifndef TCAR_NO_PDL
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.numAttrs = 2;
#endif
    return eval_mode ? (int)cudaLaunchKernelEx(&cfg, score_fwd_multi_kernel<1>, mq, mi, p)
                     : (int)cudaLaunchKernelEx(&cfg, score_fwd_multi_kernel<0>, mq, mi, p);
}

extern "C" int tcar_score_bwd_q_splits(int n_rows, int n_pad) {
    const int mtiles = (n_rows + BM - 1) / BM;
    int splits = sm_count() / (2 * mtiles);
    const int kb_total = n_pad / BK;
    if (splits > kb_total) splits = kb_total;
    if (splits < 1) splits = 1;
    return splits;
}

extern "C" int tcar_score_bwd_q(const void* e_bf16, const void* iext_bf16, float* part, float* dq, int n_rows,
                                int n_pad, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (n_rows < 1 || n_rows > QROWS || n_pad % 256 != 0) return TCAR_ERR_ARG;
    CUtensorMap me, mi;
    int rc = make_map_e(&me, e_bf16, n_pad, BM, BK / 8);
    if (rc) return rc;
    rc = make_map_bf16(&mi, iext_bf16, n_pad, KEXT, KEXT, 64, BK);
    if (rc) return rc;
    BwdQParams p;
    p.part = part;
    p.mtiles = (n_rows + BM - 1) / BM;
    p.splits = tcar_score_bwd_q_splits(n_rows, n_pad);
    p.prefetch = PREFETCH_BWD_Q;
    p.kb_total = n_pad / BK;
    p.kb_per = (p.kb_total + p.splits - 1) / p.splits;
    p.rows_total = QROWS;
    TCAR_SET_SMEM_ONCE(score_bwd_q_kernel<false>, Q_SMEM);
    launch_pdl(score_bwd_q_kernel<false>, dim3(p.splits * p.mtiles * 2), dim3(kThreads), Q_SMEM, stream, me, mi, p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
    // partial layout is [split][512][640]; rows of m-tiles that were not computed are never read by callers
    const int total = p.mtiles * BM * KEXT;
    launch_pdl(reduce_splits_kernel, dim3((total + 255) / 256), dim3(256), 0, stream, part, dq, p.splits, QROWS * KEXT, total);
    return (int)cudaGetLastError();
}

// All session groups of a catalog-sharded step in one launch (see score_bwd_q_kernel<true>): dq [groups][512][640],
// part >= tcar_score_bwd_q_multi_part_elems(groups) floats.  Groups with n_rows[g] <= 0 are skipped (their dq rows
// receive whatever the unused partial rows hold -- never read by callers).
extern "C" long long tcar_score_bwd_q_multi_part_elems(int groups) {
    return (long long)(groups > 24 ? groups : 24) * QROWS * KEXT;
}

extern "C" int tcar_score_bwd_q_multi(const void* e_bf16, long long e_stride, const void* iext_bf16, float* part,
                                      float* dq, const int* n_rows, int groups, int n_pad, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (!n_rows || groups < 1 || groups > 16 || n_pad % 256 != 0 || e_stride < (long long)QROWS * n_pad ||
        (e_stride & 7))
        return TCAR_ERR_ARG;
    BwdQParams p = {};
    int mt = 0;
    for (int g = 0; g < groups; ++g) {
        if (n_rows[g] > QROWS) return TCAR_ERR_ARG;
        const int m = n_rows[g] > 0 ? (n_rows[g] + BM - 1) / BM : 0;
        for (int l = 0; l < m; ++l, ++mt) {
            p.grp[mt] = (unsigned char)g;
            p.lmt[mt] = (unsigned char)l;
        }
    }
    if (mt == 0) return 0;
    CUtensorMap me, mi;
    int rc = make_map_e4(&me, e_bf16, n_pad, BM, BK / 8, groups, (uint64_t)e_stride);
    if (rc) return rc;
    rc = make_map_bf16(&mi, iext_bf16, n_pad, KEXT, KEXT, 64, BK);
    if (rc) return rc;
    p.part = part;
    p.mtiles = mt;
    p.kb_total = n_pad / BK;
    int splits = sm_count() / (2 * mt);
    const int cap = 24 / groups > 0 ? 24 / groups : 1;      // part holds 24 x 512 rows
    if (splits > cap) splits = cap;
    if (splits > p.kb_total) splits = p.kb_total;
    if (splits < 1) splits = 1;
    p.splits = splits;
    p.prefetch = PREFETCH_BWD_Q;
    p.kb_per = (p.kb_total + splits - 1) / splits;
    p.rows_total = groups * QROWS;
    TCAR_SET_SMEM_ONCE(score_bwd_q_kernel<true>, Q_SMEM);
    launch_pdl(score_bwd_q_kernel<true>, dim3(splits * mt * 2), dim3(kThreads), Q_SMEM, stream, me, mi, p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
    const int total = groups * QROWS * KEXT;
    launch_pdl(reduce_splits_kernel, dim3((total + 255) / 256), dim3(256), 0, stream, part, dq, splits, total, total);
    return (int)cudaGetLastError();
}

// Qs blocks of several session groups, `group_stride` bf16 elements apart: (feature column | session | group), SW128.
static int make_map_qs3(CUtensorMap* m, const void* base, uint32_t groups, uint64_t group_stride) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return TCAR_ERR_DRIVER;
    cuuint64_t dims[3] = {256, QROWS, groups};
    cuuint64_t strides[2] = {256 * 2, group_stride * 2};
    cuuint32_t box[3] = {64, BK, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = tmap_encode_cached(fn, m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : TCAR_ERR_TENSORMAP;
}

// Dense item gradient [rows, 256] fp32 as the destination of the staged [128 rows x 32 columns] blocks (SW128).
static int make_map_g(CUtensorMap* m, float* base, uint64_t rows) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return TCAR_ERR_DRIVER;
    cuuint64_t dims[2] = {256, rows};
    cuuint64_t strides[1] = {256 * 4};
    cuuint32_t box[2] = {32, BM};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = tmap_encode_cached(fn, m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : TCAR_ERR_TENSORMAP;
}

static int bwd_i_grid(int n_pad) {
    int grid = (sm_count() / 2) * 2;
    const int n_tiles = n_pad / BM;
    if (grid > 2 * n_tiles) grid = 2 * n_tiles;
    return grid;
}

extern "C" int tcar_score_bwd_i_ctas(int n_pad) { return bwd_i_grid(n_pad); }

extern "C" int tcar_score_bwd_i(const void* e_bf16, const void* qs_bf16, float* g_item, float* sq_partial, int n_rows,
                                int n_items, int n_pad, void* stream_) {
    return tcar_score_bwd_i_acc(e_bf16, qs_bf16, g_item, sq_partial, n_rows, n_items, n_pad, 0, stream_);
}

extern "C" int tcar_score_bwd_i_multi(const void* e_bf16, long long e_stride, const void* qs_bf16, long long qs_stride,
                                      float* g_item, float* sq_partial, const int* n_rows, int groups, int n_items,
                                      int n_pad, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (!n_rows || groups < 1 || groups > TCAR_MAX_PEERS || n_pad % 256 != 0 || n_items < 1 || n_items > n_pad)
        return TCAR_ERR_ARG;
    BwdI2Params p;
    p.sq_partial = sq_partial;
    p.n_items = n_items;
    p.n_tiles = n_pad / BM;
    p.groups = groups;
    p.prefetch = PREFETCH_BWD_I;
    int present = 0, only = -1;
    for (int g = 0; g < TCAR_MAX_PEERS; ++g) {
        const int b = g < groups ? n_rows[g] : 0;
        if (b < 0 || b > QROWS) return TCAR_ERR_ARG;
        p.nkb[g] = (b + BK - 1) / BK;
        if (b > 0) { ++present; only = g; }
    }
    if (present == 0) return 0;
    const bool multi = present > 1;
    const uint16_t* e0 = static_cast<const uint16_t*>(e_bf16);
    const uint16_t* q0 = static_cast<const uint16_t*>(qs_bf16);
    if (!multi) {              // one group: its Qs half stays resident, group index 0 of maps based at that group
        e0 += (long long)only * e_stride;
        q0 += (long long)only * qs_stride;
        p.nkb[0] = p.nkb[only];
        for (int g = 1; g < TCAR_MAX_PEERS; ++g) p.nkb[g] = 0;
        p.groups = 1;
    }
    CUtensorMap me, mq, mg;
    int rc = make_map_e4(&me, e0, n_pad, BK, BM / 8, multi ? groups : 1, multi ? (uint64_t)e_stride : (uint64_t)QROWS * n_pad);
    if (rc) return rc;
    rc = make_map_qs3(&mq, q0, multi ? groups : 1, multi ? (uint64_t)qs_stride : (uint64_t)QROWS * 256);
    if (rc) return rc;
    rc = make_map_g(&mg, g_item, (uint64_t)n_items + 1);
    if (rc) return rc;
    const int grid = bwd_i_grid(n_pad);
    if (multi) {
        TCAR_SET_SMEM_ONCE(score_bwd_i_tma_kernel<true>, I2_SMEM_MULTI);
        launch_pdl(score_bwd_i_tma_kernel<true>, dim3(grid), dim3(kThreads), I2_SMEM_MULTI, stream, me, mq, mg, p);
    } else {
        TCAR_SET_SMEM_ONCE(score_bwd_i_tma_kernel<false>, I2_SMEM_ONE);
        launch_pdl(score_bwd_i_tma_kernel<false>, dim3(grid), dim3(kThreads), I2_SMEM_ONE, stream, me, mq, mg, p);
    }
    return (int)cudaGetLastError();
}

extern "C" int tcar_score_bwd_i_acc(const void* e_bf16, const void* qs_bf16, float* g_item, float* sq_partial,
                                    int n_rows, int n_items, int n_pad, int accumulate, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (n_rows < 1 || n_rows > QROWS || n_pad % 256 != 0) return TCAR_ERR_ARG;
    if (!accumulate)
        return tcar_score_bwd_i_multi(e_bf16, 0, qs_bf16, 0, g_item, sq_partial, &n_rows, 1, n_items, n_pad, stream_);
    CUtensorMap me, mq;
    int rc = make_map_e(&me, e_bf16, n_pad, BK, BM / 8);
    if (rc) return rc;
    rc = make_map_bf16(&mq, qs_bf16, QROWS, 256, 256, 64, BK);
    if (rc) return rc;
    BwdIParams p;
    p.sq_partial = sq_partial;
    p.g_item = g_item;
    p.n_items = n_items;
    p.n_tiles = n_pad / BM;
    p.nkb = (n_rows + BK - 1) / BK;
    p.accumulate = accumulate;
    TCAR_SET_SMEM_ONCE(score_bwd_i_kernel, I_SMEM);
    const int grid = bwd_i_grid(n_pad);
    launch_pdl(score_bwd_i_kernel, dim3(grid), dim3(kThreads), I_SMEM, stream, me, mq, p);
    return (int)cudaGetLastError();
}
