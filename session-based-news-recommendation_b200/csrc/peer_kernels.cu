// Peer-memory plumbing of the catalog-sharded train step (SURVEY 8e row 2 / 8f-3): every rank owns a contiguous range
// of item-table rows (fp32 master copy + Adam moments); the rows a rank's sessions gather (clicks, labels, negatives)
// are read straight out of the owner's HBM over NVLink / NVSwitch with plain loads -- no staging buffer, no
// collective, ~1 KB per row.  The reference has no multi-device code; this replaces what would otherwise be an
// all-gather of the whole updated table (364 MB per step) after model_combine.py:163.
#include <cuda_runtime.h>
#include <cuda.h>
#include <stdint.h>
#include <string.h>
#include "tcar_b200.h"
#include "launch.cuh"

namespace tcar {

struct PeerTable {
    const float* base[TCAR_MAX_PEERS];   // table origin (row 0) in every rank's address space mapping
    int bound[TCAR_MAX_PEERS + 1];       // rank g owns rows [bound[g], bound[g+1])
    int G, self;
};

// one warp per listed row (clicks [0,M): seq as is; labels [M,M+B) and negatives [M+B, M+B+B*Nn): id + 1): 2 x 128-bit
// loads per lane from the owner (L1 bypassed: the owner rewrites its rows every step), 2 x 128-bit stores into the
// local replica.  Rows the caller owns, rows outside the table and duplicates (same bytes written twice) need no
// special care.
__global__ void __launch_bounds__(256)
peer_fetch_rows_kernel(const int32_t* __restrict__ seq, const int32_t* __restrict__ label,
                       const int32_t* __restrict__ neg, int M, int B, int n, const PeerTable pt,
                       float* __restrict__ table) {
    PDL_ENTER();
    const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (e >= n) return;
    const int row = e < M ? seq[e] : (e < M + B ? label[e - M] + 1 : neg[e - M - B] + 1);
    if (row < pt.bound[0] || row >= pt.bound[pt.G]) return;
    int owner = 0;
    while (row >= pt.bound[owner + 1]) ++owner;
    if (owner == pt.self) return;
    const float4* src = reinterpret_cast<const float4*>(pt.base[owner] + (size_t)row * TCAR_HP);
    float4* dst = reinterpret_cast<float4*>(table + (size_t)row * TCAR_HP);
    const float4 v0 = __ldcg(src + lane), v1 = __ldcg(src + 32 + lane);
    dst[lane] = v0;
    dst[32 + lane] = v1;
}

typedef CUresult (*AddrRangeFn)(CUdeviceptr*, size_t*, CUdeviceptr);

static AddrRangeFn addr_range_fn() {
    static AddrRangeFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            return nullptr;
        fn = reinterpret_cast<AddrRangeFn>(p);
    }
    return fn;
}

}  // namespace tcar

using namespace tcar;

extern "C" int tcar_peer_export(const void* ptr, unsigned char* handle, long long* offset) {
    if (!ptr || !handle || !offset) return TCAR_ERR_ARG;
    static_assert(sizeof(cudaIpcMemHandle_t) == TCAR_PEER_HANDLE_BYTES, "IPC handle size");
    AddrRangeFn fn = addr_range_fn();
    if (!fn) return TCAR_ERR_DRIVER;
    CUdeviceptr base = 0;
    size_t size = 0;
    if (fn(&base, &size, reinterpret_cast<CUdeviceptr>(ptr)) != CUDA_SUCCESS) return TCAR_ERR_DRIVER;
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, reinterpret_cast<void*>(base));
    if (e != cudaSuccess) return (int)e;
    memcpy(handle, &h, sizeof(h));
    *offset = (long long)(reinterpret_cast<CUdeviceptr>(ptr) - base);
    return 0;
}

extern "C" int tcar_peer_open(const unsigned char* handle, long long offset, void** ptr) {
    if (!handle || !ptr || offset < 0) return TCAR_ERR_ARG;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    void* base = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return (int)e;
    *ptr = static_cast<char*>(base) + offset;
    return 0;
}

extern "C" int tcar_peer_close(void* ptr, long long offset) {
    if (!ptr) return TCAR_ERR_ARG;
    return (int)cudaIpcCloseMemHandle(static_cast<char*>(ptr) - offset);
}

extern "C" int tcar_peer_fetch_rows(const int32_t* seq, const int32_t* label, const int32_t* neg, int B, int T, int Nn,
                                    const void* const* peers, const int32_t* row_bounds, int G, int self,
                                    float* table, void* stream) {
    if (B < 0 || T < 1 || Nn < 0 || G < 1 || G > TCAR_MAX_PEERS || self < 0 || self >= G || !peers || !row_bounds ||
        !table)
        return TCAR_ERR_ARG;
    const int n = B * T + B + B * Nn;
    if (n == 0) return 0;
    if (!seq || !label || (Nn > 0 && !neg)) return TCAR_ERR_ARG;
    PeerTable pt = {};
    for (int g = 0; g < G; ++g) {
        if (!peers[g] || row_bounds[g + 1] < row_bounds[g]) return TCAR_ERR_ARG;
        pt.base[g] = static_cast<const float*>(peers[g]);
    }
    for (int g = 0; g <= G; ++g) pt.bound[g] = row_bounds[g];
    pt.G = G;
    pt.self = self;
    launch_pdl(peer_fetch_rows_kernel, dim3((n + 7) / 8), dim3(256), 0, static_cast<cudaStream_t>(stream), seq, label,
               neg, B * T, B, n, pt, table);
    return (int)cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------
// Session groups of a catalog-sharded step: group g (rank g's sessions, n_rows[g] <= 512 of them; 0 = absent) is scored
// against the caller's item range with the single-group kernels; the loops live here so that the host pays one call per
// phase instead of one per group.  Strides are in ELEMENTS of the respective array.
extern "C" int tcar_score_fwd_groups(const void* q_bf16, long long q_stride, const float* c_ref, long long c_stride,
                                     const void* iext_bf16, void* e_out, long long e_stride, float* rowsum_part,
                                     long long part_stride, const int* n_rows, int groups, int n_items, int n_pad,
                                     int cluster, void* stream) {
    return tcar_score_fwd_groups_guarded(q_bf16, q_stride, c_ref, c_stride, iext_bf16, e_out, e_stride, rowsum_part,
                                         part_stride, nullptr, nullptr, n_rows, groups, n_items, n_pad, cluster, stream);
}

// With the softmax overflow guard (tcar_score_fwd_guarded): pass 1 = rowmax_part given (group g's block part_stride
// floats apart, like rowsum_part), pass 2 = rowmax given ([groups][512]; after tcar_rowmax_groups and, across ranks, an
// all-reduce(MAX) -- every rank must shift a session row by the same amount).
extern "C" int tcar_score_fwd_groups_guarded(const void* q_bf16, long long q_stride, const float* c_ref,
                                             long long c_stride, const void* iext_bf16, void* e_out, long long e_stride,
                                             float* rowsum_part, long long part_stride, float* rowmax_part,
                                             const float* rowmax, const int* n_rows, int groups, int n_items, int n_pad,
                                             int cluster, void* stream) {
    if (!n_rows || groups < 1) return TCAR_ERR_ARG;
    int present = 0;
    for (int g = 0; g < groups; ++g) present += n_rows[g] > 0;
    // several groups: one launch over all of them
    const bool multi = cluster == TCAR_CLUSTER_PAIR && groups <= TCAR_MAX_PEERS && (q_stride & 7) == 0 && present > 1;
    if (multi)
        return tcar_score_fwd_multi(q_bf16, q_stride, c_ref, c_stride, iext_bf16, e_out, e_stride, rowsum_part,
                                    part_stride, rowmax_part, rowmax, n_rows, groups, n_items, n_pad, stream);
    for (int g = 0; g < groups; ++g) {
        if (n_rows[g] <= 0) continue;
        const int rc = tcar_score_fwd_guarded(static_cast<const uint16_t*>(q_bf16) + g * q_stride, iext_bf16,
                                              c_ref + g * c_stride, static_cast<uint16_t*>(e_out) + g * e_stride,
                                              rowsum_part + g * part_stride, nullptr, nullptr,
                                              rowmax_part ? rowmax_part + g * part_stride : nullptr,
                                              rowmax ? rowmax + (size_t)g * TCAR_QROWS : nullptr, n_rows[g], n_items,
                                              n_pad, 0, cluster, stream);
        if (rc) return rc;
    }
    return 0;
}

extern "C" int tcar_score_bwd_q_groups(const void* e_bf16, long long e_stride, const void* iext_bf16, float* part,
                                       float* dq, long long dq_stride, const float* rowsum_part,
                                       long long part_stride, int n_tiles, const int* n_rows, int groups, int n_pad,
                                       void* stream) {
    if (!n_rows || groups < 1) return TCAR_ERR_ARG;
    int present = 0;
    for (int g = 0; g < groups; ++g) present += n_rows[g] > 0;
    // several groups: one launch over all of them (needs the groups' dQ blocks back to back and a part buffer of
    // tcar_score_bwd_q_multi_part_elems floats)
    const bool multi = present > 1 && groups <= 16 && dq_stride == (long long)TCAR_QROWS * TCAR_KEXT;
    if (multi) {
        const int rc = tcar_score_bwd_q_multi(e_bf16, e_stride, iext_bf16, part, dq, n_rows, groups, n_pad, stream);
        if (rc) return rc;
    }
    for (int g = 0; g < groups; ++g) {
        if (n_rows[g] <= 0) continue;
        float* dq_g = dq + g * dq_stride;
        int rc = 0;
        if (!multi) {
            rc = tcar_score_bwd_q(static_cast<const uint16_t*>(e_bf16) + g * e_stride, iext_bf16, part, dq_g,
                                  n_rows[g], n_pad, stream);
            if (rc) return rc;
        }
        // the zero pad column 639 of dQ carries the group's softmax partial sums through the same reduce-scatter
        if (rowsum_part) {
            rc = tcar_rowsum_finish(rowsum_part + g * part_stride, dq_g + (TCAR_KEXT - 1), TCAR_KEXT, n_tiles,
                                    n_rows[g], stream);
            if (rc) return rc;
        }
    }
    return 0;
}

extern "C" int tcar_score_bwd_i_groups(const void* e_bf16, long long e_stride, const void* qs_bf16, long long qs_stride,
                                       float* g_item, float* sq_partial, const int* n_rows, int groups, int n_items,
                                       int n_pad, void* stream) {
    if (!n_rows || groups < 1) return TCAR_ERR_ARG;
    // all groups concatenated along K in ONE launch, the gradient written once (score_bwd_i_tma_kernel<MULTI>); more
    // groups than that kernel takes: one launch per group with read-modify-write accumulation
    if (groups <= TCAR_MAX_PEERS)
        return tcar_score_bwd_i_multi(e_bf16, e_stride, qs_bf16, qs_stride, g_item, sq_partial, n_rows, groups, n_items,
                                      n_pad, stream);
    int done = 0, last = -1;
    for (int g = 0; g < groups; ++g)
        if (n_rows[g] > 0) last = g;
    for (int g = 0; g < groups; ++g) {
        if (n_rows[g] <= 0) continue;
        const int rc = tcar_score_bwd_i_acc(static_cast<const uint16_t*>(e_bf16) + g * e_stride,
                                            static_cast<const uint16_t*>(qs_bf16) + g * qs_stride, g_item,
                                            g == last ? sq_partial : nullptr, n_rows[g], n_items, n_pad, done > 0,
                                            stream);
        if (rc) return rc;
        ++done;
    }
    return 0;
}

extern "C" int tcar_scatter_add_rows_groups(const int32_t* ids, long long ids_stride, const float* payload,
                                            long long payload_stride, const float* item, float* g_item,
                                            int32_t* hash_keys, int32_t* hash_cnt, long long* hash_acc,
                                            int32_t* entry_slot, float* slot_sq, int hash_size, const int* n_rows,
                                            int groups, int T, int Nn, int row_lo, int row_hi, void* stream) {
    if (!n_rows || groups < 1 || !ids || !payload) return TCAR_ERR_ARG;
    for (int g = 0; g < groups; ++g) {
        const int B = n_rows[g];
        if (B <= 0) {
            // absent group: its block of per-slot norm corrections must not keep an earlier step's values
            if (slot_sq) {
                const cudaError_t e = cudaMemsetAsync(slot_sq + (size_t)g * hash_size, 0, sizeof(float) * hash_size,
                                                      static_cast<cudaStream_t>(stream));
                if (e != cudaSuccess) return (int)e;
            }
            continue;
        }
        // packed batch of rank g: [7*B*T idx | 2*B ctx | B label | B*Nn neg]; payload: [a_ic 512x500 | coef 512 | dXi]
        const int32_t* base = ids + g * ids_stride;
        const size_t M = (size_t)B * T;
        const float* pay = payload + g * payload_stride;
        const int rc = tcar_scatter_add_rows_range(
            base, base + 7 * M + 2 * (size_t)B, Nn > 0 ? base + 7 * M + 3 * (size_t)B : nullptr,
            pay + TCAR_QROWS * TCAR_XW + TCAR_QROWS, pay, pay + TCAR_QROWS * TCAR_XW, item, g_item, hash_keys, hash_cnt,
            hash_acc, entry_slot, slot_sq ? slot_sq + (size_t)g * hash_size : nullptr, hash_size, B, T, Nn, row_lo,
            row_hi, stream);
        if (rc) return rc;
    }
    return 0;
}
