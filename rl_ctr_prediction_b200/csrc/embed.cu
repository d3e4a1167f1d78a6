// embed.cu -- K1 fused gather + first-order + FM second-order forward, the plain row gather,
// and K5 the Feature_Embedding RL state encoder.  sm_100a.
//
// Thread mapping (all three kernels): one warp per sample, LPR lanes per gathered row, each
// lane reading one aligned float4 (128-bit) chunk of the fused row (K1 also takes LPR = 16 for the
// 36-float rows of D = 32 with a first-order column: lanes 9..15 of a row slot idle).  For the default
// latent_dims=10 the row is [w, v0..v9, pad] = 12 floats = 3 chunks -> LPR=4, 8 rows per warp
// request, the 15 fields of a sample in two requests.  Lanes of one row hit one or two 32 B
// sectors in a single request (1.25 L1 wavefronts/row instead of 3 for a lane-per-row map).
#include <cstdlib>

#include "common.cuh"

namespace rlctr {

// id of gathered element e = b * fields + f; ids == NULL: the rows are already in sample order (rlctr_rows_lookup's `gathered`)
__device__ __forceinline__ int64_t id_at(const int64_t* __restrict__ ids, int64_t e) { return ids ? __ldg(ids + e) : e; }

// ------------------------------------------------------------------------------------------
// K1
// ------------------------------------------------------------------------------------------
template <int LPR>
__global__ void __launch_bounds__(256, 5)
embed_fwd_kernel(const int64_t* __restrict__ ids, const float* __restrict__ tab, const __grid_constant__ ShardView sv, int64_t n_rows, int pitch,
                 int rs, int lin_col, int emb_col, int dim, const float* __restrict__ bias,
                 float* __restrict__ logit, float* __restrict__ pctr, int64_t pctr_stride,
                 float* __restrict__ sums, float* __restrict__ rows_out, int64_t rows_pitch,
                 int64_t batch, int fields, int flags) {
    constexpr int RPW = 32 / LPR;                   // rows per warp request
    const int lane = threadIdx.x & 31;
    const int c = lane % LPR;                       // chunk of the row this lane owns
    const int g = lane / LPR;                       // row slot within the request
    const int col0 = 4 * c;
    const bool chunk_on = col0 < rs;
    const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const bool fm = (flags & RLCTR_FM_TERM) != 0;

    bool is_emb[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) is_emb[k] = (col0 + k >= emb_col) && (col0 + k < emb_col + dim);
    const float b0 = bias ? __ldg(bias) : 0.f;

    // software pipeline: the ids of this warp's NEXT sample are fetched while the rows of the
    // current one are in flight (two dependent DRAM latencies -> one on the critical path).
    int64_t b = warp0;
    int64_t id_a = -1, id_b = -1;                   // first two row slots of the next sample
    if (b < batch && chunk_on) {
        if (g < fields) id_a = id_at(ids, b * fields + g);
        if (g + RPW < fields) id_b = id_at(ids, b * fields + g + RPW);
    }
    for (; b < batch; b += nwarps) {
        const int64_t cur_a = id_a, cur_b = id_b;
        const int64_t nb = b + nwarps;
        id_a = -1; id_b = -1;
        if (nb < batch && chunk_on) {
            if (g < fields) id_a = id_at(ids, nb * fields + g);
            if (g + RPW < fields) id_b = id_at(ids, nb * fields + g + RPW);
        }
        float4 s = f4zero();
        float q = 0.f;
        for (int f0 = 0; f0 < fields; f0 += 2 * RPW) {
            const int fa = f0 + g, fb = f0 + RPW + g;
            int64_t ia = -1, ib = -1;
            if (f0 == 0) { ia = cur_a; ib = cur_b; }
            else if (chunk_on) {
                if (fa < fields) ia = id_at(ids, b * fields + fa);
                if (fb < fields) ib = id_at(ids, b * fields + fb);
            }
            float4 ra = f4zero(), rb = f4zero();
            const bool oka = (uint64_t)ia < (uint64_t)n_rows, okb = (uint64_t)ib < (uint64_t)n_rows;
            if (oka) ra = ldg4_once(row_ptr(tab, sv, ia, pitch) + col0);
            if (okb) rb = ldg4_once(row_ptr(tab, sv, ib, pitch) + col0);
            s = f4add(s, f4add(ra, rb));
            if (fm) {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (is_emb[k]) { float x = f4get(ra, k), y = f4get(rb, k); q = fmaf(x, x, q); q = fmaf(y, y, q); }
            }
            if (rows_out) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (!is_emb[k]) continue;
                    const int d = col0 + k - emb_col;
                    if (chunk_on && fa < fields) rows_out[b * rows_pitch + fa * dim + d] = f4get(ra, k);
                    if (chunk_on && fb < fields) rows_out[b * rows_pitch + fb * dim + d] = f4get(rb, k);
                }
            }
        }
        // sum over the F rows: lanes owning the same chunk sit LPR apart
#pragma unroll
        for (int off = LPR; off < 32; off <<= 1) {
            s = f4add(s, shfl_xor4(s, off));
            q += __shfl_xor_sync(RLCTR_FULL, q, off);
        }
        float t = 0.f;
        if (fm) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (is_emb[k]) { float x = f4get(s, k); t = fmaf(x, x, t); }
            t -= q;                                  // sum over this chunk of (S_d^2 - sum_f v_d^2)
#pragma unroll
            for (int off = 1; off < LPR; off <<= 1) t += __shfl_xor_sync(RLCTR_FULL, t, off);
        }
        float first = 0.f;
        if (lin_col >= 0) {
            const int src = lin_col >> 2;            // lane (group 0) holding the linear column
            const float4 sv = make_float4(__shfl_sync(RLCTR_FULL, s.x, src), __shfl_sync(RLCTR_FULL, s.y, src),
                                          __shfl_sync(RLCTR_FULL, s.z, src), __shfl_sync(RLCTR_FULL, s.w, src));
            first = f4get(sv, lin_col & 3);
        }
        if (lane == 0) {
            const float z = fmaf(0.5f, t, b0 + first);    // explicit contraction: group_fwd_kernel reproduces it bit for bit
            if (logit) logit[b] = z;
            if (pctr) pctr[b * pctr_stride] = sigmoidf_ref(z);
        }
        if (sums && g == 0 && chunk_on) st4(sums + b * rs + col0, s);
    }
}

// ------------------------------------------------------------------------------------------
// K1 over a CO-LOCATED record (rlctr_group_fwd): one gather per (sample, field) feeds every member model.
// Warp per sample, 8 lanes per joint row (one 128-bit chunk each, up to 128 B = one DRAM line per row), four row slots per
// request, the 16 fields of a block in four requests that are all issued before any is consumed.  The reduction trees are
// those of embed_fwd_kernel<4> on the member's stand-alone table -- slot j of that kernel holds rows j and j + 8, here row
// slot g holds (g, g + 8) in its A accumulators and (g + 4, g + 12) in its B accumulators, and the butterflies pair them in
// the same order -- so a member's column sums, sum of squares and logit are bit-identical to the stand-alone kernel's.
// ------------------------------------------------------------------------------------------
struct GroupFwdView {
    int n;
    int lin_col[RLCTR_GROUP_MAX], emb_col[RLCTR_GROUP_MAX], dim[RLCTR_GROUP_MAX], fm[RLCTR_GROUP_MAX];
    const float* bias[RLCTR_GROUP_MAX];
    float* logit[RLCTR_GROUP_MAX];
    float* pctr[RLCTR_GROUP_MAX];
    int64_t pctr_stride[RLCTR_GROUP_MAX];
    float* rows_out[RLCTR_GROUP_MAX];
    int rows_pitch[RLCTR_GROUP_MAX];
    int tile_off[RLCTR_GROUP_MAX];           // float offset of the member's tower-input tile in the warp's shared memory, -1 = none
    int chunk_member[RLCTR_GROUP_CHUNKS];    // vector member whose latent columns chunk c holds, -1 = none (one member per chunk)
    int lpr[RLCTR_GROUP_MAX];                // lanes per row of the member's stand-alone table (embed_fwd_kernel<LPR>): 4, 8 or 16
    int warp_floats;                         // shared memory per warp: 32 (column sums) + 8 (per-chunk t) + the tiles; wide records:
                                             // per sample of the warp, 128 (column sums) + 32 (per-chunk t) + the tiles
};
template <int LD>
__device__ __forceinline__ float4 group_ld(const float* p) {
    if (LD == 1) return ldg4(p);                     // default: L1 allocation, L2 promotion as the hardware sees fit
    if (LD == 2) {                                   // no L1 allocation, fill the whole 128-byte line (the row spans both halves)
        float4 v;
        asm volatile("ld.global.nc.L1::no_allocate.L2::128B.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
        return v;
    }
    return ldg4_once(p);
}
// per-lane constants of the group kernel
struct GroupLaneFwd {
    int c, g, col0;
    bool chunk_on, m_fm;
    int m_dim;
    int dk[4];                                      // latent index of column col0 + k in the chunk's vector member, -1 = none
    float* tile;                                    // that member's tower-input tile in the warp's shared memory, or NULL
};
__device__ __forceinline__ int group_field(int g, int u) { return g + ((u & 1) ? 8 : 0) + ((u & 2) ? 4 : 0); }
// the ids of one 16-field block of sample b: fields f0 + (g, g + 8, g + 4, g + 12)
__device__ __forceinline__ void group_ids(int64_t id[4], const int64_t* __restrict__ ids, int64_t b, int f0, int fields,
                                          const GroupLaneFwd& L, bool live) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int f = f0 + group_field(L.g, u);
        id[u] = -1;
        if (live && L.chunk_on && f < fields) id[u] = __ldg(ids + b * fields + f);
    }
}
// unconditional, straight-line loads, all four back to back (an id load or a branch between two row loads makes ptxas wait for
// the earlier row and the four DRAM round trips of a sample serialise): an out-of-range id, or an inactive chunk lane, reads a
// valid address it shares with a neighbour and drops the result
template <int LD>
__device__ __forceinline__ void group_issue(float4 r[4], const int64_t id[4], const float* __restrict__ tab, const ShardView& sv,
                                            int64_t n_rows, int pitch, const GroupLaneFwd& L) {
    const float* ptr[4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
        ptr[u] = row_ptr(tab, sv, (uint64_t)id[u] < (uint64_t)n_rows ? id[u] : 0, pitch) + (L.chunk_on ? L.col0 : 0);
#pragma unroll
    for (int u = 0; u < 4; ++u) r[u] = group_ld<LD>(ptr[u]);
}
__device__ __forceinline__ void group_accumulate(float4 r[4], const int64_t id[4], int64_t n_rows, int f0, int fields,
                                                 const GroupLaneFwd& L, float4& sA, float4& sB, float& qA, float& qB) {
#pragma unroll
    for (int u = 0; u < 4; ++u)
        if (!(L.chunk_on && (uint64_t)id[u] < (uint64_t)n_rows)) r[u] = f4zero();
    sA = f4add(sA, f4add(r[0], r[1]));               // slot g of the stand-alone kernel: rows (g, g + 8)
    sB = f4add(sB, f4add(r[2], r[3]));               // slot g + 4: rows (g + 4, g + 12)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (L.dk[k] < 0) continue;
        if (L.m_fm) {
            float x = f4get(r[0], k), y = f4get(r[1], k);
            qA = fmaf(x, x, qA); qA = fmaf(y, y, qA);
            x = f4get(r[2], k); y = f4get(r[3], k);
            qB = fmaf(x, x, qB); qB = fmaf(y, y, qB);
        }
        if (L.tile) {                                // tower input: staged in shared memory, written out as whole rows later
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int f = f0 + group_field(L.g, u);
                if (f < fields) L.tile[f * L.m_dim + L.dk[k]] = f4get(r[u], k);
            }
        }
    }
}
// butterflies, per-member logits (lane m finishes member m from the staged column sums / per-chunk t), tower rows, saved sums
__device__ __forceinline__ void group_finish(float4 sA, float4 sB, float qA, float qB, const GroupLaneFwd& L, float* wsm,
                                             const GroupFwdView& gv, float* __restrict__ sums, int sums_pitch, int64_t b, int fields) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int off = 8; off < 32; off <<= 1) {
        sA = f4add(sA, shfl_xor4(sA, off));
        sB = f4add(sB, shfl_xor4(sB, off));
        qA += __shfl_xor_sync(RLCTR_FULL, qA, off);
        qB += __shfl_xor_sync(RLCTR_FULL, qB, off);
    }
    const float4 s = f4add(sA, sB);
    const float q = qA + qB;
    float t = 0.f;
    if (L.m_fm) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (L.dk[k] >= 0) { float x = f4get(s, k); t = fmaf(x, x, t); }
    }
    t -= q;                                          // this chunk's sum of (S_d^2 - sum_f v_d^2)
    if (L.g == 0) {
        *reinterpret_cast<float4*>(wsm + L.col0) = s;
        wsm[32 + L.c] = t;
        if (sums && L.chunk_on) st4(sums + b * sums_pitch + L.col0, s);
    }
    __syncwarp();
    if (lane < gv.n) {
        const int m = lane;
        float tm = 0.f;
        if (gv.fm[m] && gv.dim[m] > 0) {             // ((t0 + t1) + (t2 + t3)) over the member's chunks: the stand-alone butterfly
            const int base = gv.emb_col[m] >> 2, last = (gv.emb_col[m] + gv.dim[m] - 1) >> 2;
            const float t0 = wsm[32 + base];
            const float t1 = base + 1 <= last ? wsm[32 + base + 1] : 0.f;
            const float t2 = base + 2 <= last ? wsm[32 + base + 2] : 0.f;
            const float t3 = base + 3 <= last ? wsm[32 + base + 3] : 0.f;
            tm = (t0 + t1) + (t2 + t3);
        }
        const float first = gv.lin_col[m] >= 0 ? wsm[gv.lin_col[m]] : 0.f;
        const float b0 = gv.bias[m] ? __ldg(gv.bias[m]) : 0.f;
        const float z = fmaf(0.5f, tm, b0 + first);
        if (gv.logit[m]) gv.logit[m][b] = z;
        if (gv.pctr[m]) gv.pctr[m][b * gv.pctr_stride[m]] = sigmoidf_ref(z);
    }
#pragma unroll
    for (int m = 0; m < RLCTR_GROUP_MAX; ++m) {      // tower inputs: whole rows, 16 bytes per lane
        if (m < gv.n && gv.tile_off[m] >= 0) {
            const float* src = wsm + gv.tile_off[m];
            float* dst = gv.rows_out[m] + b * (int64_t)gv.rows_pitch[m];
            if ((gv.rows_pitch[m] & 3) == 0) {
                for (int i = lane; 4 * i < fields * gv.dim[m]; i += 32) st4(dst + 4 * i, *reinterpret_cast<const float4*>(src + 4 * i));
            } else {
                for (int i = lane; i < fields * gv.dim[m]; i += 32) dst[i] = src[i];
            }
        }
    }
    __syncwarp();                                    // the next sample overwrites the staging area
}
template <int LD, bool ONE>      // ONE: fields <= 16, a single block of row loads per sample: software-pipelined
__global__ void __launch_bounds__(256, 3)
group_fwd_kernel(const int64_t* __restrict__ ids, const float* __restrict__ tab, const __grid_constant__ ShardView sv, int64_t n_rows,
                 int pitch, int rs, const __grid_constant__ GroupFwdView gv, float* __restrict__ sums, int sums_pitch, int64_t batch,
                 int fields) {
    extern __shared__ __align__(16) float gsm[];
    const int lane = threadIdx.x & 31;
    GroupLaneFwd L;
    L.c = lane & 7;                                 // chunk of the joint row this lane owns
    L.g = lane >> 3;                                // row slot within the request (0..3)
    L.col0 = 4 * L.c;
    L.chunk_on = L.col0 < rs;
    float* wsm = gsm + (threadIdx.x >> 5) * gv.warp_floats;          // this warp's [sums 32 | t 8 | tower tiles]
    const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    // the vector member (if any) whose latent columns this lane's chunk holds: they enter the sum of squares when the member
    // has the FM term, and the member's tower-input tile when it has a dense tail
    const int mem = L.chunk_on ? gv.chunk_member[L.c] : -1;
    const int m_emb = mem >= 0 ? gv.emb_col[mem] : 0;
    L.m_dim = mem >= 0 ? gv.dim[mem] : 0;
    L.m_fm = mem >= 0 && gv.fm[mem] != 0;
    L.tile = (mem >= 0 && gv.tile_off[mem] >= 0) ? wsm + gv.tile_off[mem] : nullptr;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int d = L.col0 + k - m_emb;
        L.dk[k] = (mem >= 0 && d >= 0 && d < L.m_dim) ? d : -1;
    }
    for (int i = lane; i < gv.warp_floats; i += 32) wsm[i] = 0.f;   // tile padding columns are copied out with the rows
    __syncwarp();

    int64_t b = warp0;
    if (b >= batch) return;
    if (ONE) {
        // Two-deep software pipeline: while sample b is reduced (shuffles, shared-memory staging: a chain of a few hundred
        // dependent instructions), the rows of sample b + nwarps are already in flight and the ids of b + 2 nwarps are being
        // fetched -- the warp always has 16 row requests outstanding instead of a burst followed by a long quiet phase.
        int64_t id_c[4], id_n[4];
        float4 r_c[4], r_n[4];
        group_ids(id_c, ids, b, 0, fields, L, true);
        group_issue<LD>(r_c, id_c, tab, sv, n_rows, pitch, L);
        group_ids(id_n, ids, b + nwarps, 0, fields, L, b + nwarps < batch);
        for (; b < batch; b += nwarps) {
            const bool more = b + nwarps < batch;                     // warp-uniform
            if (more) group_issue<LD>(r_n, id_n, tab, sv, n_rows, pitch, L);
            int64_t id_nn[4];
            group_ids(id_nn, ids, b + 2 * nwarps, 0, fields, L, b + 2 * nwarps < batch);
            float4 sA = f4zero(), sB = f4zero();
            float qA = 0.f, qB = 0.f;
            group_accumulate(r_c, id_c, n_rows, 0, fields, L, sA, sB, qA, qB);
            group_finish(sA, sB, qA, qB, L, wsm, gv, sums, sums_pitch, b, fields);
#pragma unroll
            for (int u = 0; u < 4; ++u) { r_c[u] = r_n[u]; id_c[u] = id_n[u]; id_n[u] = id_nn[u]; }
        }
    } else {
        for (; b < batch; b += nwarps) {
            float4 sA = f4zero(), sB = f4zero();
            float qA = 0.f, qB = 0.f;
            for (int f0 = 0; f0 < fields; f0 += 16) {
                int64_t id[4];
                float4 r[4];
                group_ids(id, ids, b, f0, fields, L, true);
                group_issue<LD>(r, id, tab, sv, n_rows, pitch, L);
                group_accumulate(r, id, n_rows, f0, fields, L, sA, sB, qA, qB);
            }
            group_finish(sA, sB, qA, qB, L, wsm, gv, sums, sums_pitch, b, fields);
        }
    }
}

// ------------------------------------------------------------------------------------------
// K1 over a WIDE co-located record: joint rows of up to four lines (128 floats), or members whose stand-alone rows are wider than
// 16 floats.  W lanes per joint row, one 16-byte chunk each (W = 16: two samples per warp; W = 32: one), and each lane walks ALL
// fields of its sample, 16 row loads in flight per block of fields.  A lane reproduces in registers the reduction tree of
// embed_fwd_kernel<LPR> for the stand-alone table of the member that owns its chunk: RPW = 32 / LPR row slots, slot j adds
// (row f0 + j + row f0 + RPW + j) per block of 2 RPW fields, then the slots pair as the butterflies xor 1, 2, .. RPW / 2 do; the
// per-chunk FM terms pair over the member's LPR chunks.  Column sums, sums of squares and logits are bit-identical to the
// stand-alone kernel's for every member, whatever its row width.
// ------------------------------------------------------------------------------------------
template <int RPW>
__device__ __forceinline__ void wide_block(const float4 (&r)[16], int f0, int fields, const int (&dk)[4], bool fm, float4 (&s)[8],
                                           float (&q)[8]) {
#pragma unroll
    for (int h = 0; h < 16; h += 2 * RPW) {
        if (f0 + h >= fields) break;                 // the stand-alone loop stops at the last field
#pragma unroll
        for (int j = 0; j < RPW; ++j) {
            const float4 ra = r[h + j], rb = r[h + RPW + j];
            s[j] = f4add(s[j], f4add(ra, rb));
            if (fm) {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (dk[k] >= 0) { float x = f4get(ra, k), y = f4get(rb, k); q[j] = fmaf(x, x, q[j]); q[j] = fmaf(y, y, q[j]); }
            }
        }
    }
}
template <int RPW>
__device__ __forceinline__ void wide_slots(float4 (&s)[8], float (&q)[8]) {
#pragma unroll
    for (int off = 1; off < RPW; off <<= 1) {
#pragma unroll
        for (int j = 0; j < RPW; j += 2 * off) { s[j] = f4add(s[j], s[j + off]); q[j] += q[j + off]; }
    }
}
template <int W>
__global__ void __launch_bounds__(256)
group_fwd_wide_kernel(const int64_t* __restrict__ ids, const float* __restrict__ tab, const __grid_constant__ ShardView sv,
                      int64_t n_rows, int pitch, int rs, const __grid_constant__ GroupFwdView gv, float* __restrict__ sums,
                      int sums_pitch, int64_t batch, int fields) {
    constexpr int SPW = 32 / W;                      // samples per warp
    constexpr int SLOT = 128 + RLCTR_GROUP_CHUNKS;   // staging of one sample: column sums | per-chunk t (the tiles follow)
    extern __shared__ __align__(16) float gsm[];
    const int lane = threadIdx.x & 31;
    const int c = lane % W, slot = lane / W, col0 = 4 * c;
    const bool chunk_on = col0 < rs;
    const int slot_floats = gv.warp_floats / SPW;
    float* wsm = gsm + (threadIdx.x >> 5) * gv.warp_floats + slot * slot_floats;
    const int mem = chunk_on ? gv.chunk_member[c] : -1;
    const int m_dim = mem >= 0 ? gv.dim[mem] : 0;
    const bool m_fm = mem >= 0 && gv.fm[mem] != 0;
    const int form = mem >= 0 ? gv.lpr[mem] : 4;    // a chunk without a vector member (LR's own): the 16-float form
    float* tile = (mem >= 0 && gv.tile_off[mem] >= 0) ? wsm + gv.tile_off[mem] : nullptr;
    int dk[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int d = col0 + k - (mem >= 0 ? gv.emb_col[mem] : 0);
        dk[k] = (mem >= 0 && d >= 0 && d < m_dim) ? d : -1;
    }
    for (int i = lane; i < gv.warp_floats; i += 32) gsm[(threadIdx.x >> 5) * gv.warp_floats + i] = 0.f;
    __syncwarp();
    const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t bw = warp0 * SPW; bw < batch; bw += nwarps * SPW) {        // warp-uniform trip count
        const int64_t b = bw + slot;
        const bool live = b < batch;
        float4 s[8];
        float q[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) { s[j] = f4zero(); q[j] = 0.f; }
        for (int f0 = 0; f0 < fields; f0 += 16) {
            const int fl = f0 + (lane & 15);
            const int64_t my_id = (live && fl < fields) ? __ldg(ids + b * fields + fl) : -1;
            float4 r[16];
            unsigned ok = 0;                             // bit u: field f0 + u has a row
#pragma unroll
            for (int u = 0; u < 16; ++u) {               // unconditional loads, dropped below (see group_issue)
                const int64_t id = __shfl_sync(RLCTR_FULL, my_id, slot * W + u);
                const bool in = (uint64_t)id < (uint64_t)n_rows;
                ok |= (unsigned)(in && chunk_on) << u;
                r[u] = ldg4(row_ptr(tab, sv, in ? id : 0, pitch) + (chunk_on ? col0 : 0));
            }
#pragma unroll
            for (int u = 0; u < 16; ++u) {
                if (!((ok >> u) & 1)) r[u] = f4zero();
                if (tile && f0 + u < fields) {
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (dk[k] >= 0) tile[(f0 + u) * m_dim + dk[k]] = f4get(r[u], k);
                }
            }
            if (form == 4) wide_block<8>(r, f0, fields, dk, m_fm, s, q);
            else if (form == 8) wide_block<4>(r, f0, fields, dk, m_fm, s, q);
            else wide_block<2>(r, f0, fields, dk, m_fm, s, q);
        }
        if (form == 4) wide_slots<8>(s, q);
        else if (form == 8) wide_slots<4>(s, q);
        else wide_slots<2>(s, q);
        float t = 0.f;
        if (m_fm) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (dk[k] >= 0) { float x = f4get(s[0], k); t = fmaf(x, x, t); }
        }
        t -= q[0];                                   // this chunk's sum of (S_d^2 - sum_f v_d^2)
        if (chunk_on) {
            *reinterpret_cast<float4*>(wsm + col0) = s[0];
            wsm[128 + c] = t;
            if (sums && live) st4(sums + b * sums_pitch + col0, s[0]);
        }
        __syncwarp();
        if (c < gv.n && live) {                      // lane m of the sample finishes member m
            const int m = c;
            float tm = 0.f;
            if (gv.fm[m] && gv.dim[m] > 0) {         // the member's chunks paired as its stand-alone butterfly xor 1 .. LPR / 2
                const int base = gv.emb_col[m] >> 2, last = (gv.emb_col[m] + gv.dim[m] - 1) >> 2, L = gv.lpr[m];
                float v[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) v[i] = (i < L && base + i <= last) ? wsm[128 + base + i] : 0.f;
#pragma unroll
                for (int w = 1; w < 16; w <<= 1) {
#pragma unroll
                    for (int i = 0; i < 16; i += 2 * w)
                        if (w < L) v[i] = v[i] + v[i + w];
                }
                tm = v[0];
            }
            const float first = gv.lin_col[m] >= 0 ? wsm[gv.lin_col[m]] : 0.f;
            const float b0 = gv.bias[m] ? __ldg(gv.bias[m]) : 0.f;
            const float z = fmaf(0.5f, tm, b0 + first);
            if (gv.logit[m]) gv.logit[m][b] = z;
            if (gv.pctr[m]) gv.pctr[m][b * gv.pctr_stride[m]] = sigmoidf_ref(z);
        }
        if (live) {
#pragma unroll
            for (int m = 0; m < RLCTR_GROUP_MAX; ++m) {      // tower inputs: whole rows, 16 bytes per lane
                if (m < gv.n && gv.tile_off[m] >= 0) {
                    const float* src = wsm + gv.tile_off[m];
                    float* dst = gv.rows_out[m] + b * (int64_t)gv.rows_pitch[m];
                    if ((gv.rows_pitch[m] & 3) == 0) {
                        for (int i = c; 4 * i < fields * gv.dim[m]; i += W) st4(dst + 4 * i, *reinterpret_cast<const float4*>(src + 4 * i));
                    } else {
                        for (int i = c; i < fields * gv.dim[m]; i += W) dst[i] = src[i];
                    }
                }
            }
        }
        __syncwarp();                                // the next sample overwrites the staging area
    }
}

// LR table: one float per row (row_stride == 1).  Lane f gathers w[x_f]; warp-sum.
__global__ void __launch_bounds__(256)
embed_fwd_scalar_kernel(const int64_t* __restrict__ ids, const float* __restrict__ tab, const __grid_constant__ ShardView sv, int64_t n_rows, int pitch,
                        const float* __restrict__ bias, float* __restrict__ logit,
                        float* __restrict__ pctr, int64_t pctr_stride, float* __restrict__ sums,
                        int64_t batch, int fields) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const float b0 = bias ? __ldg(bias) : 0.f;
    for (int64_t b = warp0; b < batch; b += nwarps) {
        float s = 0.f;
        for (int f = lane; f < fields; f += 32) {
            const int64_t id = id_at(ids, b * fields + f);
            if ((uint64_t)id < (uint64_t)n_rows) s += ldg1_once(row_ptr(tab, sv, id, pitch));
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(RLCTR_FULL, s, off);
        if (lane == 0) {
            const float z = b0 + s;
            if (logit) logit[b] = z;
            if (pctr) pctr[b * pctr_stride] = sigmoidf_ref(z);
            if (sums) sums[b] = s;
        }
    }
}

// ------------------------------------------------------------------------------------------
// plain gather
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gather_rows_kernel(const int64_t* __restrict__ ids, int64_t n, const float* __restrict__ tab,
                   int64_t n_rows, int pitch, int rs, float* __restrict__ out) {
    const int chunks = rs >> 2;
    const int64_t total = n * chunks;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t k = t / chunks;
        const int c = (int)(t - k * chunks);
        const int64_t id = __ldg(ids + k);
        float4 r = f4zero();
        if ((uint64_t)id < (uint64_t)n_rows) r = ldg4(tab + id * pitch + 4 * c);
        st4_stream(out + k * rs + 4 * c, r);
    }
}
__global__ void __launch_bounds__(256)
gather_rows_scalar_kernel(const int64_t* __restrict__ ids, int64_t n, const float* __restrict__ tab,
                          int64_t n_rows, int pitch, float* __restrict__ out) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n;
         t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t id = __ldg(ids + t);
        out[t] = ((uint64_t)id < (uint64_t)n_rows) ? __ldg(tab + id * pitch) : 0.f;
    }
}

// ------------------------------------------------------------------------------------------
// K5  Feature_Embedding: gather, stage the F latent vectors of the sample in shared memory
// (F*D contiguous floats == the second block of the output row), P pairwise dots from smem.
// ------------------------------------------------------------------------------------------
template <int LPR>
__global__ void __launch_bounds__(128)
featemb_fwd_kernel(const int64_t* __restrict__ ids, const float* __restrict__ tab, int64_t n_rows, int pitch,
                   int rs, int emb_col, int dim, float* __restrict__ out, int64_t out_stride,
                   int64_t batch, int fields) {
    constexpr int RPW = 32 / LPR;
    extern __shared__ float smem[];
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nw = blockDim.x >> 5;
    const int fd = fields * dim;
    const int npair = fields * (fields - 1) / 2;
    float* stage = smem + wib * fd;
    unsigned char* pi = reinterpret_cast<unsigned char*>(smem + nw * fd);
    unsigned char* pj = pi + npair;
    for (int i = threadIdx.x; i < fields - 1; i += blockDim.x) {
        int base = i * fields - i * (i + 1) / 2;     // pairs (i, i+1..F-1), Feature_embedding.py:40-43
        for (int j = i + 1; j < fields; ++j) { pi[base + j - i - 1] = (unsigned char)i; pj[base + j - i - 1] = (unsigned char)j; }
    }
    __syncthreads();
    const int c = lane % LPR, g = lane / LPR, col0 = 4 * c;
    const bool chunk_on = col0 < rs;
    const int64_t warp0 = (int64_t)blockIdx.x * nw + wib;
    const int64_t nwarps = (int64_t)gridDim.x * nw;
    for (int64_t b = warp0; b < batch; b += nwarps) {
        for (int f0 = 0; f0 < fields; f0 += 2 * RPW) {
            const int fa = f0 + g, fb = f0 + RPW + g;
            int64_t ia = -1, ib = -1;
            if (chunk_on && fa < fields) ia = __ldg(ids + b * fields + fa);
            if (chunk_on && fb < fields) ib = __ldg(ids + b * fields + fb);
            float4 ra = f4zero(), rb = f4zero();
            if ((uint64_t)ia < (uint64_t)n_rows) ra = ldg4_once(tab + ia * pitch + col0);
            if ((uint64_t)ib < (uint64_t)n_rows) rb = ldg4_once(tab + ib * pitch + col0);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int d = col0 + k - emb_col;
                if (d < 0 || d >= dim || !chunk_on) continue;
                if (fa < fields) stage[fa * dim + d] = f4get(ra, k);
                if (fb < fields) stage[fb * dim + d] = f4get(rb, k);
            }
        }
        __syncwarp();
        float* o = out + b * out_stride;
        for (int p = lane; p < npair; p += 32) {
            const float* vi = stage + pi[p] * dim;
            const float* vj = stage + pj[p] * dim;
            float acc = 0.f;
            for (int d = 0; d < dim; ++d) acc += vi[d] * vj[d];    // mul then sum over d, in d order
            __stcs(o + p, acc);
        }
        for (int i = lane; i < fd; i += 32) __stcs(o + npair + i, stage[i]);
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// Pairwise inner products over already-gathered rows (InnerPNN, p_model.py:178-198): the tower input
// [E (F*D) | ip (P)] (or [ip | E], the Feature_Embedding order) and its backward
//     d E[i] = g_E[i] + sum_{j != i} g_ip[pair(i,j)] * E[j]
// Warp per sample; E and g_ip are staged in shared memory; pair index by a byte table.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void pair_tables(unsigned char* pi, unsigned char* pj, unsigned char* pidx, int fields) {
    for (int i = threadIdx.x; i < fields; i += blockDim.x) {
        const int base = i * fields - i * (i + 1) / 2;       // pairs (i, i+1..F-1) in the reference's order
        for (int j = i + 1; j < fields; ++j) {
            const int p = base + j - i - 1;
            if (pi) { pi[p] = (unsigned char)i; pj[p] = (unsigned char)j; }
            if (pidx) { pidx[i * fields + j] = (unsigned char)p; pidx[j * fields + i] = (unsigned char)p; }
        }
    }
}
__global__ void __launch_bounds__(128)
pairdots_fwd_kernel(const float* __restrict__ rows, int64_t ld_rows, float* __restrict__ out, int64_t ld_out, int64_t batch,
                    int fields, int dim, int ip_first) {
    extern __shared__ float smem[];
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int fd = fields * dim, npair = fields * (fields - 1) / 2;
    float* stage = smem + wib * fd;
    unsigned char* pi = reinterpret_cast<unsigned char*>(smem + nw * fd);
    unsigned char* pj = pi + npair;
    pair_tables(pi, pj, nullptr, fields);
    __syncthreads();
    const int e_off = ip_first ? npair : 0, ip_off = ip_first ? 0 : fd;
    for (int64_t b = (int64_t)blockIdx.x * nw + wib; b < batch; b += (int64_t)gridDim.x * nw) {
        const float* r = rows + b * ld_rows;
        float* o = out + b * ld_out;
        for (int i = lane; i < fd; i += 32) { const float v = __ldg(r + i); stage[i] = v; o[e_off + i] = v; }
        __syncwarp();
        for (int p = lane; p < npair; p += 32) {
            const float* vi = stage + pi[p] * dim;
            const float* vj = stage + pj[p] * dim;
            float acc = 0.f;
            for (int d = 0; d < dim; ++d) acc += vi[d] * vj[d];      // mul then sum over d, in d order
            o[ip_off + p] = acc;
        }
        __syncwarp();
    }
}
__global__ void __launch_bounds__(128)
pairdots_bwd_kernel(const float* __restrict__ rows, int64_t ld_rows, const float* __restrict__ gout, int64_t ld_g,
                    float* __restrict__ grows, int64_t ld_grows, int64_t batch, int fields, int dim, int ip_first) {
    extern __shared__ float smem[];
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int fd = fields * dim, npair = fields * (fields - 1) / 2;
    float* stage = smem + wib * (fd + npair);
    float* gip = stage + fd;
    unsigned char* pidx = reinterpret_cast<unsigned char*>(smem + nw * (fd + npair));
    pair_tables(nullptr, nullptr, pidx, fields);
    __syncthreads();
    const int e_off = ip_first ? npair : 0, ip_off = ip_first ? 0 : fd;
    for (int64_t b = (int64_t)blockIdx.x * nw + wib; b < batch; b += (int64_t)gridDim.x * nw) {
        const float* r = rows + b * ld_rows;
        const float* g = gout + b * ld_g;
        for (int i = lane; i < fd; i += 32) stage[i] = __ldg(r + i);
        for (int p = lane; p < npair; p += 32) gip[p] = __ldg(g + ip_off + p);
        __syncwarp();
        for (int t = lane; t < fd; t += 32) {
            const int i = t / dim, d = t - i * dim;
            const unsigned char* prow = pidx + i * fields;
            float a0 = __ldg(g + e_off + t), a1 = 0.f;                  // two chains: a string of dependent LDS -> FMA otherwise
            int j = 0;
            for (; j + 1 < fields; j += 2) {
                if (j != i) a0 = fmaf(gip[prow[j]], stage[j * dim + d], a0);
                if (j + 1 != i) a1 = fmaf(gip[prow[j + 1]], stage[(j + 1) * dim + d], a1);
            }
            if (j < fields && j != i) a0 = fmaf(gip[prow[j]], stage[j * dim + d], a0);
            grows[b * ld_grows + t] = a0 + a1;
        }
        __syncwarp();
    }
}

static int grid_for_warps(int64_t items, int warps_per_block, int blocks_per_sm) {
    int64_t want = (items + warps_per_block - 1) / warps_per_block;
    int64_t cap = (int64_t)RLCTR_SMS * blocks_per_sm;
    if (want < 1) want = 1;
    return (int)(want < cap ? want : cap);
}

}  // namespace rlctr

using namespace rlctr;

static inline int pitch_of(const rlctr_table* t) { return t->row_pitch > 0 ? t->row_pitch : t->row_stride; }

static int check_table(const rlctr_table* t) {
    if (!t || !t->data || t->n_rows <= 0) return RLCTR_EINVAL;
    if (pitch_of(t) < t->row_stride || (t->row_stride != 1 && pitch_of(t) % 4 != 0)) return RLCTR_EUNSUPPORTED;
    if (t->row_stride != 1 && (t->row_stride % 4 != 0 || t->row_stride <= 0)) return RLCTR_EUNSUPPORTED;
    if (t->row_stride != 1 && !rlctr_aligned16(t->data)) return RLCTR_EALIGN;
    if (t->dim < 0 || t->emb_col < 0 || t->emb_col + t->dim > t->row_stride) return RLCTR_EINVAL;
    if (t->lin_col >= t->row_stride) return RLCTR_EINVAL;
    return RLCTR_OK;
}

extern "C" int rlctr_embed_fwd(const int64_t* ids, const rlctr_table* table, const float* bias,
                               float* logit, float* pctr, int64_t pctr_stride, float* sums,
                               float* rows_out, int64_t rows_pitch, int64_t batch, int32_t fields, int32_t flags,
                               rlctr_stream_t stream) {
    int rc = check_table(table);
    if (rc) return rc;
    if (batch < 0 || fields <= 0) return RLCTR_EINVAL;
    if (!ids && (table->world > 1 || table->n_rows < batch * fields)) return RLCTR_EINVAL;   // sample-ordered rows: local
    if (batch == 0) return RLCTR_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const int rs = table->row_stride;
    ShardView sv;
    if (!shard_view_of(table, &sv)) return RLCTR_EUNSUPPORTED;
    if (pctr && pctr_stride < 1) return RLCTR_EINVAL;
    if (rows_pitch == 0) rows_pitch = (int64_t)fields * table->dim;
    if (rows_out && rows_pitch < (int64_t)fields * table->dim) return RLCTR_EINVAL;
    if (rs == 1) {
        if (rows_out || (flags & RLCTR_FM_TERM) || table->lin_col != 0) return RLCTR_EUNSUPPORTED;
        int grid = grid_for_warps(batch, 8, 8);
        embed_fwd_scalar_kernel<<<grid, 256, 0, st>>>(ids, table->data, sv, table->n_rows, pitch_of(table), bias, logit, pctr,
                                                     pctr_stride, sums, batch, fields);
        RLCTR_LAUNCH_CHECK();
        return RLCTR_OK;
    }
    if (rs > 36) return RLCTR_EUNSUPPORTED;      // 36: a first-order column + 32 latent floats, padded
    if (sums && !rlctr_aligned16(sums)) return RLCTR_EALIGN;
    int grid = grid_for_warps(batch, 8, 5);      // 5 resident CTAs of 8 warps per SM (48 registers)
#define LAUNCH_EMBED(L)                                                                              \
    embed_fwd_kernel<L><<<grid, 256, 0, st>>>(ids, table->data, sv, table->n_rows, pitch_of(table), rs, table->lin_col,   \
                                              table->emb_col, table->dim, bias, logit, pctr,         \
                                              pctr_stride, sums, rows_out, rows_pitch, batch, fields, flags)
    switch (rlctr_lanes_per_row(rs)) {
        case 1: LAUNCH_EMBED(1); break;
        case 2: LAUNCH_EMBED(2); break;
        case 4: LAUNCH_EMBED(4); break;
        case 8: LAUNCH_EMBED(8); break;
        default: LAUNCH_EMBED(16); break;        // 33..36 floats: 9 chunks on 16 lanes, two rows per warp request
    }
#undef LAUNCH_EMBED
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

extern "C" int rlctr_group_fwd(const int64_t* ids, const rlctr_table* table, const rlctr_member* members, int32_t n_members,
                               float* sums, int32_t sums_pitch, int64_t batch, int32_t fields, rlctr_stream_t stream) {
    int rc = check_table(table);
    if (rc) return rc;
    if (!ids || !members || n_members < 1 || n_members > RLCTR_GROUP_MAX || batch < 0 || fields <= 0) return RLCTR_EINVAL;
    const int rs = table->row_stride;
    if (rs == 1 || rs > RLCTR_GROUP_MAX_FLOATS) return RLCTR_EUNSUPPORTED;
    if (sums && !rlctr_aligned16(sums)) return RLCTR_EALIGN;
    if (sums_pitch == 0) sums_pitch = rs;
    if (sums_pitch < rs || sums_pitch % 4 != 0) return RLCTR_EINVAL;
    if (batch == 0) return RLCTR_OK;
    ShardView sv;
    if (!shard_view_of(table, &sv)) return RLCTR_EUNSUPPORTED;
    GroupFwdView gv{};
    gv.n = n_members;
    // one line and every vector member a 16-float stand-alone row: group_fwd_kernel; anything else: group_fwd_wide_kernel
    bool wide = rs > 32;
    int fm_owner[RLCTR_GROUP_CHUNKS];                    // chunk -> the FM-term member whose latent columns it holds
    for (int ch = 0; ch < RLCTR_GROUP_CHUNKS; ++ch) fm_owner[ch] = -1;
    for (int m = 0; m < n_members; ++m) {
        const rlctr_member& mm = members[m];
        if (mm.lin_col >= rs || mm.dim < 0 || mm.emb_col < 0 || mm.emb_col + mm.dim > rs) return RLCTR_EINVAL;
        if (mm.pctr && mm.pctr_stride < 1) return RLCTR_EINVAL;
        int64_t rp = mm.rows_pitch ? mm.rows_pitch : (int64_t)fields * mm.dim;
        if (mm.rows_out && (rp < (int64_t)fields * mm.dim || rp > 0x7fffffff || mm.dim == 0)) return RLCTR_EINVAL;
        gv.lin_col[m] = mm.lin_col; gv.emb_col[m] = mm.emb_col; gv.dim[m] = mm.dim; gv.fm[m] = (mm.flags & RLCTR_FM_TERM) ? 1 : 0;
        gv.bias[m] = mm.bias; gv.logit[m] = mm.logit; gv.pctr[m] = mm.pctr; gv.pctr_stride[m] = mm.pctr_stride;
        gv.rows_out[m] = mm.rows_out; gv.rows_pitch[m] = (int)rp;
        gv.lpr[m] = mm.dim > 0 ? rlctr_member_lpr(mm.lin_col, mm.emb_col, mm.dim) : 4;
        if (gv.lpr[m] == 0) return RLCTR_EUNSUPPORTED;                     // stand-alone rows of at most 36 floats
        if (gv.lpr[m] != 4) wide = true;
        if (gv.fm[m] && mm.dim > 0) {
            if (((mm.emb_col + mm.dim - 1) >> 2) - (mm.emb_col >> 2) > gv.lpr[m] - 1) return RLCTR_EUNSUPPORTED;
            for (int ch = mm.emb_col >> 2; ch <= (mm.emb_col + mm.dim - 1) >> 2; ++ch) {
                if (fm_owner[ch] >= 0) return RLCTR_EUNSUPPORTED;       // a chunk's sum of squares belongs to one member
                fm_owner[ch] = m;
            }
        }
    }
    for (int ch = 0; ch < RLCTR_GROUP_CHUNKS; ++ch) gv.chunk_member[ch] = -1;
    int wf = wide ? 128 + RLCTR_GROUP_CHUNKS : 40;       // [column sums | per-chunk t] (per sample of the warp when wide)
    for (int m = 0; m < n_members; ++m) {
        gv.tile_off[m] = -1;
        if (gv.dim[m] <= 0) continue;
        for (int ch = gv.emb_col[m] >> 2; ch <= (gv.emb_col[m] + gv.dim[m] - 1) >> 2; ++ch) {
            if (gv.chunk_member[ch] >= 0) return RLCTR_EUNSUPPORTED;       // latent columns of two members in one 16-byte chunk
            gv.chunk_member[ch] = m;
        }
        if (gv.rows_out[m]) {
            if ((gv.rows_pitch[m] & 3) == 0 && !rlctr_aligned16(gv.rows_out[m])) return RLCTR_EALIGN;
            gv.tile_off[m] = wf;
            wf += (fields * gv.dim[m] + 3) & ~3;
        }
    }
    if (wide) {
        // W lanes per joint row: 16 (two samples per warp) when it has at most 16 chunks, else 32
        const int W = rs <= 64 ? 16 : 32;
        gv.warp_floats = (32 / W) * wf;
        const size_t smem = (size_t)8 * gv.warp_floats * sizeof(float);
        if (smem > 227 * 1024) return RLCTR_EUNSUPPORTED;
        const int grid = grid_for_warps((batch + 32 / W - 1) / (32 / W), 8, 8);
        // tower tiles past 48 KB: the opt-in to the whole 227 KB is set once per device (not per launch, which may be captured)
        int dev = 0;
        RLCTR_CUDA(cudaGetDevice(&dev));
        static bool opted[2][64] = {};
#define LAUNCH_WIDE(WW)                                                                                                        \
        {                                                                                                                      \
            bool& done = opted[WW == 32][dev & 63];                                                                            \
            if (smem > 48 * 1024 && !done) {                                                                                   \
                RLCTR_CUDA(cudaFuncSetAttribute(group_fwd_wide_kernel<WW>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)); \
                done = true;                                                                                                   \
            }                                                                                                                  \
            group_fwd_wide_kernel<WW><<<grid, 256, smem, (cudaStream_t)stream>>>(ids, table->data, sv, table->n_rows, pitch_of(table), \
                                                                                rs, gv, sums, sums_pitch, batch, fields);      \
        }
        if (W == 16) LAUNCH_WIDE(16) else LAUNCH_WIDE(32)
#undef LAUNCH_WIDE
        RLCTR_LAUNCH_CHECK();
        return RLCTR_OK;
    }
    gv.warp_floats = wf;
    const size_t smem = (size_t)8 * wf * sizeof(float);
    if (smem > 48 * 1024) return RLCTR_EUNSUPPORTED;
    const int grid = grid_for_warps(batch, 8, 3);
    static int ld_env = -1;
    // Default: plain read-only loads.  A joint row spans both 64-byte halves of its line, and the one-shot qualifiers that pay for
    // a 64-byte row (L1::no_allocate + L2::64B / ::128B: embed_fwd_kernel) make this gather slower: 83 against 52 us for 983,040 rows
    // of 96 bytes (profiles/r2_colocated.md) -- without L1 allocation the three sectors of a row travel as separate L2 requests.
    if (ld_env < 0) { const char* e = getenv("RLCTR_GROUP_LD"); ld_env = e ? atoi(e) : 1; }
#define LAUNCH_GROUP(L)                                                                                                          \
    if (fields <= 16) group_fwd_kernel<L, true><<<grid, 256, smem, (cudaStream_t)stream>>>(ids, table->data, sv, table->n_rows,       \
                                                                                          pitch_of(table), rs, gv, sums, sums_pitch, batch, fields); \
    else group_fwd_kernel<L, false><<<grid, 256, smem, (cudaStream_t)stream>>>(ids, table->data, sv, table->n_rows, pitch_of(table), \
                                                                               rs, gv, sums, sums_pitch, batch, fields)
    if (ld_env == 1) { LAUNCH_GROUP(1); } else if (ld_env == 2) { LAUNCH_GROUP(2); } else { LAUNCH_GROUP(0); }
#undef LAUNCH_GROUP
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

extern "C" int rlctr_gather_rows(const int64_t* ids, int64_t n, const rlctr_table* table, float* out,
                                 rlctr_stream_t stream) {
    int rc = check_table(table);
    if (rc) return rc;
    if (!ids || !out || n < 0) return RLCTR_EINVAL;
    if (n == 0) return RLCTR_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const int rs = table->row_stride;
    if (rs == 1) {
        int64_t blocks = (n + 255) / 256;
        int grid = (int)(blocks < RLCTR_SMS * 8 ? blocks : RLCTR_SMS * 8);
        gather_rows_scalar_kernel<<<grid, 256, 0, st>>>(ids, n, table->data, table->n_rows, pitch_of(table), out);
    } else {
        if (!rlctr_aligned16(out)) return RLCTR_EALIGN;
        int64_t blocks = (n * (rs / 4) + 255) / 256;
        int grid = (int)(blocks < RLCTR_SMS * 8 ? blocks : RLCTR_SMS * 8);
        gather_rows_kernel<<<grid, 256, 0, st>>>(ids, n, table->data, table->n_rows, pitch_of(table), rs, out);
    }
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

extern "C" int rlctr_featemb_fwd(const int64_t* ids, const rlctr_table* table, float* out,
                                 int64_t out_stride, int64_t batch, int32_t fields,
                                 rlctr_stream_t stream) {
    int rc = check_table(table);
    if (rc) return rc;
    if (!ids || !out || batch < 0 || fields < 2) return RLCTR_EINVAL;
    const int rs = table->row_stride, dim = table->dim;
    if (rs == 1 || rs > 32 || dim <= 0 || fields > 255) return RLCTR_EUNSUPPORTED;
    const int npair = fields * (fields - 1) / 2;
    if (out_stride < npair + fields * dim) return RLCTR_EINVAL;
    if (batch == 0) return RLCTR_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const int nw = 4;
    size_t smem = (size_t)nw * fields * dim * sizeof(float) + 2 * (size_t)npair;
    if (smem > 48 * 1024) return RLCTR_EUNSUPPORTED;
    int grid = grid_for_warps(batch, nw, 16);
#define LAUNCH_FE(L)                                                                               \
    featemb_fwd_kernel<L><<<grid, nw * 32, smem, st>>>(ids, table->data, table->n_rows, pitch_of(table), rs, \
                                                       table->emb_col, dim, out, out_stride, batch, fields)
    switch (rlctr_lanes_per_row(rs)) {
        case 1: LAUNCH_FE(1); break;
        case 2: LAUNCH_FE(2); break;
        case 4: LAUNCH_FE(4); break;
        default: LAUNCH_FE(8); break;
    }
#undef LAUNCH_FE
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}


extern "C" int rlctr_pairdots_fwd(const float* rows, int64_t ld_rows, float* out, int64_t ld_out, int64_t batch,
                                  int32_t fields, int32_t dim, int32_t ip_first, rlctr_stream_t stream) {
    if (!rows || !out || batch < 0 || fields < 2 || dim <= 0) return RLCTR_EINVAL;
    if (fields > 23) return RLCTR_EUNSUPPORTED;                         // pair indices are bytes: F <= 23 (P <= 253)
    const int fd = fields * dim, npair = fields * (fields - 1) / 2;
    if (ld_rows < fd || ld_out < fd + npair) return RLCTR_EINVAL;
    if (batch == 0) return RLCTR_OK;
    const int nw = 4;
    const size_t smem = (size_t)nw * fd * sizeof(float) + 2 * (size_t)npair;
    if (smem > 48 * 1024) return RLCTR_EUNSUPPORTED;
    pairdots_fwd_kernel<<<grid_for_warps(batch, nw, 16), nw * 32, smem, (cudaStream_t)stream>>>(rows, ld_rows, out, ld_out, batch,
                                                                                               fields, dim, ip_first ? 1 : 0);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

extern "C" int rlctr_pairdots_bwd(const float* rows, int64_t ld_rows, const float* gout, int64_t ld_g, float* grows,
                                  int64_t ld_grows, int64_t batch, int32_t fields, int32_t dim, int32_t ip_first,
                                  rlctr_stream_t stream) {
    if (!rows || !gout || !grows || batch < 0 || fields < 2 || dim <= 0) return RLCTR_EINVAL;
    if (fields > 23) return RLCTR_EUNSUPPORTED;
    const int fd = fields * dim, npair = fields * (fields - 1) / 2;
    if (ld_rows < fd || ld_g < fd + npair || ld_grows < fd) return RLCTR_EINVAL;
    if (batch == 0) return RLCTR_OK;
    const int nw = 4;
    const size_t smem = (size_t)nw * (fd + npair) * sizeof(float) + (size_t)fields * fields;
    if (smem > 48 * 1024) return RLCTR_EUNSUPPORTED;
    pairdots_bwd_kernel<<<grid_for_warps(batch, nw, 16), nw * 32, smem, (cudaStream_t)stream>>>(rows, ld_rows, gout, ld_g, grows,
                                                                                               ld_grows, batch, fields, dim,
                                                                                               ip_first ? 1 : 0);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}
