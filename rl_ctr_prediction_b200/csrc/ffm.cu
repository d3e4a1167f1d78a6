// ffm.cu -- K2: FFM forward over the interleaved table (p_model.py:59-100).  sm_100a.
//
// The reference keeps F tables of [N, D] and gathers F*F rows of 40 B per sample (p_model.py:87).
// Here one id owns ONE contiguous fused row
//     [ T_0[id] | T_1[id] | ... | T_{F-1}[id] | w[id] | pad ]      (F*D + 1 floats, padded to x4)
// so a sample reads F contiguous rows of ~600 B as coalesced 128-bit chunks instead of F*F
// scattered 40 B rows (SURVEY H3).  A warp owns a sample: the F rows are staged in shared
// memory, then the P = F(F-1)/2 pair dots <T_j[x_i], T_i[x_j]> are taken from there.
//
// Training: the same kernel optionally writes the "partner rows"
//     partners[b*F + i, block j] = T_i[x_j]     (j != i; zero on the diagonal, lin col = 1)
// i.e. d logit / d row_i, so the backward is a pure scale by dlogit[b] done inside the
// sort/segment-reduce/Adam kernel (optim.cu, RLCTR_STAGED_PARTNER) and never re-gathers.
#include "common.cuh"

namespace rlctr {

constexpr unsigned short FFM_ZERO = 0xffffu, FFM_ONE = 0xfffeu;

// 16-byte asynchronous copy global -> shared; src_bytes = 0 writes zeros (an id outside the table is an all-zero row)
__device__ __forceinline__ void ffm_cp16(float* smem_dst, const float* gsrc, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc),
                 "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void ffm_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void ffm_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
// the F rows of one sample into `dst` [F][rs]: lane f holds the id of field f in `my_id` and, when F64, that of field f + 32 in
// `my_id_hi` (fields <= 32, or <= 64 with F64); the lanes take chunks lane, lane + 32 ...
template <bool F64>
__device__ __forceinline__ void ffm_issue_rows(float* dst, int64_t my_id, int64_t my_id_hi, const float* __restrict__ tab,
                                               const ShardView& sv, int64_t n_rows, int pitch, int rs, int fields, int lane) {
    const int chunks = rs >> 2;
    for (int f = 0; f < fields; ++f) {
        int64_t id;
        if constexpr (F64) id = __shfl_sync(RLCTR_FULL, f < 32 ? my_id : my_id_hi, f & 31);
        else id = __shfl_sync(RLCTR_FULL, my_id, f);
        const bool ok = (uint64_t)id < (uint64_t)n_rows;
        const float* src = row_ptr(tab, sv, ok ? id : 0, pitch);
        for (int c = lane; c < chunks; c += 32) ffm_cp16(dst + f * rs + 4 * c, src + 4 * c, ok ? 16 : 0);
    }
    ffm_commit();
}

// smem bytes of a CTA of `warps` warps with `nbuf` [F][rs] stage buffers each, the pair tables and the partner table
static inline size_t ffm_smem_bytes(int warps, int nbuf, int fields, int rs) {
    const size_t npair = (size_t)fields * (fields - 1) / 2;
    return (size_t)warps * nbuf * fields * rs * sizeof(float) + 2 * npair + 2 + (size_t)fields * rs;
}

// VEC: latent, emb_col and lin_col even -- a float2 of a partner row never straddles two column blocks, so the partner rows are
// written as coalesced 8-byte stores driven by a per-block table (built once: no divisions in the per-sample loop).
// WARPS samples per CTA, each warp with NBUF stage buffers; F64: fields up to 64 (two ids per lane).  <VEC, 2, 2, false> serves
// F <= 32 at up to 200 KB; the others (one warp, double- or single-buffered) serve the shapes it cannot hold.  A sample's
// arithmetic (lane-strided pair loop, butterfly) is the same in every variant, so its logit has the same bits in each.
template <bool VEC, int WARPS, int NBUF, bool F64>
__global__ void __launch_bounds__(WARPS * 32)
ffm_fwd_kernel(const int64_t* __restrict__ ids, const float* __restrict__ tab, const __grid_constant__ ShardView sv,
               int64_t n_rows, int pitch, int rs,
               int lin_col, int emb_col, const float* __restrict__ bias, float* __restrict__ logit,
               float* __restrict__ pctr, int64_t pctr_stride, float* __restrict__ partners,
               int64_t batch, int fields, int latent) {
    extern __shared__ __align__(16) float smem[];
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int npair = fields * (fields - 1) / 2;
    // NBUF = 2: two [F][rs] buffers per warp, the rows of the warp's NEXT sample arrive (cp.async) while the current one is reduced
    // and its partner rows are written -- the gather never waits for the arithmetic and the stores
    float* buf0 = smem + (size_t)wib * NBUF * fields * rs;
    unsigned char* pi = reinterpret_cast<unsigned char*>(smem + (size_t)WARPS * NBUF * fields * rs);
    unsigned char* pj = pi + npair;
    // partner table: for destination float2 e = i * (rs / 2) + q of a sample's partner rows, the source float offset in `stage`
    unsigned short* ptab = reinterpret_cast<unsigned short*>(pj + npair + ((2 * npair) & 1));
    const int half = rs >> 1, per2 = fields * half;
    for (int i = threadIdx.x; i < fields - 1; i += blockDim.x) {
        const int base = i * fields - i * (i + 1) / 2;                     // pair order of p_model.py:89-91
        for (int j = i + 1; j < fields; ++j) {
            pi[base + j - i - 1] = (unsigned char)i;
            pj[base + j - i - 1] = (unsigned char)j;
        }
    }
    if (VEC && partners) {
        for (int e = threadIdx.x; e < per2; e += blockDim.x) {
            const int i = e / half, col = 2 * (e - i * half);
            unsigned short code = FFM_ZERO;
            const int x = col - emb_col;
            if (col == lin_col) code = FFM_ONE;
            else if (x >= 0 && x < fields * latent) {
                const int j = x / latent, k = x - j * latent;
                if (j != i) code = (unsigned short)(j * rs + emb_col + i * latent + k);
            }
            ptab[e] = code;
        }
    }
    __syncthreads();
    const float b0 = bias ? __ldg(bias) : 0.f;
    const int64_t warp0 = (int64_t)blockIdx.x * WARPS + wib;
    const int64_t nwarps = (int64_t)gridDim.x * WARPS;
    // ids of a sample: field `lane` (and `lane + 32` when F64); -1 past the last field
    auto load_ids = [&](int64_t b, int64_t& lo, int64_t& hi) {
        lo = (lane < fields) ? __ldg(ids + b * fields + lane) : -1;
        if constexpr (F64) hi = (lane + 32 < fields) ? __ldg(ids + b * fields + lane + 32) : -1;
    };
    int64_t id_next = -1, id_next_hi = -1;
    int cur = 0;
    if constexpr (NBUF == 2) {
        // prologue: ids of the first two samples, rows of the first in flight
        if (warp0 < batch) {
            int64_t id0 = -1, id0_hi = -1;
            load_ids(warp0, id0, id0_hi);
            ffm_issue_rows<F64>(buf0, id0, id0_hi, tab, sv, n_rows, pitch, rs, fields, lane);
            if (warp0 + nwarps < batch) load_ids(warp0 + nwarps, id_next, id_next_hi);
        }
    }
    for (int64_t b = warp0; b < batch; b += nwarps, cur ^= (NBUF - 1)) {
        float* stage = buf0 + cur * fields * rs;
        if constexpr (NBUF == 2) {
            const bool more = b + nwarps < batch;                          // warp-uniform
            if (more) ffm_issue_rows<F64>(buf0 + (cur ^ 1) * fields * rs, id_next, id_next_hi, tab, sv, n_rows, pitch, rs, fields, lane);
            id_next = -1;
            id_next_hi = -1;
            if (b + 2 * nwarps < batch) load_ids(b + 2 * nwarps, id_next, id_next_hi);
            if (more) ffm_wait<1>(); else ffm_wait<0>();
        } else {                                                           // one buffer: this sample's rows, then its arithmetic
            int64_t id = -1, id_hi = -1;
            load_ids(b, id, id_hi);
            ffm_issue_rows<F64>(stage, id, id_hi, tab, sv, n_rows, pitch, rs, fields, lane);
            ffm_wait<0>();
        }
        __syncwarp();
        // ---- first order + pair dots
        float acc = 0.f;
        if (lin_col >= 0)
            for (int f = lane; f < fields; f += 32) acc += stage[f * rs + lin_col];
        for (int p = lane; p < npair; p += 32) {
            const int i = pi[p], j = pj[p];
            const float* a = stage + i * rs + emb_col + j * latent;        // T_j[x_i]
            const float* c = stage + j * rs + emb_col + i * latent;        // T_i[x_j]
            float d = 0.f;
            for (int k = 0; k < latent; ++k) d = fmaf(a[k], c[k], d);
            acc += d;
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(RLCTR_FULL, acc, off);
        if (lane == 0) {
            const float z = b0 + acc;
            if (logit) logit[b] = z;
            if (pctr) pctr[b * pctr_stride] = sigmoidf_ref(z);
        }
        // ---- partner rows (training): row (b,i), column block j  <-  stage[j][block i]
        if (partners) {
            float* out = partners + (b * fields) * (int64_t)rs;
            if (VEC) {
                float2* out2 = reinterpret_cast<float2*>(out);
#pragma unroll 4
                for (int e = lane; e < per2; e += 32) {
                    const unsigned short code = ptab[e];
                    float2 v = make_float2(0.f, 0.f);
                    if (code == FFM_ONE) v.x = 1.0f;
                    else if (code != FFM_ZERO) v = *reinterpret_cast<const float2*>(stage + code);
                    __stcs(out2 + e, v);
                }
            } else {
                const int per_sample = fields * rs;
                for (int t = lane; t < per_sample; t += 32) {
                    const int i = t / rs, col = t - i * rs;
                    float v = 0.f;
                    const int e = col - emb_col;
                    if (col == lin_col) v = 1.0f;
                    else if (e >= 0 && e < fields * latent) {
                        const int j = e / latent, k = e - j * latent;
                        if (j != i) v = stage[j * rs + emb_col + i * latent + k];
                    }
                    __stcs(out + t, v);
                }
            }
        }
        __syncwarp();
    }
}

}  // namespace rlctr

using namespace rlctr;

extern "C" int rlctr_ffm_fwd(const int64_t* ids, const rlctr_table* table, const float* bias, float* logit,
                             float* pctr, int64_t pctr_stride, float* partners, int64_t batch, int32_t fields,
                             int32_t latent, rlctr_stream_t stream) {
    if (!ids || !table || !table->data || table->n_rows <= 0 || batch < 0) return RLCTR_EINVAL;
    if (fields < 2 || fields > 64 || latent <= 0) return RLCTR_EUNSUPPORTED;   // a lane holds the ids of fields lane, lane + 32
    const int rs = table->row_stride;
    if (rs % 4 != 0 || table->dim != fields * latent || table->emb_col < 0 ||
        table->emb_col + table->dim > rs || table->lin_col >= rs)
        return RLCTR_EINVAL;
    if (!rlctr_aligned16(table->data) || (partners && !rlctr_aligned16(partners))) return RLCTR_EALIGN;
    if (pctr && pctr_stride < 1) return RLCTR_EINVAL;
    if (batch == 0) return RLCTR_OK;
    ShardView sv;
    if (!shard_view_of(table, &sv)) return RLCTR_EUNSUPPORTED;
    const bool vec = (latent % 2 == 0) && (table->emb_col % 2 == 0) && (table->lin_col < 0 || table->lin_col % 2 == 0) &&
                     (size_t)fields * rs < 0xfff0u;
    const int pitch = table->row_pitch > 0 ? table->row_pitch : rs;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t smem = ffm_smem_bytes(2, 2, fields, rs);
    if (fields <= 32 && smem <= 200 * 1024) {
        RLCTR_CUDA(cudaFuncSetAttribute(ffm_fwd_kernel<true, 2, 2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        RLCTR_CUDA(cudaFuncSetAttribute(ffm_fwd_kernel<false, 2, 2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        int64_t want = (batch + 1) / 2;
        int per_sm = (int)((size_t)(220 * 1024) / (smem + 1024));
        if (per_sm < 1) per_sm = 1;
        if (per_sm > 16) per_sm = 16;
        const int64_t cap = (int64_t)RLCTR_SMS * per_sm;
        const int grid = (int)(want < cap ? want : cap);
        if (vec)
            ffm_fwd_kernel<true, 2, 2, false><<<grid, 64, smem, st>>>(ids, table->data, sv, table->n_rows, pitch, rs, table->lin_col,
                                                                     table->emb_col, bias, logit, pctr, pctr_stride, partners, batch,
                                                                     fields, latent);
        else
            ffm_fwd_kernel<false, 2, 2, false><<<grid, 64, smem, st>>>(ids, table->data, sv, table->n_rows, pitch, rs, table->lin_col,
                                                                      table->emb_col, bias, logit, pctr, pctr_stride, partners, batch,
                                                                      fields, latent);
        RLCTR_LAUNCH_CHECK();
        return RLCTR_OK;
    }
    // Shapes the two-warp kernel cannot hold: F = 33..64, or stage buffers past 200 KB.  One warp per CTA, so a CTA takes the least
    // shared memory one sample needs; double-buffered where two buffers fit in 227 KB, else single-buffered (one [F][rs] buffer of
    // a row of at most 512 floats is 128 KB at F = 64).  The opt-in is set once per device (not per launch, which may be captured).
    const int nbuf = ffm_smem_bytes(1, 2, fields, rs) <= 227 * 1024 ? 2 : 1;
    const size_t smem1 = ffm_smem_bytes(1, nbuf, fields, rs);
    if (smem1 > 227 * 1024) return RLCTR_EUNSUPPORTED;
    int dev = 0;
    RLCTR_CUDA(cudaGetDevice(&dev));
    static bool opted[2][2][64] = {};
    bool& done = opted[vec][nbuf - 1][dev & 63];
    if (!done) {
        if (vec && nbuf == 2)
            RLCTR_CUDA(cudaFuncSetAttribute(ffm_fwd_kernel<true, 1, 2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        else if (vec)
            RLCTR_CUDA(cudaFuncSetAttribute(ffm_fwd_kernel<true, 1, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        else if (nbuf == 2)
            RLCTR_CUDA(cudaFuncSetAttribute(ffm_fwd_kernel<false, 1, 2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        else
            RLCTR_CUDA(cudaFuncSetAttribute(ffm_fwd_kernel<false, 1, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        done = true;
    }
    int per_sm = (int)((size_t)(228 * 1024) / (smem1 + 1024));     // 228 KB of shared memory per SM, 1 KB reserved per CTA
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 32) per_sm = 32;
    const int64_t cap = (int64_t)RLCTR_SMS * per_sm;
    const int grid = (int)(batch < cap ? batch : cap);
#define LAUNCH_FFM1(V, NB)                                                                                                     \
    ffm_fwd_kernel<V, 1, NB, true><<<grid, 32, smem1, st>>>(ids, table->data, sv, table->n_rows, pitch, rs, table->lin_col,    \
                                                            table->emb_col, bias, logit, pctr, pctr_stride, partners, batch,   \
                                                            fields, latent)
    if (vec) { if (nbuf == 2) LAUNCH_FFM1(true, 2); else LAUNCH_FFM1(true, 1); }
    else { if (nbuf == 2) LAUNCH_FFM1(false, 2); else LAUNCH_FFM1(false, 1); }
#undef LAUNCH_FFM1
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}
