// mlp_tma.cu -- K4: the dense-layer GEMMs with TMA-fed operand tiles and tcgen05 MMAs.
//
//     C[M,N] = A[M,K] * B[N,K]^T (+ bias[N]) (ReLU)        fp32 in, fp32 out, 3xTF32 split (see mlp.cu)
//
// The software-staged gemm3x_tf32_kernel (mlp.cu) is latency-bound at 14 % tensor-pipe activity with every warp parked on an
// mbarrier (profiles/r1_ncu_top_kernels.md).  This kernel keeps the tensor pipe fed:
//   * operand tiles are fetched by TMA (cp.async.bulk.tensor, SWIZZLE_128B, zero fill outside the tensor): one elected thread
//     issues whole boxes, no per-thread address arithmetic, no LDGSTS issue slots;
//   * the small operand of forward / dgrad -- the WEIGHT -- is split into (hi, lo) ONCE per call by a tiny elementwise kernel
//     and arrives ready-made through two tensor maps; wgrad's raw B tile is split in shared memory by the converter warps
//     (raw -> hi in place and lo, elementwise at identical byte offsets: independent of the swizzle and of the major-ness);
//   * operands that are contiguous along M/N instead of K (dgrad's W, wgrad's dY^T and X) are consumed in place as MN-major
//     UMMA operands (TMA boxes of 32 mn x 32 k in the SWIZZLE_128B_BASE32B layout): no 4-byte transposing copies;
//   * the streamed A operand lives in TENSOR MEMORY: a converter thread owns one row of the raw 128 x 32 tile, reads its 32
//     k-values from the swizzled shared-memory tile, splits them and writes (A_hi, A_lo) with tcgen05.st; the MMAs take A from
//     TMEM (tcgen05.mma ... [d_tmem], [a_tmem], b_desc), so A crosses the shared-memory port once per k-block (profiles/r1e_*);
//     for wgrad the same thread's sum over its row is the bias gradient;
//   * C leaves through per-warp 32 x 32 staging blocks and TMA stores (cp.async.bulk.tensor ... global.shared::cta): full
//     128-byte row segments instead of 16-byte pieces of 32 different lines per store instruction.  Split-K partials, C that
//     TMA cannot address and the 16-column tail of a tile are stored per thread;
//   * dgrad takes the ReLU / dropout mask of the layer below from TMA-loaded 32 x 32 blocks, one per epilogue warp, requested a
//     chunk ahead (instantiation MASK = true); a mask TMA cannot address is read per thread, with the same bits;
//   * the all-zero k-steps of a ragged last k-block (K % 32 != 0: TMA zero fill) are not issued;
//   * RLCTR_GEMM_DBG records per-stage clock stamps of block 0 (scratch/gemm_trace.py).
//
// Warp roles (320 threads, one CTA per SM, persistent over output tiles):
//     warps 0-3  converters        wait raw[s] -> row of A: split -> tcgen05.st (hi | lo) -> arrive full[s]
//     warp  4    TMA producer      wait empty[s] -> expect_tx + boxes of A (raw), B(hi), B(lo) -> raw[s]
//     warp  5    MMA issuer        wait raw[s], full[s] -> 4 k-steps x 3 tcgen05.mma (A from TMEM) -> commit empty[s] / tmem_full[acc]
//     warps 6-9  epilogue          tcgen05.ld -> bias / ReLU / dropout / mask -> staging block -> TMA store   (TMEM double-buffered)
// TMEM columns: accumulator stage s at s * round32(n_tile); A stage s at 2 * round32(n_tile) + 64 * s (32 columns hi, 32 lo).
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>

#include "common.cuh"
#include "mlp_tma.cuh"

namespace rlctr {
namespace tma {

constexpr int BM = 128;                   // UMMA M
constexpr int BK = 32;                    // fp32 per k-block row: 128 B = one swizzle atom
constexpr int UK = 8;                     // K of one tcgen05.mma kind::tf32
constexpr int CONV_WARPS = 4;
constexpr int EPI_WARPS = 4;
constexpr int PRODUCER_WARP = CONV_WARPS;
constexpr int MMA_WARP = CONV_WARPS + 1;
constexpr int THREADS = 32 * (CONV_WARPS + 2 + EPI_WARPS);
constexpr int MAX_STAGES = 8;
constexpr int TMEM_COLS = 512;
constexpr uint32_t A_TILE_BYTES = BM * 128;
constexpr int BIAS_SMEM = 1024;              // bias values staged in shared memory for the epilogue

struct Args {
    float* C; int64_t ldc;                // C[(split*M + m)*ldc + n]
    int cvec;
    const float* bias;
    int M, N, K;
    int n_tile, m_tiles, n_tiles, splits, kb_per_split, stages;
    int a_mn, b_mn;                       // 1: operand is contiguous along M (N) instead of K
    int b_presplit;                       // 1: B arrives as (hi, lo) through mapB / mapBlo
    int relu;
    int acc_stride, a_col0;               // TMEM columns: accumulator stage s at s*acc_stride, A stage s at a_col0 + 64*s (hi | lo)
    int c_tma;                            // 1: the epilogue stages 32x32 blocks of C in shared memory and TMA-stores them (mapC)
    long long* dbg;                       // RLCTR_GEMM_DBG: per-stage clock64 stamps of block 0 (scratch/gemm_trace.py), else null
    float* colsum_part;                   // wgrad only: [splits][M] partial column sums of the MN-major A operand (db), or null
    Epilogue epi;                         // fused dropout (forward) / ReLU-dropout mask of the layer below (dgrad)
};

// ---- PTX wrappers ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// A protocol bug must surface as an error, not as a hung GPU box: give up after ~4 s.
__device__ __noinline__ void mbar_timeout(uint32_t bar, uint32_t parity) {
    printf("rlctr gemm3x_tma_kernel: mbarrier wait timed out (block %d thread %d bar 0x%x parity %u)\n", (int)blockIdx.x,
           (int)threadIdx.x, bar, parity);
    __trap();
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (mbar_try(bar, parity)) return;
    uint64_t t0 = 0;
    uint32_t spins = 0;
    while (!mbar_try(bar, parity)) {
        if ((++spins & 0x3fffu) == 0) {
            uint64_t now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000ull) mbar_timeout(bar, parity);
        }
    }
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// A operand from tensor memory (lanes = rows of A, one 32-bit column per k): no shared-memory read for A
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc),
        "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t* r) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
        "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
        "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]),
        "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]),
        "r"(r[31]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ float lds32(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
template <int W>
__device__ __forceinline__ void tmem_ld(uint32_t taddr, uint32_t* r) {
    if (W == 32) tmem_ld32(taddr, r); else tmem_ld16(taddr, r);
}
// the registers of a tcgen05.ld are valid only after tcgen05.wait::ld: pin every use behind the wait
template <int W>
__device__ __forceinline__ void tmem_ld_fence(uint32_t* r) {
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < W; ++j) asm volatile("" : "+r"(r[j]));
}
// one TMA box: 2-D tile of the tensor described by `map`, coordinates (c0 = innermost, c1), lands at `dst` and
// reports its bytes on `bar`
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
// shared -> global store of one box (clipped at the tensor bounds), tracked by the issuing thread's bulk async-group
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)),
                 "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

// shared-memory matrix descriptors (cute::UMMA::SmemDescriptor bit layout), SWIZZLE_128B, version 1
//   K-major : rows of 128 B (32 fp32 of K), 8-row groups 1024 B apart (SBO); one MMA (K = 8) advances 32 B
//   MN-major: 32-bit operands have ONE legal MN-major layout, SWIZZLE_128B_BASE32B (Swizzle<2,5,2>: 32-byte chunks
//             XOR-ed with (k-row & 3); TMA mode SWIZZLE_128B_ATOM_32B): k-rows of 128 B (32 mn), groups of 4 k-rows
//             512 B apart (SBO), blocks of 32 mn 4096 B apart (LBO = one 32x32 TMA box); one MMA (K = 8) advances 1024 B
__device__ __forceinline__ uint64_t desc_k_major(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
__device__ __forceinline__ uint64_t desc_mn_major(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)(4096 >> 4) << 16;                  // LBO: next block of 32 mn
    d |= (uint64_t)(512 >> 4) << 32;                   // SBO: next group of 4 k-rows
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)1 << 61;                            // SWIZZLE_128B_BASE32B
    return d;
}

__device__ __forceinline__ float tf32_rn(float x) {
    return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
}
__device__ __forceinline__ float4 lds128(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts128(uint32_t a, const float4& v) {
    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void split4(const float4& x, float4& h, float4& l) {
    h = make_float4(tf32_rn(x.x), tf32_rn(x.y), tf32_rn(x.z), tf32_rn(x.w));
    l = make_float4(x.x - h.x, x.y - h.y, x.z - h.z, x.w - h.w);
}
// raw -> (hi in place, lo): elementwise, same byte offset in both tiles (layout-agnostic).  `bytes` is a multiple
// of 2048 (16 rows of 128 B); the 128 converter threads take two 16-byte chunks per iteration.
__device__ __forceinline__ void split_tile(uint32_t hi, uint32_t lo, int bytes, int tid) {
    constexpr int STEP = CONV_WARPS * 32 * 16;
    for (int off = tid * 16; off < bytes; off += 2 * STEP) {
        const bool two = off + STEP < bytes;
        const float4 x0 = lds128(hi + off);
        float4 x1 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (two) x1 = lds128(hi + off + STEP);
        float4 h, l;
        split4(x0, h, l);
        sts128(hi + off, h);
        sts128(lo + off, l);
        if (two) {
            split4(x1, h, l);
            sts128(hi + off + STEP, h);
            sts128(lo + off + STEP, l);
        }
    }
}

// Converters: thread t owns row m = t of the 128 x 32 raw A tile.  It reads its 32 k-values from the swizzled
// shared-memory tile (K-major: eight 16-byte chunks, chunk c stored at c ^ (t & 7) -- a quarter-warp covers all 32 banks;
// MN-major: one 4-byte element per k-row, a warp reads 128 contiguous bytes), splits them and writes hi to TMEM columns
// [col, col + 32) and lo to [col + 32, col + 64) of its lane.  Returns the sum of the raw values (wgrad's bias gradient).
__device__ __forceinline__ float split_row_to_tmem(uint32_t raw, bool a_mn, int t, uint32_t taddr) {
    uint32_t hi[BK], lo[BK];
    float sum = 0.f;
    if (!a_mn) {
        const uint32_t row = raw + (uint32_t)t * 128u;
#pragma unroll
        for (int c = 0; c < BK / 4; ++c) {
            const float4 x = lds128(row + (uint32_t)((c ^ (t & 7)) << 4));
            float4 h, l;
            split4(x, h, l);
            hi[4 * c] = __float_as_uint(h.x); hi[4 * c + 1] = __float_as_uint(h.y);
            hi[4 * c + 2] = __float_as_uint(h.z); hi[4 * c + 3] = __float_as_uint(h.w);
            lo[4 * c] = __float_as_uint(l.x); lo[4 * c + 1] = __float_as_uint(l.y);
            lo[4 * c + 2] = __float_as_uint(l.z); lo[4 * c + 3] = __float_as_uint(l.w);
        }
    } else {
        const int mm = t & 31;
        const uint32_t blk = raw + (uint32_t)(t >> 5) * 4096u + (uint32_t)((mm & 7) << 2);
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            const float x = lds32(blk + (uint32_t)k * 128u + (uint32_t)((((mm >> 3) ^ (k & 3))) << 5));
            const float h = tf32_rn(x);
            hi[k] = __float_as_uint(h);
            lo[k] = __float_as_uint(x - h);
            sum += x;
        }
    }
    tmem_st32(taddr, hi);
    tmem_st32(taddr + (uint32_t)BK, lo);
    tmem_st_wait();
    return sum;
}

#define DBG_STAMP(it, slot)                                                                         \
    do {                                                                                           \
        if (g.dbg && blockIdx.x == 0 && (it) < 256) g.dbg[(it) * 16 + (slot)] = clock64();          \
    } while (0)

struct TileWalk {                          // this CTA's (tile, k-block) sequence, identical in every role
    int tile, kb0, kb1, mt, nt, split;
};
__device__ __forceinline__ bool tile_decode(TileWalk& w, const Args& g, int total_tiles) {
    if (w.tile >= total_tiles) return false;
    const int mn = g.m_tiles * g.n_tiles;
    w.split = w.tile / mn;
    const int r = w.tile - w.split * mn;
    w.mt = r / g.n_tiles;
    w.nt = r - w.mt * g.n_tiles;
    const int kb_total = (g.K + BK - 1) / BK;
    w.kb0 = w.split * g.kb_per_split;
    w.kb1 = min(w.kb0 + g.kb_per_split, kb_total);
    return true;
}


struct EpiCtx {
    float* crow;               // &C[row of this thread][0]
    const float* bias;         // global bias (null: none)
    const float* sbias;        // the same bias staged in shared memory (null: read it from global)
    int N, cvec;
    bool row_ok, relu, zero;
    // dropout of the forward output: element index = row * N + n
    bool drop;
    uint64_t drop_seed, drop_base;        // drop_base = counter + row * N
    uint32_t drop_thresh;
    float drop_scale;
    // dgrad: dx *= (mask_row[n] > 0 ? mask_scale : 0)  (mask_row = the layer input's row: ReLU+dropout of the layer below)
    const float* mask_row;
    int mvec;
    float mask_scale;
    uint32_t mbuf;             // != 0: the chunk's mask sits in this warp's TMA-loaded 32 x 32 block (applied in epilogue_stage)
};
// W accumulator columns [n0, n0 + W) of this thread's row: bias, ReLU, dropout, mask of the layer below -> v[]
template <int W>
__device__ __forceinline__ void epilogue_compute(const EpiCtx& e, const uint32_t* r, int n0, float (&v)[W]) {
#pragma unroll
    for (int j = 0; j < W; ++j) v[j] = e.zero ? 0.f : __uint_as_float(r[j]);
    if (e.sbias) {
#pragma unroll
        for (int j = 0; j < W; j += 4) {
            const float4 b = *reinterpret_cast<const float4*>(e.sbias + n0 + j);     // warp-wide broadcast
            v[j] += b.x; v[j + 1] += b.y; v[j + 2] += b.z; v[j + 3] += b.w;
        }
    } else if (e.bias) {
#pragma unroll
        for (int j = 0; j < W; ++j)
            if (n0 + j < e.N) v[j] += __ldg(e.bias + n0 + j);
    }
    if (e.relu) {
#pragma unroll
        for (int j = 0; j < W; ++j) v[j] = fmaxf(v[j], 0.f);
    }
    if (e.drop) {
        const uint64_t i0 = e.drop_base + (uint64_t)n0;                   // element index of column n0 of this row
        const uint64_t p0 = i0 >> 1, p1 = (i0 + (uint64_t)(W - 1)) >> 1;
        if (!(i0 & 1) && (p0 >> 32) == (p1 >> 32)) {                      // pairs aligned with the columns, one key: the usual case
            const uint32_t key = dropout_key(e.drop_seed, (uint32_t)(p0 >> 32)), lo = (uint32_t)p0;
#pragma unroll
            for (int j = 0; j < W; j += 2) {
                const uint32_t h = dropout_bits(key, lo + (uint32_t)(j >> 1));
                v[j] = (h & 0xffffu) >= e.drop_thresh ? v[j] * e.drop_scale : 0.f;
                v[j + 1] = (h >> 16) >= e.drop_thresh ? v[j + 1] * e.drop_scale : 0.f;
            }
        } else {
#pragma unroll
            for (int j = 0; j < W; ++j)
                v[j] = dropout_keep(e.drop_seed, i0 + (uint64_t)j, e.drop_thresh) ? v[j] * e.drop_scale : 0.f;
        }
    }
    if (e.mask_row && e.row_ok && !(W == 32 && e.mbuf)) {
        const float* mr = e.mask_row + n0;
        if (n0 + W <= e.N && e.mvec == 4) {
#pragma unroll
            for (int j = 0; j < W; j += 4) {
                const float4 x = __ldg(reinterpret_cast<const float4*>(mr + j));
                v[j] = x.x > 0.f ? v[j] * e.mask_scale : 0.f;
                v[j + 1] = x.y > 0.f ? v[j + 1] * e.mask_scale : 0.f;
                v[j + 2] = x.z > 0.f ? v[j + 2] * e.mask_scale : 0.f;
                v[j + 3] = x.w > 0.f ? v[j + 3] * e.mask_scale : 0.f;
            }
        } else {
#pragma unroll
            for (int j = 0; j < W; ++j)
                if (n0 + j < e.N) v[j] = __ldg(mr + j) > 0.f ? v[j] * e.mask_scale : 0.f;
        }
    }
}
// ... and straight to global memory from the thread's registers (one row per thread: 16-byte pieces of 32 different lines)
template <int W>
__device__ __forceinline__ void epilogue_emit(const EpiCtx& e, const uint32_t* r, int n0) {
    if (!e.row_ok || n0 >= e.N) return;
    float v[W];
    epilogue_compute<W>(e, r, n0, v);
    float* dst = e.crow + n0;
    if (n0 + W <= e.N && e.cvec == 4) {
#pragma unroll
        for (int j = 0; j < W; j += 4) *reinterpret_cast<float4*>(dst + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    } else if (n0 + W <= e.N && e.cvec == 2) {
#pragma unroll
        for (int j = 0; j < W; j += 2) *reinterpret_cast<float2*>(dst + j) = make_float2(v[j], v[j + 1]);
    } else {
#pragma unroll
        for (int j = 0; j < W; ++j)
            if (n0 + j < e.N) dst[j] = v[j];
    }
}
// ... or into this warp's 32 x 32 staging block (SWIZZLE_128B: row = lane, 16-byte chunk c at c ^ (lane & 7): a quarter-warp
// covers all 32 banks), from where ONE TMA store writes 32 full 128-byte row segments (clipped at the tensor bounds)
template <bool MASK>
__device__ __forceinline__ void epilogue_stage(const EpiCtx& e, const uint32_t* r, int n0, uint32_t buf, int lane) {
    float v[32];
    epilogue_compute<32>(e, r, n0, v);
    const uint32_t row = buf + (uint32_t)lane * 128u;
    if (MASK && e.mbuf) {
        // the mask block has the staging block's layout (TMA SWIZZLE_128B box {32 n, 32 m}): same offsets, 16 bytes at a time
        const uint32_t mrow = e.mbuf + (uint32_t)lane * 128u;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const uint32_t off = (uint32_t)((c ^ (lane & 7)) << 4);
            const float4 x = lds128(mrow + off);
            sts128(row + off, make_float4(x.x > 0.f ? v[4 * c] * e.mask_scale : 0.f, x.y > 0.f ? v[4 * c + 1] * e.mask_scale : 0.f,
                                          x.z > 0.f ? v[4 * c + 2] * e.mask_scale : 0.f, x.w > 0.f ? v[4 * c + 3] * e.mask_scale : 0.f));
        }
        return;
    }
#pragma unroll
    for (int c = 0; c < 8; ++c)
        sts128(row + (uint32_t)((c ^ (lane & 7)) << 4), make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]));
}
// one accumulator tile: the TMEM load of chunk c+1 is in flight while chunk c is written out
template <int W>
__device__ __forceinline__ void epilogue_tile(const EpiCtx& e, uint32_t taddr, int n_base, int n_tile) {
    uint32_t ra[W], rb[W];
    const int nch = n_tile / W;
    tmem_ld<W>(taddr, ra);
    for (int c = 0; c < nch; c += 2) {
        tmem_ld_fence<W>(ra);
        if (c + 1 < nch) tmem_ld<W>(taddr + (uint32_t)((c + 1) * W), rb);
        epilogue_emit<W>(e, ra, n_base + c * W);
        if (c + 1 < nch) {
            tmem_ld_fence<W>(rb);
            if (c + 2 < nch) tmem_ld<W>(taddr + (uint32_t)((c + 2) * W), ra);
            epilogue_emit<W>(e, rb, n_base + (c + 1) * W);
        }
    }
}

// the same walk with the 32-column chunks leaving through shared memory + TMA (two staging blocks per warp, toggled per
// chunk; a block is reused once the bulk group that read it has finished reading); a 16-column tail goes out directly
template <bool MASK>
__device__ __forceinline__ void epilogue_chunk_tma(const EpiCtx& e, const uint32_t* r, int n0, const CUtensorMap* mapC,
                                                   uint32_t stage0, int& buf, int m0, int lane) {
    if (n0 >= e.N) return;                              // warp-uniform
    if (lane == 0) bulk_wait_read<1>();                 // the group that last read this block (two chunks ago) is done
    __syncwarp();
    const uint32_t sb = stage0 + (uint32_t)buf * 4096u;
    epilogue_stage<MASK>(e, r, n0, sb, lane);
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) { tma_store_2d(mapC, sb, n0, m0); bulk_commit(); }
    buf ^= 1;
}
// TMA-loaded dgrad mask: one 32 x 32 block per epilogue warp, requested one chunk ahead (the first chunk of a tile before the
// accumulator is awaited), landing on the warp's own mbarrier.  Read per thread from global memory the same 4 KB are eight 16-byte
// pieces of 32 different lines per load instruction -- 2x the sectors and 8x the L1 wavefronts: +41 us on the 300 -> 200 dgrad.
// (the block and its barrier are addressed from the warp's C staging area: nothing but the barrier phase stays live)
__device__ __forceinline__ void mask_request(const CUtensorMap* mapM, uint32_t mbuf, uint32_t mbar, int n0, int m0, int lane) {
    if (lane == 0) {
        mbar_expect_tx(mbar, 4096u);
        tma_load_2d(mbuf, mapM, n0, m0, mbar);
    }
}
template <bool MASK>
__device__ __forceinline__ void epilogue_tile_tma(const EpiCtx& e, uint32_t taddr, int n_base, int n_tile, const CUtensorMap* mapC,
                                                  uint32_t stage0, int& buf, int m0, int lane, const CUtensorMap* mapM,
                                                  uint32_t mbar, uint32_t& mphase) {
    const int nch = n_tile / 32;
    for (int c = 0; c < nch; ++c) {
        uint32_t ra[32];
        tmem_ld<32>(taddr + (uint32_t)(c * 32), ra);
        tmem_ld_fence<32>(ra);
        const int n0 = n_base + c * 32;
        if (MASK && e.mbuf && n0 < e.N) {                   // warp-uniform
            mbar_wait(mbar, mphase);
            mphase ^= 1;
        }
        epilogue_chunk_tma<MASK>(e, ra, n0, mapC, stage0, buf, m0, lane);      // ends behind a __syncwarp: every lane has read the mask block
        if (MASK && e.mbuf && c + 1 < nch && n0 + 32 < e.N) mask_request(mapM, e.mbuf, mbar, n0 + 32, m0, lane);
    }
    if (n_tile & 31) {
        uint32_t rt[16];
        tmem_ld<16>(taddr + (uint32_t)(nch * 32), rt);
        tmem_ld_fence<16>(rt);
        epilogue_emit<16>(e, rt, n_base + nch * 32);
    }
}

// MASK: the dgrad instantiation whose epilogue takes the mask of the layer below from TMA-loaded blocks (its own instantiation:
// the mask pipeline's registers must not cost the other GEMMs theirs -- measured +2-3 us each when it was a runtime switch)
template <bool MASK>
__global__ void __launch_bounds__(THREADS, 1)
gemm3x_tma_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                  const __grid_constant__ CUtensorMap mapBlo, const __grid_constant__ CUtensorMap mapC,
                  const __grid_constant__ CUtensorMap mapM, const Args g) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t raw_bar[MAX_STAGES], full_bar[MAX_STAGES], empty_bar[MAX_STAGES];
    __shared__ __align__(8) uint64_t tmem_full_bar[2], tmem_empty_bar[2];
    __shared__ __align__(8) uint64_t mask_bar[EPI_WARPS];
    __shared__ uint32_t tmem_base_smem;
    __shared__ __align__(16) float s_bias[BIAS_SMEM];

    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool bias_in_smem = g.bias != nullptr && g.n_tiles * g.n_tile <= BIAS_SMEM;
    if (bias_in_smem)
        for (int i = threadIdx.x; i < g.n_tiles * g.n_tile; i += THREADS) s_bias[i] = i < g.N ? __ldg(g.bias + i) : 0.f;
    const uint32_t b_bytes = (uint32_t)g.n_tile * 128u;
    const uint32_t stage_bytes = A_TILE_BYTES + 2 * b_bytes;         // raw A, then B (hi, lo)
    const int total_tiles = g.m_tiles * g.n_tiles * g.splits;

    if (threadIdx.x == 0) {
        for (int s = 0; s < g.stages; ++s) {
            mbar_init(smem_u32(&raw_bar[s]), 1);
            mbar_init(smem_u32(&full_bar[s]), (uint32_t)(CONV_WARPS * 32));
            mbar_init(smem_u32(&empty_bar[s]), 1);
        }
        for (int s = 0; s < EPI_WARPS; ++s) mbar_init(smem_u32(&mask_bar[s]), 1);
        for (int s = 0; s < 2; ++s) {
            mbar_init(smem_u32(&tmem_full_bar[s]), 1);
            mbar_init(smem_u32(&tmem_empty_bar[s]), (uint32_t)(EPI_WARPS * 32));
        }
        fence_barrier_init();
    }
    if (warp == PRODUCER_WARP && lane == 0) {
        tma_prefetch_desc(&mapA);
        tma_prefetch_desc(&mapB);
        if (g.b_presplit) tma_prefetch_desc(&mapBlo);
        if (g.c_tma) tma_prefetch_desc(&mapC);
        if (MASK) tma_prefetch_desc(&mapM);
    }
    if (warp == MMA_WARP) tmem_alloc(smem_u32(&tmem_base_smem), TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_smem;
    if (g.dbg && threadIdx.x == 0) {                       // RLCTR_GEMM_DBG: per-CTA (start, end, SM) behind the stage stamps
        uint64_t now; uint32_t sm;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        asm volatile("mov.u32 %0, %%smid;" : "=r"(sm));
        g.dbg[4096 + 4 * blockIdx.x] = (long long)now;
        g.dbg[4096 + 4 * blockIdx.x + 2] = (long long)sm;
    }

    if (warp < CONV_WARPS) {
        // ================= converters =================
        const int tid = threadIdx.x;
        int stage = 0, dbg_it = 0;
        uint32_t phase = 0;
        TileWalk w{(int)blockIdx.x, 0, 0, 0, 0, 0};
        const bool colsum = g.colsum_part != nullptr && g.a_mn;
        for (; tile_decode(w, g, total_tiles); w.tile += (int)gridDim.x) {
            const bool sum_tile = colsum && w.nt == 0;     // every (split, m-tile) is met exactly once with nt == 0
            float row_sum = 0.f;
            for (int kb = w.kb0; kb < w.kb1; ++kb) {
                mbar_wait(smem_u32(&raw_bar[stage]), phase);
                if (tid == 0) DBG_STAMP(dbg_it, 1);
                if (tid == 96) DBG_STAMP(dbg_it, 12);
                const uint32_t st = smem_u32(smem + (size_t)stage * stage_bytes);
                // this TMEM slot was last read by the MMAs of the previous round of this stage: they retired before the
                // producer refilled the stage (empty_bar), i.e. before raw_bar flipped
                tc_fence_after();
                const uint32_t ta = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(g.a_col0 + stage * 2 * BK);
                row_sum += split_row_to_tmem(st, g.a_mn != 0, tid, ta);
                if (!g.b_presplit) split_tile(st + A_TILE_BYTES, st + A_TILE_BYTES + b_bytes, b_bytes, tid);
                tc_fence_before();
                if (!g.b_presplit) fence_proxy_async();       // generic-proxy smem stores -> visible to the tensor core
                if (tid == 0) DBG_STAMP(dbg_it, 2);
                if (tid == 96) DBG_STAMP(dbg_it, 11);
                ++dbg_it;
                mbar_arrive(smem_u32(&full_bar[stage]));
                if (++stage == g.stages) { stage = 0; phase ^= 1; }
            }
            if (sum_tile) {
                const int m = w.mt * BM + tid;             // thread t owns row m: its k-sum IS the partial column sum
                if (m < g.M) g.colsum_part[(int64_t)w.split * g.M + m] = row_sum;
            }
        }
    } else if (warp == PRODUCER_WARP) {
        // ================= TMA producer =================
        int stage = 0;
        uint32_t phase = 0;
        const uint32_t tx = A_TILE_BYTES + (g.b_presplit ? 2 * b_bytes : b_bytes);
        int dbg_it = 0;
        TileWalk w{(int)blockIdx.x, 0, 0, 0, 0, 0};
        for (; tile_decode(w, g, total_tiles); w.tile += (int)gridDim.x) {
            const int m0 = w.mt * BM, n0 = w.nt * g.n_tile;
            for (int kb = w.kb0; kb < w.kb1; ++kb) {
                mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1);
                if (lane == 0) {
                    DBG_STAMP(dbg_it, 0);
                    const uint32_t bar = smem_u32(&raw_bar[stage]);
                    const uint32_t sa = smem_u32(smem + (size_t)stage * stage_bytes);
                    const uint32_t sb = sa + A_TILE_BYTES;
                    const int k0 = kb * BK;
                    mbar_expect_tx(bar, tx);
                    if (g.a_mn) {
                        for (int j = 0; j < BM / 32; ++j) tma_load_2d(sa + j * 4096, &mapA, m0 + 32 * j, k0, bar);
                    } else {
                        tma_load_2d(sa, &mapA, k0, m0, bar);
                    }
                    if (g.b_mn) {
                        for (int j = 0; j < g.n_tile / 32; ++j) {
                            tma_load_2d(sb + j * 4096, &mapB, n0 + 32 * j, k0, bar);
                            if (g.b_presplit) tma_load_2d(sb + b_bytes + j * 4096, &mapBlo, n0 + 32 * j, k0, bar);
                        }
                    } else {
                        tma_load_2d(sb, &mapB, k0, n0, bar);
                        if (g.b_presplit) tma_load_2d(sb + b_bytes, &mapBlo, k0, n0, bar);
                    }
                }
                __syncwarp();
                ++dbg_it;
                if (++stage == g.stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == MMA_WARP) {
        // ================= MMA issuer =================
        // instruction descriptor (cute::UMMA::InstrDescriptor): D = f32, A = B = tf32, M = 128, N = n_tile,
        // bit 15 / 16 = A / B is MN-major (A comes from TMEM: always K-major)
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(g.b_mn ? 1 : 0) << 16) |
                               ((uint32_t)(g.n_tile >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
        const uint32_t b_step = g.b_mn ? 1024u : (uint32_t)UK * 4u;      // bytes per MMA along K
        int stage = 0;
        uint32_t phase = 0;
        int acc = 0, dbg_it = 0;
        uint32_t acc_phase = 0;
        TileWalk w{(int)blockIdx.x, 0, 0, 0, 0, 0};
        for (; tile_decode(w, g, total_tiles); w.tile += (int)gridDim.x) {
            if (lane == 0) DBG_STAMP(dbg_it, 5);
            mbar_wait(smem_u32(&tmem_empty_bar[acc]), acc_phase ^ 1);  // epilogue drained this accumulator
            if (lane == 0) DBG_STAMP(dbg_it, 6);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(acc * g.acc_stride);
            for (int kb = w.kb0; kb < w.kb1; ++kb) {
                mbar_wait(smem_u32(&raw_bar[stage]), phase);                 // TMA bytes (the pre-split B tiles) landed
                if (lane == 0) DBG_STAMP(dbg_it, 8);
                mbar_wait(smem_u32(&full_bar[stage]), phase);                // converters done
                if (lane == 0) DBG_STAMP(dbg_it, 9);
                tc_fence_after();
                if (lane == 0) DBG_STAMP(dbg_it, 3);
                if (lane == 0) {
                    const uint32_t b_hi = smem_u32(smem + (size_t)stage * stage_bytes) + A_TILE_BYTES, b_lo = b_hi + b_bytes;
                    const uint32_t ta_hi = tmem_base + (uint32_t)(g.a_col0 + stage * 2 * BK), ta_lo = ta_hi + (uint32_t)BK;
                    // the last k-block of a K that is no multiple of 32 is zero-filled by TMA: its all-zero k-steps are not issued
                    const int ksteps = min(BK / UK, (g.K - kb * BK + UK - 1) / UK);
#pragma unroll
                    for (int k = 0; k < BK / UK; ++k) {
                        if (k >= ksteps) break;
                        const uint32_t bo = (uint32_t)k * b_step;
                        const uint64_t dbh = g.b_mn ? desc_mn_major(b_hi + bo) : desc_k_major(b_hi + bo);
                        const uint64_t dbl = g.b_mn ? desc_mn_major(b_lo + bo) : desc_k_major(b_lo + bo);
                        const uint32_t first = (kb > w.kb0 || k > 0) ? 1u : 0u;
                        umma_tf32_ts(d_tmem, ta_lo + (uint32_t)(k * UK), dbh, idesc, first);
                        umma_tf32_ts(d_tmem, ta_hi + (uint32_t)(k * UK), dbl, idesc, 1u);
                        umma_tf32_ts(d_tmem, ta_hi + (uint32_t)(k * UK), dbh, idesc, 1u);
                    }
                    DBG_STAMP(dbg_it, 10);
                    umma_commit(smem_u32(&empty_bar[stage]));                // frees the smem slot when these MMAs retire
                    if (kb == w.kb1 - 1) umma_commit(smem_u32(&tmem_full_bar[acc]));
                    DBG_STAMP(dbg_it, 4);
                }
                ++dbg_it;
                __syncwarp();
                if (++stage == g.stages) { stage = 0; phase ^= 1; }
            }
            if (w.kb1 <= w.kb0 && lane == 0) umma_commit(smem_u32(&tmem_full_bar[acc]));     // empty split
            __syncwarp();
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    } else {
        // ================= epilogue =================
        const int q = warp & 3;                        // TMEM lane quadrant this warp may read
        uint64_t drop_seed = 0, drop_ctr = 0;
        if (g.epi.drop_state) { drop_seed = g.epi.drop_state[0]; drop_ctr = g.epi.drop_state[1]; }
        int acc = 0, dbg_tile = 0, cbuf = 0;
        const uint32_t cstage = smem_u32(smem + (size_t)g.stages * stage_bytes) + (uint32_t)q * 8192u;   // 2 x 4 KB per warp
        uint32_t acc_phase = 0;
        uint32_t mphase = 0;
        TileWalk w{(int)blockIdx.x, 0, 0, 0, 0, 0};
        for (; tile_decode(w, g, total_tiles); w.tile += (int)gridDim.x) {
            const bool empty_split = w.kb1 <= w.kb0;
            // the previous tile's last chunk ended behind a __syncwarp: the block is free for this tile's first chunk
            const uint32_t mbuf = MASK ? cstage + (uint32_t)((EPI_WARPS - q) * 8192 + q * 4096) : 0u;   // behind the C staging blocks
            if (MASK && w.nt * g.n_tile < g.N && g.n_tile >= 32)
                mask_request(&mapM, mbuf, smem_u32(&mask_bar[q]), w.nt * g.n_tile, w.mt * BM + q * 32, lane);
            mbar_wait(smem_u32(&tmem_full_bar[acc]), acc_phase);
            tc_fence_after();
            if (warp == CONV_WARPS + 2 && lane == 0) DBG_STAMP(dbg_tile * (w.kb1 - w.kb0), 7);
            const int m = w.mt * BM + q * 32 + lane;
            EpiCtx e;
            e.crow = g.C + ((int64_t)w.split * g.M + m) * g.ldc;
            e.row_ok = m < g.M;
            e.N = g.N;
            e.cvec = g.cvec;
            e.relu = (g.splits == 1) && g.relu;
            e.bias = (g.splits == 1) ? g.bias : nullptr;
            e.sbias = (g.splits == 1 && g.bias && bias_in_smem) ? s_bias : nullptr;
            e.zero = empty_split;
            e.drop = g.epi.drop_state != nullptr && g.splits == 1;
            e.drop_seed = drop_seed;
            e.drop_base = drop_ctr + (uint64_t)m * (uint64_t)g.N;
            e.drop_thresh = g.epi.drop_thresh;
            e.drop_scale = g.epi.drop_scale;
            e.mask_row = (g.epi.mask_src && g.splits == 1) ? g.epi.mask_src + (int64_t)m * g.epi.mask_ld : nullptr;
            e.mvec = g.epi.mvec;
            e.mask_scale = g.epi.mask_scale;
            e.mbuf = mbuf;
            const uint32_t taddr = tmem_base + (uint32_t)(acc * g.acc_stride) + ((uint32_t)(q * 32) << 16);
            if (g.c_tma) epilogue_tile_tma<MASK>(e, taddr, w.nt * g.n_tile, g.n_tile, &mapC, cstage, cbuf, w.mt * BM + q * 32, lane, &mapM,
                                           smem_u32(&mask_bar[q]), mphase);
            else if (g.n_tile % 32 == 0) epilogue_tile<32>(e, taddr, w.nt * g.n_tile, g.n_tile);
            else epilogue_tile<16>(e, taddr, w.nt * g.n_tile, g.n_tile);
            tc_fence_before();
            if (warp == CONV_WARPS + 2 && lane == 0) DBG_STAMP(dbg_tile * (w.kb1 - w.kb0) + 1, 7);
            ++dbg_tile;
            mbar_arrive(smem_u32(&tmem_empty_bar[acc]));
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        if (g.c_tma && lane == 0) bulk_wait_read<0>();      // the staging blocks must outlive the stores that read them
    }
    tc_fence_before();
    __syncthreads();
    if (g.dbg && threadIdx.x == 0) {
        uint64_t now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        g.dbg[4096 + 4 * blockIdx.x + 1] = (long long)now;
    }
    if (warp == MMA_WARP) tmem_dealloc(tmem_base, TMEM_COLS);
}

// (hi, lo) images of a weight matrix [rows, cols] -> [rows, pitch] (pitch % 4 == 0, zero padded): the B
// operand of forward (K-major) and dgrad (MN-major) reads them through TMA without any conversion.
__global__ void __launch_bounds__(256)
split_weight_kernel(const float* __restrict__ w, float* __restrict__ hi, float* __restrict__ lo, int rows, int cols, int pitch) {
    const int64_t total = (int64_t)rows * pitch;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / pitch), c = (int)(i - (int64_t)r * pitch);
        const float x = c < cols ? __ldg(w + (int64_t)r * cols + c) : 0.f;
        const float h = tf32_rn(x);
        hi[i] = h;
        lo[i] = x - h;
    }
}

// ---- host side ------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}
// fp32 tensor [dim1][dim0] (dim0 contiguous, `pitch` floats between rows), box {32, box1}, SWIZZLE_128B, zero fill
static bool make_map(CUtensorMap* map, const float* ptr, int64_t dim0, int64_t dim1, int64_t pitch, int box1,
                     bool mn_major = false) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return false;
    cuuint64_t dims[2] = {(cuuint64_t)dim0, (cuuint64_t)dim1};
    cuuint64_t strides[1] = {(cuuint64_t)pitch * sizeof(float)};
    cuuint32_t box[2] = {32u, (cuuint32_t)box1};
    cuuint32_t estr[2] = {1u, 1u};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}
static bool tma_ok(const float* p, int64_t pitch) { return p && (((uintptr_t)p) & 15u) == 0 && pitch % 4 == 0 && pitch > 0; }

static int env_int(const char* name, int dflt) {
    const char* s = getenv(name);
    return s && *s ? atoi(s) : dflt;
}
int enabled() {
    return env_int("RLCTR_GEMM_TMA", 1) != 0 && encode_fn() != nullptr;   // env read per call: tests switch paths
}

static constexpr int round_to(int n, int q) { return (n + q - 1) / q * q; }

// Tile-width cap: a 160-column tile leaves three 56 KB stages in shared memory and three (A_hi | A_lo) stages in tensor memory;
// 128 measured slower (profiles/r2p_gemm_probes.md).
constexpr int NT_MAX = 160;
static_assert(NT_MAX % 32 == 0 && NT_MAX <= 256, "every tile width make_plan picks must be a UMMA N for both operand majors");
// A always lives in tensor memory, behind the two accumulator stages: the widest tile must leave it room for two stages
static_assert((TMEM_COLS - 2 * round_to(NT_MAX, 32)) / (2 * BK) >= 2, "a full-width tile must leave two TMEM stages of A");

struct Plan {
    int n_tile, n_tiles, m_tiles, splits, kb_per_split, stages;
    int acc_stride, a_col0, c_tma;
    size_t smem;
};
constexpr size_t C_STAGE_BYTES = (size_t)EPI_WARPS * 2 * 4096;     // two 32 x 32 fp32 blocks per epilogue warp
constexpr size_t M_STAGE_BYTES = (size_t)EPI_WARPS * 4096;         // one 32 x 32 mask block per epilogue warp (dgrad, behind C's)
static Plan make_plan(int M, int N, int K, bool b_mn, bool allow_split, bool c_tma_ok = false) {
    Plan p;
    const int q = b_mn ? 32 : 16;
    p.n_tiles = (N + NT_MAX - 1) / NT_MAX;
    p.n_tile = round_to((N + p.n_tiles - 1) / p.n_tiles, q);
    p.m_tiles = (M + BM - 1) / BM;
    const int kb_total = (K + BK - 1) / BK;
    p.splits = 1;
    if (allow_split) {
        const int tiles = p.m_tiles * p.n_tiles;
        int s = RLCTR_SMS / (tiles > 0 ? tiles : 1);
        if (s < 1) s = 1;
        int max_s = kb_total / 8;
        if (max_s < 1) max_s = 1;
        p.splits = s < max_s ? s : max_s;
    }
    p.kb_per_split = (kb_total + p.splits - 1) / p.splits;
    if (p.kb_per_split < 1) p.kb_per_split = 1;
    p.splits = (kb_total + p.kb_per_split - 1) / p.kb_per_split;
    if (p.splits < 1) p.splits = 1;
    // tensor memory: two accumulator stages of the tile width, then (512 - 2 * acc_stride) / 64 stages of (A_hi | A_lo);
    // shared memory carries the raw A tile and B (hi, lo) per stage
    p.acc_stride = round_to(p.n_tile, 32);
    p.a_col0 = 2 * p.acc_stride;
    const int tmem_stages = (TMEM_COLS - p.a_col0) / (2 * BK);
    const size_t stage_bytes = (size_t)A_TILE_BYTES + 2 * (size_t)p.n_tile * 128;
    int st = (int)((size_t)(220 * 1024) / stage_bytes);
    if (st > MAX_STAGES) st = MAX_STAGES;
    if (st > tmem_stages) st = tmem_stages;
    p.stages = st;
    // TMA-stored C: only when the staging blocks fit beside the pipeline without costing it a stage, and never for split-K
    // partials (a box clipped at the tensor bound, not at the split's M rows, would spill into the next split)
    p.c_tma = (c_tma_ok && p.splits == 1 && stage_bytes * st + C_STAGE_BYTES <= (size_t)(220 * 1024)) ? 1 : 0;
    p.smem = stage_bytes * st + (p.c_tma ? C_STAGE_BYTES : 0) + 1024;
    return p;
}
int plan_splits(int M, int N, int K, bool b_mn) { return make_plan(M, N, K, b_mn, true).splits; }

static int vec_of(const float* p, int64_t pitch) {
    const uintptr_t a = (uintptr_t)p;
    if (pitch % 4 == 0 && a % 16 == 0) return 4;
    if (pitch % 2 == 0 && a % 8 == 0) return 2;
    return 1;
}

int split_weight(const float* w, float* hi, float* lo, int rows, int cols, int pitch, cudaStream_t st) {
    const int64_t total = (int64_t)rows * pitch;
    int64_t blocks = (total + 255) / 256;
    split_weight_kernel<<<(unsigned)(blocks < RLCTR_SMS * 4 ? blocks : RLCTR_SMS * 4), 256, 0, st>>>(w, hi, lo, rows, cols, pitch);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

// RLCTR_EUNSUPPORTED: the caller falls back to the software-staged kernel (mlp.cu)
int gemm(const Operand& A, const Operand& B, float* C, int64_t ldc, const float* bias, int M, int N, int K, int relu,
         bool allow_split, cudaStream_t st, const Epilogue* epi, float* colsum_part) {
    if (!enabled()) return RLCTR_EUNSUPPORTED;
    if (!tma_ok(A.ptr, A.pitch) || !tma_ok(B.ptr, B.pitch) || (B.lo && !tma_ok(B.lo, B.pitch))) return RLCTR_EUNSUPPORTED;
    if (A.lo) return RLCTR_EUNSUPPORTED;                  // the streamed operand is always converted in the kernel
    const Plan p = make_plan(M, N, K, B.mn_major, allow_split, tma_ok(C, ldc));
    CUtensorMap mA, mB, mBlo;
    // K-major operand [R rows][K]: dims {K, R}, box {32, tile rows}.  MN-major operand [K rows][R]: dims {R, K}, box {32, 32}.
    bool ok = A.mn_major ? make_map(&mA, A.ptr, M, K, A.pitch, 32, true) : make_map(&mA, A.ptr, K, M, A.pitch, BM);
    ok = ok && (B.mn_major ? make_map(&mB, B.ptr, N, K, B.pitch, 32, true) : make_map(&mB, B.ptr, K, N, B.pitch, p.n_tile));
    if (B.lo) ok = ok && (B.mn_major ? make_map(&mBlo, B.lo, N, K, B.pitch, 32, true) : make_map(&mBlo, B.lo, K, N, B.pitch, p.n_tile));
    else mBlo = mB;
    CUtensorMap mC = mA, mM = mA;
    if (p.c_tma) ok = ok && make_map(&mC, C, N, M, ldc, 32);          // box {32 n, 32 m}, SWIZZLE_128B
    if (!ok) return RLCTR_EUNSUPPORTED;
    // the dgrad mask through TMA: beside TMA-stored C, when its blocks fit behind the pipeline and the mask rows are addressable
    size_t smem = p.smem;
    bool m_tma = false;
    if (epi && epi->mask_src && p.c_tma && p.splits == 1 && tma_ok(epi->mask_src, epi->mask_ld) && p.smem + M_STAGE_BYTES <= (size_t)(221 * 1024) &&
        make_map(&mM, epi->mask_src, N, M, epi->mask_ld, 32)) {
        m_tma = true;
        smem += M_STAGE_BYTES;
    }
    Args g;
    g.C = C; g.ldc = ldc; g.cvec = vec_of(C, ldc); g.bias = bias;
    g.M = M; g.N = N; g.K = K;
    g.n_tile = p.n_tile; g.m_tiles = p.m_tiles; g.n_tiles = p.n_tiles; g.splits = p.splits; g.kb_per_split = p.kb_per_split;
    g.stages = p.stages;
    g.acc_stride = p.acc_stride; g.a_col0 = p.a_col0; g.c_tma = p.c_tma;
    g.a_mn = A.mn_major ? 1 : 0; g.b_mn = B.mn_major ? 1 : 0; g.b_presplit = B.lo ? 1 : 0; g.relu = relu;
    g.colsum_part = (colsum_part && A.mn_major && !bias) ? colsum_part : nullptr;
    if (colsum_part && !g.colsum_part) return RLCTR_EUNSUPPORTED;
    {
        const char* d = getenv("RLCTR_GEMM_DBG");             // hex device address of a zeroed long long [256 * 8] buffer
        g.dbg = (d && *d) ? reinterpret_cast<long long*>(strtoull(d, nullptr, 16)) : nullptr;
    }
    g.epi = epi ? *epi : Epilogue{};
    if ((g.epi.drop_state || g.epi.mask_src) && p.splits != 1) return RLCTR_EUNSUPPORTED;
    if (g.epi.mask_src) g.epi.mvec = vec_of(g.epi.mask_src, g.epi.mask_ld);
    const auto kernel = m_tma ? gemm3x_tma_kernel<true> : gemm3x_tma_kernel<false>;
    RLCTR_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int total = p.m_tiles * p.n_tiles * p.splits;    // persistent CTAs, one per SM
    kernel<<<total < RLCTR_SMS ? total : RLCTR_SMS, THREADS, smem, st>>>(mA, mB, mBlo, mC, mM, g);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

}  // namespace tma
}  // namespace rlctr
