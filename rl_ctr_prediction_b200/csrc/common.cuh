// common.cuh -- shared device helpers for librlctr_sm100a (B200, sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/rlctr.h"

#define RLCTR_FULL 0xffffffffu
#define RLCTR_SMS 148          // B200: 2 dies x 74 SMs; grids are sized in multiples of this

// host-side tally of kernels this library launched (rlctr_launch_count): bench.py reports it as
// `gpu_launches`; it is the only process-global the library keeps and nothing reads it back.
extern unsigned long long g_rlctr_launches;
#define RLCTR_COUNT_LAUNCH(n) __atomic_fetch_add(&g_rlctr_launches, (unsigned long long)(n), __ATOMIC_RELAXED)

#define RLCTR_LAUNCH_CHECK()                         \
    do {                                             \
        cudaError_t e__ = cudaGetLastError();        \
        if (e__ != cudaSuccess) return (int)e__;     \
        RLCTR_COUNT_LAUNCH(1);                       \
    } while (0)

#define RLCTR_CUDA(call)                             \
    do {                                             \
        cudaError_t e__ = (call);                    \
        if (e__ != cudaSuccess) return (int)e__;     \
    } while (0)

static inline bool rlctr_aligned16(const void* p) { return (((uintptr_t)p) & 15u) == 0; }

// lanes-per-row for a fused row of `rs` floats read as float4 chunks: 1, 2, 4, 8 (rs <= 32) or 16 (rs <= 64)
static inline int rlctr_lanes_per_row(int rs) {
    int chunks = rs / 4;
    int l = 1;
    while (l < chunks) l <<= 1;
    return l;
}

// co-located records (rlctr_group_fwd / rlctr_group_rows_adam): 16-byte chunks of the widest joint row
#define RLCTR_GROUP_CHUNKS (RLCTR_GROUP_MAX_FLOATS / 4)
// lanes per row of a vector member's STAND-ALONE table (tables.Geometry.fm: [w?, v_0 .. v_{D-1}] padded to 16 floats, else to 4):
// its row starts at the chunk of its first column in the joint row.  The stand-alone kernels' reduction trees depend on it.
// 0: a stand-alone row wider than 36 floats, which no FM-type model has.
static inline int rlctr_member_lpr(int lin_col, int emb_col, int dim) {
    const int first = (lin_col >= 0 && lin_col < emb_col) ? lin_col : emb_col;
    const int last = lin_col > emb_col + dim - 1 ? lin_col : emb_col + dim - 1;
    const int used = last + 1 - 4 * (first >> 2);
    if (used > 36) return 0;
    return rlctr_lanes_per_row(used <= 16 ? 16 : (used + 3) & ~3);
}

namespace rlctr {

// 128-bit read-only gather of one row chunk.  Rows are touched once per kernel (random ids),
// so skip L1 allocation is NOT requested: neighbouring chunks of one row share 32 B sectors
// across the three per-row requests and L1 merges them.
__device__ __forceinline__ float4 ldg4(const float* p) {
    return __ldg(reinterpret_cast<const float4*>(p));
}
// One-shot gather of a row that nothing else in the kernel re-reads: no L1 allocation, and the L2 fill limited to the 64 bytes
// asked for (the default promotes a miss to the whole 128-byte line: ncu showed 128 B of DRAM reads per 64 B row; rowprobe:
// 36.9 -> 30.8 us for 983,040 random 64 B rows).  SASS: LDG.E.NA.LTC64B.128.CONSTANT.
__device__ __forceinline__ float4 ldg4_once(const float* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::64B.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ float4 ld4(const float* p) {
    return *reinterpret_cast<const float4*>(p);
}
__device__ __forceinline__ void st4(float* p, float4 v) {
    *reinterpret_cast<float4*>(p) = v;
}
// streaming store: outputs written once and not re-read by this kernel
__device__ __forceinline__ void st4_stream(float* p, float4 v) {
    __stcs(reinterpret_cast<float4*>(p), v);
}

__device__ __forceinline__ float4 f4zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float4 f4add(float4 a, float4 b) {
    return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}
__device__ __forceinline__ float f4get(const float4& v, int i) {
    return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w));
}
__device__ __forceinline__ void f4set(float4& v, int i, float x) {
    if (i == 0) v.x = x; else if (i == 1) v.y = x; else if (i == 2) v.z = x; else v.w = x;
}
__device__ __forceinline__ float4 shfl_xor4(float4 v, int off) {
    v.x = __shfl_xor_sync(RLCTR_FULL, v.x, off);
    v.y = __shfl_xor_sync(RLCTR_FULL, v.y, off);
    v.z = __shfl_xor_sync(RLCTR_FULL, v.z, off);
    v.w = __shfl_xor_sync(RLCTR_FULL, v.w, off);
    return v;
}

// torch.sigmoid in fp32: 1/(1+exp(-z)) with the accurate expf (saturates to exactly 0/1 like
// the reference -- SURVEY N2; do not replace with __expf or a logits-BCE).
__device__ __forceinline__ float sigmoidf_ref(float z) { return 1.0f / (1.0f + expf(-z)); }

// ---- torch.optim.Adam (_single_tensor_adam, non-capturable branch), one element ----------
struct AdamHyper {
    float beta2, omb1, omb2, eps, wd;     // omb = float(1 - beta) taken in DOUBLE first, like torch's Python scalars
};
static inline AdamHyper adam_hyper(double beta1, double beta2, double eps, double wd) {
    return AdamHyper{(float)beta2, (float)(1.0 - beta1), (float)(1.0 - beta2), (float)eps, (float)wd};
}

// one step with gradient g (L2 folded in like torch: g += wd*p)
__device__ __forceinline__ void adam_elem(float& p, float& m, float& v, float g, const AdamHyper& h,
                                          float step_size, float bc2_sqrt) {
    g = g + h.wd * p;
    m = m + h.omb1 * (g - m);                           // exp_avg.lerp_(grad, 1-beta1)
    v = v * h.beta2 + h.omb2 * g * g;                   // mul_(beta2).addcmul_(g, g, 1-beta2)
    float denom = sqrtf(v) / bc2_sqrt + h.eps;
    p = p + (-step_size) * m / denom;                   // addcdiv_(exp_avg, denom, value=-step_size)
}

// ---- the L2-only step (g = wd*p): what dense Adam does to a row no sample touched (SURVEY N3) ----------
// These steps are replayed by the million (every row, every step), so they are the one place where the
// IEEE sqrt and divisions are replaced by the SFU approximations: sqrt(v) = v * rsqrt(v) and a / d =
// a * rcp(d) (about 2 ulp each).  The perturbation is ~2e-7 of an update of size ~lr, i.e. ~1e-10 per
// step on parameters of size ~0.1 -- far inside the 1e-5 parity bar -- and it does not accumulate
// faster than sqrt(steps).  Steps that carry a data gradient keep the exact formula (adam_elem).
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rsqrt_approx(float x) {
    float y;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float sqrt_approx(float x) {       // one MUFU.SQRT (sqrt(0) = 0: no guard needed)
    float y;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void adam_l2_elem(float& p, float& m, float& v, const AdamHyper& h, float step_size,
                                             float inv_bc2_sqrt) {
    const float g = h.wd * p;
    m = fmaf(h.omb1, g - m, m);
    v = fmaf(h.omb2 * g, g, v * h.beta2);
    const float denom = fmaf(sqrt_approx(v), inv_bc2_sqrt, h.eps);       // 2 MUFU + 7 FMA-pipe instructions per element-step
    p = fmaf(-step_size * m, rcp_approx(denom), p);
}
// The data step of a TABLE row (gradient g from the batch): same formula as adam_elem with the two IEEE divisions and the IEEE
// square root (~25 instructions each with their fix-up sequences: ncu counted ~770 instructions per lane per row in the update
// kernel, which made it issue-bound at ~90 M warp instructions per launch) replaced by MUFU.SQRT / MUFU.RCP (1-2 ulp each).
// The perturbation is ~3e-7 of an update of size ~lr: ~3e-10 per step on parameters of size ~0.1, four orders of magnitude
// inside the 1e-5 parity bar (tests: final state of every row against torch.optim.Adam).  Dense parameters (bias, tower, policy
// nets: rlctr_dense_adam*) keep the exact adam_elem.
__device__ __forceinline__ void adam_elem_fast(float& p, float& m, float& v, float g, const AdamHyper& h, float step_size,
                                               float inv_bc2_sqrt) {
    g = fmaf(h.wd, p, g);
    m = fmaf(h.omb1, g - m, m);
    v = fmaf(h.omb2 * g, g, v * h.beta2);
    const float denom = fmaf(sqrt_approx(v), inv_bc2_sqrt, h.eps);
    p = fmaf(-step_size * m, rcp_approx(denom), p);
}
__device__ __forceinline__ void adam_l2_step4(float4& p, float4& m, float4& v, float2 s, const AdamHyper& h) {
    const float ib = rcp_approx(s.y);
    adam_l2_elem(p.x, m.x, v.x, h, s.x, ib);
    adam_l2_elem(p.y, m.y, v.y, h, s.x, ib);
    adam_l2_elem(p.z, m.z, v.z, h, s.x, ib);
    adam_l2_elem(p.w, m.w, v.w, h, s.x, ib);
}
// replay the L2-only steps (from, to] a row missed.  sched[t] = (step_size_t, bc2_sqrt_t).
__device__ __forceinline__ void adam_replay4(float4& p, float4& m, float4& v, int from, int to,
                                             const float2* __restrict__ sched, const AdamHyper& h) {
    for (int t = from + 1; t <= to; ++t) adam_l2_step4(p, m, v, __ldg(&sched[t]), h);
}
__device__ __forceinline__ void adam_replay1(float& p, float& m, float& v, int from, int to,
                                             const float2* __restrict__ sched, const AdamHyper& h) {
    for (int t = from + 1; t <= to; ++t) {
        const float2 s = __ldg(&sched[t]);
        adam_l2_elem(p, m, v, h, s.x, rcp_approx(s.y));
    }
}

__device__ __forceinline__ float ldg1_once(const float* p) {       // the same for a single float (the LR weight of a 16-byte record)
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::64B.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
// row-sharded tables: id -> (rank id & mask, local row id >> shift); mask == 0: one local table
struct ShardView {
    const float* peers[RLCTR_MAX_WORLD];
    int shift, mask;
};
__device__ __forceinline__ const float* row_ptr(const float* tab, const ShardView& sv, int64_t id, int pitch) {
    if (sv.mask == 0) return tab + id * pitch;
    return sv.peers[id & sv.mask] + (id >> sv.shift) * (int64_t)pitch;      // NVLink read when the owner is a peer
}
static inline bool shard_view_of(const rlctr_table* t, ShardView* sv) {
    sv->shift = 0; sv->mask = 0;
    for (int r = 0; r < RLCTR_MAX_WORLD; ++r) sv->peers[r] = nullptr;
    if (t->world <= 1) return true;
    if (t->world != 2 && t->world != 4 && t->world != 8) return false;
    while ((1 << sv->shift) < t->world) ++sv->shift;
    sv->mask = t->world - 1;
    for (int r = 0; r < t->world; ++r) {
        if (!t->peers[r]) return false;
        sv->peers[r] = t->peers[r];
    }
    return true;
}

// ---- fixed-order reduction of per-block partials: out[i] = sum_q part[q * stride + i], i < n_a + n_b ----------------------
// One warp per column; lane l adds parts l, l + 32, ... (independent loads: the L2 latency is paid once, not once per part),
// then a butterfly.  The order depends only on `parts`, so results are bit-identical from run to run.  Columns [0, n_a) go to
// out_a, columns [n_a, n_a + n_b) to out_b (either may be null).
static __global__ void __launch_bounds__(256)
colsum_parts_kernel(const float* __restrict__ part, float* __restrict__ out_a, float* __restrict__ out_b, int n_a, int n_b,
                    int64_t stride, int parts) {
    const int lane = threadIdx.x & 31;
    const int col = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (col >= n_a + n_b) return;
    float s = 0.f;
#pragma unroll 8
    for (int q = lane; q < parts; q += 32) s += __ldg(part + (int64_t)q * stride + col);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(RLCTR_FULL, s, off);
    if (lane == 0) {
        if (col < n_a) { if (out_a) out_a[col] = s; }
        else if (out_b) out_b[col - n_a] = s;
    }
}
static inline int colsum_parts_grid(int n) { return (n + 7) / 8; }

// ---- counter-based dropout mask (mlp.cu / mlp_tma.cu / afm.cu) ------------------------------------------------------------
// keep(element) = r16(seed, counter + element index) >= p * 2^16: 16 random bits per element, TWO elements per 32-bit hash
// (elements 2k and 2k+1 take the low / high half of hash(k)), because the mask is drawn in GEMM epilogues where the integer
// pipe is the scarce resource: ~4 integer ops per element instead of ~20.  (seed, counter) live in device memory so that a
// CUDA-graph replay draws a fresh mask every step (rlctr_rng_advance moves the counter).  hash = one round of a 32-bit
// avalanche mix (multiply-xorshift, "lowbias32") of the pair index under a key that folds in the seed and the index's high word.
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
    return x;
}
__device__ __forceinline__ uint32_t dropout_key(uint64_t seed, uint32_t pair_hi) {
    return mix32((uint32_t)seed ^ mix32((uint32_t)(seed >> 32) ^ pair_hi ^ 0x9e3779b9U));
}
__device__ __forceinline__ uint32_t dropout_bits(uint32_t key, uint32_t pair_lo) { return mix32(pair_lo ^ key); }
__device__ __forceinline__ bool dropout_keep(uint64_t seed, uint64_t idx, uint32_t thresh) {
    const uint64_t pair = idx >> 1;
    const uint32_t h = dropout_bits(dropout_key(seed, (uint32_t)(pair >> 32)), (uint32_t)pair);
    return ((idx & 1) ? (h >> 16) : (h & 0xffffu)) >= thresh;
}
static inline uint32_t dropout_thresh(float p) {          // 16-bit threshold: P(drop) = thresh / 65536
    double t = (double)p * 65536.0;
    if (t < 0.0) t = 0.0;
    if (t > 65535.0) t = 65535.0;
    return (uint32_t)t;
}

}  // namespace rlctr
