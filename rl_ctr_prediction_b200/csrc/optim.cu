// optim.cu -- K3: deterministic scatter of embedding-row gradients fused with torch-exact Adam.
//
//   sort (id, slot) pairs  ->  one head lane-group per distinct id walks its run of equal ids
//   (stable sort => slot order, the order aten::embedding_dense_backward accumulates in on CPU)
//   -> Adam on that row in registers -> one write of p, m, v.  No atomics on the data path.
//   Runs longer than LONG_RUN (heavy-hitter ids of Zipf fields) are handed to a block-per-row
//   kernel with a fixed-shape tree so the result stays bit-identical from run to run.
//
// Modes (SURVEY H1): the reference's dense Adam moves EVERY row every step (L2 folded into the
// gradient).  rlctr_adam_flush replays those L2-only steps: called every step it is dense Adam
// (mode A); called lazily (rlctr_rows_catchup for the ids of the batch before the forward,
// rlctr_adam_flush before eval/state_dict) it gives the same numbers with O(touched) traffic
// (mode B).  With stamp == NULL untouched rows are left alone (mode C, "sparse").
#include <cub/device/device_radix_sort.cuh>

#include <cstdlib>

#include "common.cuh"

namespace rlctr {

constexpr int LONG_RUN = 32;

struct TableView {
    float* data;
    int64_t n_rows;
    int rs, lin_col, emb_col, dim;
    int pitch;           // floats between rows of data / exp_avg / exp_avg_sq
    int used;            // columns that carry parameters: chunks past ceil(used/4) are pure padding and are skipped
};
static inline TableView view_of(const rlctr_table* t) {
    int used = t->emb_col + t->dim;
    if (t->lin_col + 1 > used) used = t->lin_col + 1;
    if (used < 1) used = 1;
    return TableView{t->data, t->n_rows, t->row_stride, t->lin_col, t->emb_col, t->dim,
                     t->row_pitch > 0 ? t->row_pitch : t->row_stride, used};
}
struct AdamView {
    float* m;
    float* v;
    int32_t* stamp;      // separate per-row stamps, or
    int stamp_col;       // >= 0: the stamp is the int32 at float offset stamp_col of the row record itself
    const float2* sched;
    const int32_t* step;
    AdamHyper h;
    const float* stage;  // rlctr_rows_lookup's staging array: (p | exp_avg | exp_avg_sq) of the row at sorted position k, already
    int stage_pitch;     // current through *step -- the update reads it instead of the table record (floats per position)
};
// floats per sorted position of the staging array: three blocks of the row's ACTIVE chunks (LR: one float4 [w, m, v, 0])
static inline int stage_pitch_of(const TableView& t) { return t.rs == 1 ? 4 : 3 * ((t.used + 3) & ~3); }
static inline AdamView view_of(const rlctr_adam* a, const TableView& t) {
    return AdamView{a->exp_avg, a->exp_avg_sq, a->stamp_col >= 0 ? nullptr : a->stamp, a->stamp_col >= 0 ? a->stamp_col : -1,
                    reinterpret_cast<const float2*>(a->sched), a->step,
                    adam_hyper(a->beta1, a->beta2, a->eps, a->weight_decay), a->stage, stage_pitch_of(t)};
}
__device__ __forceinline__ bool is_lazy(const AdamView& a) { return a.stamp != nullptr || a.stamp_col >= 0; }
__device__ __forceinline__ int load_stamp(const TableView& t, const AdamView& a, int64_t id) {
    return a.stamp_col >= 0 ? __float_as_int(t.data[id * t.pitch + a.stamp_col]) : a.stamp[id];
}
// in-record stamps travel with the chunk that holds them: patch it before the chunk is stored
__device__ __forceinline__ void embed_stamp(float4& p, int col0, const AdamView& a, int value) {
    if (a.stamp_col >= 0 && (a.stamp_col & ~3) == col0) f4set(p, a.stamp_col & 3, __int_as_float(value));
}
// co-located record (rlctr_group_rows_adam): which member model owns a column of the joint row and what its gradient is made of
struct GroupCols {
    int n;                                   // 0: an ordinary single-model table
    const float* dz[RLCTR_GROUP_MAX];        // dL/dlogit of member m, [B]
    const float* extra[RLCTR_GROUP_MAX];     // dense-tail gradient on member m's latent columns, [B, fields * dim_m], or NULL
    int emb_col[RLCTR_GROUP_MAX], dim[RLCTR_GROUP_MAX];
    int ex_pitch[RLCTR_GROUP_MAX];           // floats between consecutive occurrences' rows of extra[m] (dim, or the interleaved
                                             // receive row of the routed multi-source push)
    const uint32_t* slot_of;                 // non-NULL (routed exchange): sorted_slots holds RECEIVE positions r; the global slot
                                             // (-> sample, for S and dL/dlogit) is slot_of[r], the dense-tail row is extra_m[r]
    int sums_pitch;                          // floats between the sums rows; dz[m] == NULL: dL/dlogit of member m rides in column
                                             // sums_pitch - RLCTR_GROUP_MAX + m of the sample's sums row
    signed char member[RLCTR_GROUP_MAX_FLOATS];  // column -> member, -1: padding / stamp
    signed char role[RLCTR_GROUP_MAX_FLOATS];    // 0 none, 1 first-order weight, 2 latent column with the FM term, 3 latent column without
    signed char lpr[RLCTR_GROUP_MAX];        // lanes per row of member m's stand-alone table (rlctr_member_lpr): its long-run tree
    int dz_used;                             // bit m: a column of member m (role 1 or 2) uses its dL/dlogit.  A member whose row
                                             // gradient is all dense tail (FNN, PNN, DCN: role 3 only) has no dL/dlogit load
};
struct GradView {
    GroupCols grp;
    const float* staged;
    const float* dlogit;
    const float* sums;
    const float* extra;
    int fields;
    int flags;
    // sharded tables: slots are global (src rank * n_per_rank + slot); the four arrays are read from the source
    // rank's buffers over NVLink (peer-mapped pointers)
    int world;
    uint32_t n_per_rank;
    const float* p_staged[RLCTR_MAX_WORLD];
    const float* p_dlogit[RLCTR_MAX_WORLD];
    const float* p_sums[RLCTR_MAX_WORLD];
    const float* p_extra[RLCTR_MAX_WORLD];
};
// the gradient sources of one slot: for a sharded table, those of the rank the slot came from
struct GradSrc {
    const float* staged;
    const float* dlogit;
    const float* sums;
    const float* extra;
    uint32_t slot;
};
__device__ __forceinline__ GradSrc grad_src(const GradView& g, uint32_t slot) {
    if (g.world <= 1) return GradSrc{g.staged, g.dlogit, g.sums, g.extra, slot};
    const uint32_t src = slot / g.n_per_rank;
    return GradSrc{g.p_staged[src], g.p_dlogit[src], g.p_sums[src], g.p_extra[src], slot - src * g.n_per_rank};
}
static inline GradView grad_view_of(const rlctr_rowgrad* grad) {
    GradView g{};
    g.staged = grad->staged; g.dlogit = grad->dlogit; g.sums = grad->sums; g.extra = grad->extra;
    g.fields = grad->fields; g.flags = grad->flags;
    g.world = grad->world; g.n_per_rank = grad->n_per_rank;
    if (grad->world > 1) {
        for (int r = 0; r < grad->world && r < RLCTR_MAX_WORLD; ++r) {
            g.p_staged[r] = grad->peer_staged[r]; g.p_dlogit[r] = grad->peer_dlogit[r];
            g.p_sums[r] = grad->peer_sums[r]; g.p_extra[r] = grad->peer_extra[r];
        }
        g.staged = grad->peer_staged[0]; g.dlogit = grad->peer_dlogit[0]; g.sums = grad->peer_sums[0]; g.extra = grad->peer_extra[0];
    }
    return g;
}

__global__ void __launch_bounds__(256)
sort_prep_kernel(const int64_t* __restrict__ ids, int64_t n, int64_t n_rows, uint32_t* __restrict__ keys,
                 uint32_t* __restrict__ vals) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t id = __ldg(ids + i);
        keys[i] = ((uint64_t)id < (uint64_t)n_rows) ? (uint32_t)id : (uint32_t)n_rows;   // out-of-range -> sentinel, sorted last
        vals[i] = (uint32_t)i;
    }
}

// sharded tables: keys are the local rows of the ids this rank owns; the rest sorts last (sentinel = n_local)
__global__ void __launch_bounds__(256)
sort_prep_sharded_kernel(const uint32_t* __restrict__ ids_all, int64_t n_all, int64_t n_rows_global, int shift, uint32_t mask,
                         uint32_t rank, uint32_t n_local, uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_all; i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t id = __ldg(ids_all + i);
        const bool mine = (uint64_t)id < (uint64_t)n_rows_global && (id & mask) == rank;
        keys[i] = mine ? (id >> shift) : n_local;
        vals[i] = (uint32_t)i;
    }
}

// gradient of columns col0..col0+3 of the row gathered at `slot` (rlctr_rowgrad in rlctr.h), in two halves so that a kernel can
// issue the loads of several rows before it consumes any of them: rowgrad_load (memory) and rowgrad_combine (arithmetic)
struct GradRaw {
    float4 r;            // staged[slot]
    float4 S;            // sums[b]
    float dz;
    float ex[4];         // extra[b, f*dim + col - emb_col]
    bool fm, has_ex, any;
};
__device__ __forceinline__ GradRaw rowgrad_load(const GradView& g, uint32_t gslot, int col0, const TableView& t) {
    const GradSrc q = grad_src(g, gslot);
    const uint32_t slot = q.slot;
    GradRaw w;
    w.r = f4zero(); w.S = f4zero(); w.dz = 0.f; w.fm = false; w.has_ex = false; w.any = false;
#pragma unroll
    for (int k = 0; k < 4; ++k) w.ex[k] = 0.f;
    if (q.staged) w.r = ldg4(q.staged + (int64_t)slot * t.rs + col0);
    if (g.flags & RLCTR_STAGED_PARTNER) {               // FFM: d z / d row is staged, scale by dL/dz
        w.dz = __ldg(q.dlogit + slot / (uint32_t)g.fields);
        return w;
    }
    if (q.dlogit || q.extra) {
        w.any = true;
        const uint32_t b = slot / (uint32_t)g.fields;
        const uint32_t f = slot - b * (uint32_t)g.fields;
        w.fm = q.sums && q.dlogit;
        if (w.fm && (g.flags & RLCTR_DZ_IN_SUMS)) w.dz = __ldg(q.sums + (int64_t)b * t.rs + (t.rs - 1));   // same line as S
        else if (q.dlogit) w.dz = __ldg(q.dlogit + b);
        if (w.fm) w.S = ldg4(q.sums + (int64_t)b * t.rs + col0);
        if (q.extra) {
            w.has_ex = true;
            const float* ex = q.extra + ((int64_t)b * g.fields + f) * t.dim;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int col = col0 + k;
                if (col >= t.emb_col && col < t.emb_col + t.dim) w.ex[k] = __ldg(ex + col - t.emb_col);
            }
        }
    }
    return w;
}
__device__ __forceinline__ float4 rowgrad_combine(const GradView& g, const GradRaw& w, int col0, const float4& p, const TableView& t) {
    float4 r = w.r;
    if (g.flags & RLCTR_STAGED_PARTNER) return make_float4(w.dz * r.x, w.dz * r.y, w.dz * r.z, w.dz * r.w);
    if (w.any) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int col = col0 + k;
            float add = 0.f;
            // explicit roundings (no FMA contraction): rowgrad_group below must give the same bits for the same member
            if (col == t.lin_col) {
                add = w.dz;
            } else if (col >= t.emb_col && col < t.emb_col + t.dim) {
                if (w.fm) add = __fmul_rn(w.dz, f4get(w.S, k) - f4get(p, k));
                if (w.has_ex) add = __fadd_rn(add, w.ex[k]);
            }
            f4set(r, k, __fadd_rn(f4get(r, k), add));
        }
    }
    return r;
}
// Co-located record: the four columns of a lane may belong to different member models.  (member, role) of each column are
// looked up once per thread; per occurrence the lane reads S (one float4 of the joint column sums, coalesced with the other
// chunks of the row), the dL/dlogit of the members it holds columns of, and the dense-tail terms.
struct GroupLane {
    int mem[4], role[4];
};
__device__ __forceinline__ GroupLane group_lane(const GradView& g, int col0) {
    GroupLane gl;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int col = col0 + k;
        gl.mem[k] = col < RLCTR_GROUP_MAX_FLOATS ? (int)g.grp.member[col] : -1;
        gl.role[k] = col < RLCTR_GROUP_MAX_FLOATS ? (int)g.grp.role[col] : 0;
    }
    return gl;
}
// gradient of one column of a co-located record for one occurrence (the arithmetic every group kernel shares, so that they agree
// bit for bit): role 1 first-order weight, 2 latent column with the FM term, 3 latent column without, 0 padding
__device__ __forceinline__ float group_col_grad(int role, float dz, float S, float p, bool has_ex, float ex) {
    float add = 0.f;
    if (role == 1) {
        add = dz;
    } else if (role != 0) {
        if (role == 2) add = __fmul_rn(dz, S - p);
        if (has_ex) add = __fadd_rn(add, ex);
    }
    return __fadd_rn(0.f, add);
}
__device__ __forceinline__ float4 rowgrad_group(const GradView& g, const GroupLane& gl, uint32_t slot, int col0, const float4& p,
                                                const TableView& t) {
    const uint32_t erow = slot;                          // row of the dense-tail gradients: the slot, or the receive position
    if (g.grp.slot_of) slot = __ldg(g.grp.slot_of + slot);
    const uint32_t b = slot / (uint32_t)g.fields;
    const float* srow = g.sums + (int64_t)b * g.grp.sums_pitch;
    const float4 S = ldg4(srow + col0);
    float4 r = f4zero();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int m = gl.mem[k];
        if (m < 0) continue;
        const float* dzp = g.grp.dz[m];
        const bool want_dz = gl.role[k] == 1 || gl.role[k] == 2;
        const float dz = !want_dz ? 0.f : dzp ? __ldg(dzp + b) : __ldg(srow + g.grp.sums_pitch - RLCTR_GROUP_MAX + m);
        const float* ex = gl.role[k] >= 2 ? g.grp.extra[m] : nullptr;
        const float exv = ex ? __ldg(ex + (int64_t)erow * g.grp.ex_pitch[m] + (col0 + k - g.grp.emb_col[m])) : 0.f;
        f4set(r, k, group_col_grad(gl.role[k], dz, f4get(S, k), f4get(p, k), ex != nullptr, exv));
    }
    return r;
}
template <bool GROUP>
__device__ __forceinline__ float4 rowgrad_any(const GradView& g, const GroupLane& gl, uint32_t slot, int col0, const float4& p,
                                              const TableView& t) {
    if (GROUP) return rowgrad_group(g, gl, slot, col0, p, t);
    return rowgrad_combine(g, rowgrad_load(g, slot, col0, t), col0, p, t);
}
__device__ __forceinline__ float4 rowgrad_chunk(const GradView& g, uint32_t gslot, int col0, const float4& p,
                                                const TableView& t) {
    return rowgrad_combine(g, rowgrad_load(g, gslot, col0, t), col0, p, t);
}

__device__ __forceinline__ void adam_apply4(float4& p, float4& m, float4& v, const float4& g, float2 s,
                                            const AdamHyper& h) {
    const float ib = rcp_approx(s.y);
    adam_elem_fast(p.x, m.x, v.x, g.x, h, s.x, ib);
    adam_elem_fast(p.y, m.y, v.y, g.y, h, s.x, ib);
    adam_elem_fast(p.z, m.z, v.z, g.z, h, s.x, ib);
    adam_elem_fast(p.w, m.w, v.w, g.w, h, s.x, ib);
}

// The per-record update of the row kernels is a policy: the gradient side (run walk, long-run tree, co-located roles, peer reads,
// routed slots) is shared, the step applied to the reduced gradient is AdamStep or AdagradStep.  Both see the record through an
// AdamView: for Adagrad `m` is the state sum, `v` is never touched (TWO == false), `sched` points at the fp32 clr table and
// `h` carries only eps and weight_decay.  coef(t) is the per-step scalar pair the step needs.
struct AdamStep {
    static constexpr bool TWO = true;                    // the record's third block (exp_avg_sq) is read and written
    __device__ static __forceinline__ float2 coef(const float2* __restrict__ sched, int t) { return __ldg(&sched[t]); }
    __device__ static __forceinline__ void apply4(float4& p, float4& m, float4& v, const float4& g, float2 s, const AdamHyper& h) {
        adam_apply4(p, m, v, g, s, h);
    }
    __device__ static __forceinline__ void l2_step4(float4& p, float4& m, float4& v, float2 s, const AdamHyper& h) {
        adam_l2_step4(p, m, v, s, h);
    }
    __device__ static __forceinline__ void replay4(float4& p, float4& m, float4& v, int from, int to, const float2* __restrict__ sched,
                                                   const AdamHyper& h) {
        adam_replay4(p, m, v, from, to, sched, h);
    }
    __device__ static __forceinline__ void apply1(float& p, float& m, float& v, float g, float2 s, const AdamHyper& h) {
        adam_elem_fast(p, m, v, g, h, s.x, rcp_approx(s.y));
    }
    __device__ static __forceinline__ void replay1(float& p, float& m, float& v, int from, int to, const float2* __restrict__ sched,
                                                   const AdamHyper& h) {
        adam_replay1(p, m, v, from, to, sched, h);
    }
};
// torch.optim.Adagrad on a table element: sqrt(s) and the division by (sqrt(s) + eps) on the SFU (MUFU.SQRT, MUFU.RCP), the form
// of adam_elem_fast; the L2-only step is this step with g = 0 (fmaf(wd, p, 0) == wd * p), so the lazy replay and a dense step give
// the same bits.  Dense parameters keep IEEE sqrt and division (dense_adagrad_multi_kernel).
__device__ __forceinline__ void adagrad_elem_fast(float& p, float& s, float g, float clr, const AdamHyper& h) {
    g = fmaf(h.wd, p, g);
    s = fmaf(g, g, s);
    p = fmaf(-clr * g, rcp_approx(sqrt_approx(s) + h.eps), p);
}
struct AdagradStep {
    static constexpr bool TWO = false;
    __device__ static __forceinline__ float2 coef(const float2* __restrict__ sched, int t) {
        return make_float2(__ldg(reinterpret_cast<const float*>(sched) + t), 0.f);
    }
    __device__ static __forceinline__ void apply4(float4& p, float4& s, float4&, const float4& g, float2 c, const AdamHyper& h) {
        adagrad_elem_fast(p.x, s.x, g.x, c.x, h);
        adagrad_elem_fast(p.y, s.y, g.y, c.x, h);
        adagrad_elem_fast(p.z, s.z, g.z, c.x, h);
        adagrad_elem_fast(p.w, s.w, g.w, c.x, h);
    }
    __device__ static __forceinline__ void l2_step4(float4& p, float4& s, float4& v, float2 c, const AdamHyper& h) {
        apply4(p, s, v, f4zero(), c, h);
    }
    __device__ static __forceinline__ void replay4(float4& p, float4& s, float4& v, int from, int to, const float2* __restrict__ sched,
                                                   const AdamHyper& h) {
        for (int t = from + 1; t <= to; ++t) l2_step4(p, s, v, coef(sched, t), h);
    }
    __device__ static __forceinline__ void apply1(float& p, float& s, float&, float g, float2 c, const AdamHyper& h) {
        adagrad_elem_fast(p, s, g, c.x, h);
    }
    __device__ static __forceinline__ void replay1(float& p, float& s, float& v, int from, int to, const float2* __restrict__ sched,
                                                   const AdamHyper& h) {
        for (int t = from + 1; t <= to; ++t) apply1(p, s, v, 0.f, coef(sched, t), h);
    }
};

// finish one distinct row: Adam (APPLY==0) or store into the dense gradient (APPLY==1)
template <int APPLY, class P = AdamStep>
__device__ __forceinline__ void finish_row(int64_t id, int col0, float4 p, const float4& acc, const TableView& t,
                                           const AdamView& a, float* dense_grad, int step, int stamp_in,
                                           const float4* m_pre = nullptr, const float4* v_pre = nullptr) {
    if (APPLY == 1) {
        st4(dense_grad + id * t.rs + col0, acc);
        return;
    }
    const int64_t off = id * t.pitch + col0;
    float4 m = m_pre ? *m_pre : ld4(a.m + off), v = f4zero();
    if (P::TWO) v = v_pre ? *v_pre : ld4(a.v + off);
    if (is_lazy(a) && !a.stage && stamp_in < step - 1) P::replay4(p, m, v, stamp_in, step - 1, a.sched, a.h);
    P::apply4(p, m, v, acc, P::coef(a.sched, step), a.h);
    embed_stamp(p, col0, a, step);
    st4(t.data + off, p);
    st4(a.m + off, m);
    if (P::TWO) st4(a.v + off, v);
}

// one lane-group (LPR lanes, a float4 chunk each) per sorted position; only run heads work
template <int LPR, int APPLY, bool GROUP = false, class P = AdamStep>
__global__ void __launch_bounds__(256, (LPR > 8 ? 4 : 5))      // 16 / 32 lanes: wide co-located records, 64 registers: no spills
rows_short_kernel(const uint32_t* __restrict__ sorted_ids, const uint32_t* __restrict__ sorted_slots, int64_t n,
                  const __grid_constant__ GradView g, TableView t, AdamView a, float* __restrict__ dense_grad,
                  int32_t* __restrict__ long_count, uint32_t* __restrict__ long_list) {
    GroupLane gl{};
    if (GROUP) gl = group_lane(g, 4 * (int)(threadIdx.x % LPR));
    // Blocks stride the positions (the launch caps the grid at ~1/world of them for a sharded table: 7 of 8 blocks of a full
    // grid would start in the sentinel tail and exit, and launching 100K empty blocks costs more than the update itself).
    const int64_t nblk = (n * LPR + blockDim.x - 1) / blockDim.x;
    for (int64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
    const int64_t gt = blk * blockDim.x + threadIdx.x;
    const int64_t k = gt / LPR;
    const int c = (int)(gt % LPR), col0 = 4 * c;
    // keys are sorted and everything this table does not own (out-of-range ids; for a sharded table the other ranks'
    // ids, G-1 out of G positions) sorts last as a sentinel: a block that STARTS in that tail has nothing to do -- now or later
    const int64_t k_first = (blk * blockDim.x) / LPR;
    if (k_first >= n || __ldg(sorted_ids + k_first) >= (uint64_t)t.n_rows) return;
    bool head = false;
    uint32_t id = 0, slot0 = 0;
    if (k < n) {
        // four independent loads up front: the id, its neighbours (run head? long run?) and the first slot, so that the
        // gradient-side loads (dlogit / sums / extra, addressed by the slot) leave together with the record loads
        id = __ldg(sorted_ids + k);
        const uint32_t prev = k > 0 ? __ldg(sorted_ids + k - 1) : 0xffffffffu;
        const uint32_t far = (k + LONG_RUN < n) ? __ldg(sorted_ids + k + LONG_RUN) : 0xffffffffu;
        slot0 = __ldg(sorted_slots + k);
        head = (id < (uint64_t)t.n_rows) && prev != id;
        if (head && far == id) {
            if (c == 0) long_list[atomicAdd(long_count, 1)] = (uint32_t)k;      // order is irrelevant: rows are independent
            head = false;
        }
    }
    const bool work = head && col0 < ((APPLY == 0) ? ((t.used + 3) & ~3) : t.rs);
    int step = 0, stamp_in = 0;
    if (work) {
        const bool staged = APPLY == 0 && a.stage != nullptr;
        if (APPLY == 0) {
            step = __ldg(a.step) + 1;
            if (is_lazy(a) && !staged) stamp_in = load_stamp(t, a, id);
        }
        const int64_t off = (int64_t)id * t.pitch + col0;
        float4 p, m0 = f4zero(), v0 = f4zero();
        if (staged) {                                    // (p | m | v) of this position, replayed by rlctr_rows_lookup: coalesced
            const float* sp = a.stage + k * a.stage_pitch + col0;
            const int blk = a.stage_pitch / 3;
            p = ldg4(sp); m0 = ldg4(sp + blk); v0 = ldg4(sp + 2 * blk);
        } else {
            p = ld4(t.data + off);                       // issued with m, v: one contiguous record when pitch = 3*rs
            if (APPLY == 0) { m0 = ld4(a.m + off); if (P::TWO) v0 = ld4(a.v + off); }
        }
        float4 acc = rowgrad_any<GROUP>(g, gl, slot0, col0, p, t);
        int64_t kk = k + 1;
        uint32_t nxt = (kk < n) ? __ldg(sorted_ids + kk) : 0xffffffffu;
        while (nxt == id) {                              // further occurrences of the same row, in slot order
            const uint32_t slot = __ldg(sorted_slots + kk);
            ++kk;
            nxt = (kk < n) ? __ldg(sorted_ids + kk) : 0xffffffffu;
            acc = f4add(acc, rowgrad_any<GROUP>(g, gl, slot, col0, p, t));
        }
        if (APPLY == 0 && a.stamp_col >= 0 && !staged) __syncwarp(__activemask());   // every chunk lane has read the in-record stamp
        finish_row<APPLY, P>(id, col0, p, acc, t, a, dense_grad, step, stamp_in, &m0, &v0);
    } else if (P::TWO && APPLY == 0 && a.stage != nullptr && head && col0 < t.rs) {      // (the staging array is Adam's)
        // staged update: the record was NOT read by this kernel, so its lines are not in L2.  Writing only the active chunks
        // would leave half-written 32-byte sectors that L2 has to fill from DRAM first (ncu: +94 MB of reads per launch);
        // the padding chunks are zero by construction (p = m = v = 0 stays 0 under Adam), so write them too: whole 64 B blocks.
        const int64_t off = (int64_t)id * t.pitch + col0;
        st4(t.data + off, f4zero());
        st4(a.m + off, f4zero());
        st4(a.v + off, f4zero());
    }
    if (APPLY == 0 && a.stamp) {
        __syncwarp();                                    // all chunk lanes read the stamp before lane 0 rewrites it
        if (work && c == 0) a.stamp[id] = step;
    }
    }
}

// Update from the lookup's staging array (rlctr_adam.stage): nothing here is a random READ of the table -- (p | m | v) of sorted
// position k arrive as a coalesced stream, the gradient side comes from L2-resident per-sample arrays -- so the kernel is a
// latency pipeline, not a gather.  Each lane group owns R positions per trip and works in three phases: (A) ids / neighbours /
// first slots of all R, (B) every load of all R head rows (stage chunks + gradient side), (C) reduce, Adam, one record write
// each (whole 64-byte blocks).  R rows per lane in flight instead of one, ~20x fewer block launches than one position per thread.
template <int LPR, int R>
__global__ void __launch_bounds__(256, (R > 2 ? 1 : 2))
rows_staged_kernel(const uint32_t* __restrict__ sorted_ids, const uint32_t* __restrict__ sorted_slots, int64_t n,
                   const __grid_constant__ GradView g, const __grid_constant__ TableView t, const __grid_constant__ AdamView a,
                   int32_t* __restrict__ long_count, uint32_t* __restrict__ long_list) {
    constexpr int GPB = 256 / LPR;                       // lane groups per block
    const int grp = threadIdx.x / LPR, c = threadIdx.x % LPR, col0 = 4 * c;
    const int blk = a.stage_pitch / 3;                   // floats per (p | m | v) block of a staged row
    const bool chunk_on = col0 < blk;
    const bool pad_on = !chunk_on && col0 < t.rs;
    const int step = __ldg(a.step) + 1;
    const float2 sc = __ldg(&a.sched[step]);
    for (int64_t base = (int64_t)blockIdx.x * (GPB * R); base < n; base += (int64_t)gridDim.x * (GPB * R)) {
        if (__ldg(sorted_ids + base) >= (uint64_t)t.n_rows) return;     // sorted: nothing but sentinels from here on
        uint32_t id[R], slot0[R];
        bool head[R], multi[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {                    // (A) consecutive lane groups take consecutive positions
            const int64_t k = base + r * GPB + grp;
            id[r] = 0xffffffffu; slot0[r] = 0; head[r] = false; multi[r] = false;
            if (k < n) {
                id[r] = __ldg(sorted_ids + k);
                const uint32_t prev = k > 0 ? __ldg(sorted_ids + k - 1) : 0xffffffffu;
                const uint32_t nxt = (k + 1 < n) ? __ldg(sorted_ids + k + 1) : 0xffffffffu;
                const uint32_t far = (k + LONG_RUN < n) ? __ldg(sorted_ids + k + LONG_RUN) : 0xffffffffu;
                slot0[r] = __ldg(sorted_slots + k);
                head[r] = (id[r] < (uint64_t)t.n_rows) && prev != id[r];
                if (head[r] && far == id[r]) {
                    if (c == 0) long_list[atomicAdd(long_count, 1)] = (uint32_t)k;
                    head[r] = false;
                }
                multi[r] = head[r] && nxt == id[r];
            }
        }
        float4 p[R], m[R], v[R];
        GradRaw gr[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {                    // (B) all loads of all R rows
            if (head[r] && chunk_on) {
                const float* sp = a.stage + (base + r * GPB + grp) * a.stage_pitch + col0;
                p[r] = ldg4(sp); m[r] = ldg4(sp + blk); v[r] = ldg4(sp + 2 * blk);
                gr[r] = rowgrad_load(g, slot0[r], col0, t);
            }
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {                    // (C)
            if (!head[r]) continue;
            const int64_t off = (int64_t)id[r] * t.pitch + col0;
            if (chunk_on) {
                float4 acc = rowgrad_combine(g, gr[r], col0, p[r], t);
                if (multi[r]) {                          // further occurrences of the same row, in slot order
                    int64_t kk = base + r * GPB + grp + 1;
                    uint32_t nx = id[r];
                    while (nx == id[r]) {
                        const uint32_t slot = __ldg(sorted_slots + kk);
                        ++kk;
                        nx = (kk < n) ? __ldg(sorted_ids + kk) : 0xffffffffu;
                        acc = f4add(acc, rowgrad_chunk(g, slot, col0, p[r], t));
                    }
                }
                float4 pp = p[r], mm = m[r], vv = v[r];
                adam_apply4(pp, mm, vv, acc, sc, a.h);
                embed_stamp(pp, col0, a, step);
                st4(t.data + off, pp);
                st4(a.m + off, mm);
                st4(a.v + off, vv);
            } else if (pad_on) {                         // padding chunks are zero by construction: whole 64 B blocks, no sector fills
                st4(t.data + off, f4zero());
                st4(a.m + off, f4zero());
                st4(a.v + off, f4zero());
            }
        }
    }
}

// The same update as a persistent, double-buffered tile pipeline: what streams (the staged rows, the ids and the slots of a tile
// of sorted positions) is copied global -> shared memory ASYNCHRONOUSLY (cp.async, no registers held, no thread waiting) one
// tile ahead of the arithmetic, so the only latency a thread ever waits for is the L2 hit of its gradient-side loads; the record
// writes are the kernel's DRAM traffic.  Tile = TT positions; a lane group (4 lanes) takes positions g and g + 64 of the tile.
namespace tile {
constexpr int TT = 128;                                  // sorted positions per tile
constexpr int IDS = TT + 4 + LONG_RUN;                   // ids k0-4 .. k0+TT+LONG_RUN-1 (previous id at [3], far id at [4+j+LONG_RUN])
__device__ __forceinline__ void cp16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
template <int CH> struct Buf {
    float rows[TT * 12 * CH];
    uint32_t ids[IDS];
    uint32_t slots[TT];
};
template <int CH>
__device__ __forceinline__ void issue(Buf<CH>& b, int64_t tile, int64_t n, const float* __restrict__ stage,
                                      const uint32_t* __restrict__ sorted_ids, const uint32_t* __restrict__ sorted_slots) {
    constexpr int RF = 12 * CH;
    const int64_t k0 = tile * TT;
    const int64_t rows_here = (n - k0 < TT) ? (n - k0) : TT;
    for (int i = threadIdx.x; i < rows_here * (RF / 4); i += blockDim.x) cp16(b.rows + 4 * i, stage + k0 * RF + 4 * i);
    for (int i = threadIdx.x; i < IDS / 4; i += blockDim.x) {
        const int64_t kk = k0 - 4 + 4 * i;
        if (kk >= 0 && kk + 4 <= n) cp16(b.ids + 4 * i, sorted_ids + kk);
        else
            for (int e = 0; e < 4; ++e) b.ids[4 * i + e] = (kk + e >= 0 && kk + e < n) ? __ldg(sorted_ids + kk + e) : 0xffffffffu;
    }
    for (int i = threadIdx.x; i < TT / 4; i += blockDim.x) {
        const int64_t kk = k0 + 4 * i;
        if (kk + 4 <= n) cp16(b.slots + 4 * i, sorted_slots + kk);
        else
            for (int e = 0; e < 4; ++e) b.slots[4 * i + e] = (kk + e < n) ? __ldg(sorted_slots + kk + e) : 0u;
    }
    cp_commit();
}
}  // namespace tile
template <int CH>
__global__ void __launch_bounds__(256, 3)
rows_staged_tile_kernel(const uint32_t* __restrict__ sorted_ids, const uint32_t* __restrict__ sorted_slots, int64_t n,
                        const __grid_constant__ GradView g, const __grid_constant__ TableView t, const __grid_constant__ AdamView a,
                        int32_t* __restrict__ long_count, uint32_t* __restrict__ long_list) {
    using namespace tile;
    constexpr int RF = 12 * CH;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Buf<CH>* bufs = reinterpret_cast<Buf<CH>*>(smem_raw);
    const int grp = threadIdx.x >> 2, c = threadIdx.x & 3, col0 = 4 * c;
    const bool chunk_on = c < CH;
    const bool pad_on = !chunk_on && col0 < t.rs;
    const int step = __ldg(a.step) + 1;
    const float2 sc = __ldg(&a.sched[step]);
    const int64_t tiles = (n + TT - 1) / TT;
    int64_t tl = blockIdx.x;
    if (tl >= tiles) return;
    int cur = 0;
    issue<CH>(bufs[0], tl, n, a.stage, sorted_ids, sorted_slots);
    for (; tl < tiles; tl += gridDim.x, cur ^= 1) {
        const int64_t nt = tl + gridDim.x;
        if (nt < tiles) { issue<CH>(bufs[cur ^ 1], nt, n, a.stage, sorted_ids, sorted_slots); cp_wait<1>(); }
        else cp_wait<0>();
        __syncthreads();
        const Buf<CH>& b = bufs[cur];
        if (b.ids[4] >= (uint64_t)t.n_rows) break;       // sorted: this tile and every later one hold sentinels only
        const int64_t k0 = tl * TT;
        uint32_t id[2];
        bool head[2], multi[2];
        GradRaw gr[2];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int j = grp + 64 * r;
            id[r] = b.ids[4 + j];
            head[r] = (k0 + j < n) && (id[r] < (uint64_t)t.n_rows) && b.ids[3 + j] != id[r];
            if (head[r] && b.ids[4 + j + LONG_RUN] == id[r]) {
                if (c == 0) long_list[atomicAdd(long_count, 1)] = (uint32_t)(k0 + j);
                head[r] = false;
            }
            multi[r] = head[r] && b.ids[5 + j] == id[r];
            if (head[r] && chunk_on) gr[r] = rowgrad_load(g, b.slots[j], col0, t);      // both rows' loads before either is used
        }
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            if (!head[r]) continue;
            const int j = grp + 64 * r;
            const int64_t off = (int64_t)id[r] * t.pitch + col0;
            if (chunk_on) {
                const float* sp = b.rows + j * RF + col0;
                float4 pp = *reinterpret_cast<const float4*>(sp);
                float4 mm = *reinterpret_cast<const float4*>(sp + 4 * CH);
                float4 vv = *reinterpret_cast<const float4*>(sp + 8 * CH);
                float4 acc = rowgrad_combine(g, gr[r], col0, pp, t);
                if (multi[r]) {                          // further occurrences of the same row, in slot order
                    int64_t kk = k0 + j + 1;
                    uint32_t nx = id[r];
                    while (nx == id[r]) {
                        const uint32_t slot = __ldg(sorted_slots + kk);
                        ++kk;
                        nx = (kk < n) ? __ldg(sorted_ids + kk) : 0xffffffffu;
                        acc = f4add(acc, rowgrad_chunk(g, slot, col0, pp, t));
                    }
                }
                adam_apply4(pp, mm, vv, acc, sc, a.h);
                embed_stamp(pp, col0, a, step);
                st4(t.data + off, pp);
                st4(a.m + off, mm);
                st4(a.v + off, vv);
            } else if (pad_on) {                         // padding chunks are zero by construction: whole 64 B blocks, no sector fills
                st4(t.data + off, f4zero());
                st4(a.m + off, f4zero());
                st4(a.v + off, f4zero());
            }
        }
        __syncthreads();                                 // everyone is done with bufs[cur] before the next trip refills it
    }
    cp_wait<0>();
}

// ---- co-located records, TWO lanes per record ------------------------------------------------------------------------------
// rows_short_kernel<8, 0, GROUP> spends eight lanes (six active) on one record and ~580 warp instructions on four of them: the
// per-position bookkeeping (run head? long run? slot -> sample, 64-bit addresses, member / role of every column) is repeated by
// every lane for its one 16-byte chunk, and ncu shows the kernel half issue-bound, half waiting on its own load chain
// (profiles/r2f_ncu_top_kernels.md).  Here a lane owns CH chunks of the record -- lane h of the pair takes chunks h, h+2, h+4
// (, h+6), so each load instruction of the pair covers one whole 32-byte sector of each block -- and does the bookkeeping once
// for 12-16 columns: 16 records per warp instead of 4, no idle lanes, ~2x the records in flight per register.  Same arithmetic
// as the eight-lane kernel, column by column (group_col_grad, adam_apply4): bit-identical results.
template <int CH, class P = AdamStep>
__global__ void __launch_bounds__(256, 2)
group_rows2_kernel(const uint32_t* __restrict__ sorted_ids, const uint32_t* __restrict__ sorted_slots, int64_t n,
                   const __grid_constant__ GradView g, const __grid_constant__ TableView t, const __grid_constant__ AdamView a,
                   int32_t* __restrict__ long_count, uint32_t* __restrict__ long_list) {
    const int h = threadIdx.x & 1;
    const int lane = threadIdx.x & 31;
    const unsigned pmask = 3u << (lane & ~1);
    const int chunks = (t.used + 3) >> 2;
    // per chunk of this lane: packed (member, role) of its four columns, and the dense-tail gradient of its vector member
    int desc[CH];                        // 4 x (role 2 bits | member 2 bits)
    const float* exb[CH];                // extra_m - emb_col_m + col0 of the chunk, or NULL
    int exd[CH];                         // extra_pitch_m
    bool live[CH];
#pragma unroll
    for (int j = 0; j < CH; ++j) {
        const int c = h + 2 * j, col0 = 4 * c;
        live[j] = c < chunks;
        desc[j] = 0; exb[j] = nullptr; exd[j] = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int col = col0 + k;
            const int m = (live[j] && col < 32) ? (int)g.grp.member[col] : -1;
            const int role = m >= 0 ? (int)g.grp.role[col] : 0;
            desc[j] |= ((role & 3) | ((m & 3) << 2)) << (4 * k);
            if (role >= 2 && g.grp.extra[m]) { exb[j] = g.grp.extra[m] + (col0 - g.grp.emb_col[m]); exd[j] = g.grp.ex_pitch[m]; }
        }
    }
    const int sc5 = a.stamp_col >= 0 ? (a.stamp_col >> 2) : 0;         // chunk that holds the in-record stamp
    const int stamp_src = (lane & ~1) + (sc5 & 1), stamp_j = sc5 >> 1;
    const int step = __ldg(a.step) + 1;
    const float2 sc = P::coef(a.sched, step);
    const int64_t G = ((int64_t)gridDim.x * blockDim.x) >> 1;
    for (int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1; k < n; k += G) {
        const uint32_t id = __ldg(sorted_ids + k);
        if (id >= (uint64_t)t.n_rows) return;                            // sorted: nothing but sentinels from here on
        const uint32_t prev = k > 0 ? __ldg(sorted_ids + k - 1) : 0xffffffffu;
        const uint32_t far = (k + LONG_RUN < n) ? __ldg(sorted_ids + k + LONG_RUN) : 0xffffffffu;
        uint32_t slot = __ldg(sorted_slots + k);
        uint32_t nxt = (k + 1 < n) ? __ldg(sorted_ids + k + 1) : 0xffffffffu;
        if (prev == id) continue;                                        // not a run head
        if (far == id) {                                                 // heavy hitter: rows_long_kernel
            if (h == 0) long_list[atomicAdd(long_count, 1)] = (uint32_t)k;
            continue;
        }
        const int64_t off = (int64_t)id * t.pitch + 4 * h;
        float4 p[CH], m[CH], v[CH], acc[CH];
#pragma unroll
        for (int j = 0; j < CH; ++j) {
            p[j] = f4zero(); m[j] = f4zero(); v[j] = f4zero(); acc[j] = f4zero();
            if (live[j]) { p[j] = ld4(t.data + off + 8 * j); m[j] = ld4(a.m + off + 8 * j); if (P::TWO) v[j] = ld4(a.v + off + 8 * j); }
        }
        int64_t kk = k;
        bool first = true;
        while (true) {                                                   // the occurrences of this row, in slot order
            const uint32_t erow = slot;                                  // dense-tail row: the slot, or the receive position
            if (g.grp.slot_of) slot = __ldg(g.grp.slot_of + slot);
            const uint32_t b = slot / (uint32_t)g.fields;
            const float* srow = g.sums + (int64_t)b * g.grp.sums_pitch;
            float dzv[RLCTR_GROUP_MAX];
#pragma unroll
            for (int mm = 0; mm < RLCTR_GROUP_MAX; ++mm) {
                dzv[mm] = 0.f;
                if (mm < g.grp.n && ((g.grp.dz_used >> mm) & 1)) dzv[mm] = g.grp.dz[mm] ? __ldg(g.grp.dz[mm] + b) : __ldg(srow + g.grp.sums_pitch - RLCTR_GROUP_MAX + mm);
            }
#pragma unroll
            for (int j = 0; j < CH; ++j) {
                if (!live[j]) continue;
                const float4 S = ldg4(srow + 4 * (h + 2 * j));
                const float* ex = exb[j] ? exb[j] + (int64_t)erow * exd[j] : nullptr;
                float4 gr;
#pragma unroll
                for (int kq = 0; kq < 4; ++kq) {
                    const int d4 = (desc[j] >> (4 * kq)) & 15, role = d4 & 3, mm = d4 >> 2;
                    const float dz = mm == 0 ? dzv[0] : (mm == 1 ? dzv[1] : (mm == 2 ? dzv[2] : dzv[3]));
                    const bool has_ex = ex != nullptr && role >= 2;
                    const float exv = has_ex ? __ldg(ex + kq) : 0.f;
                    f4set(gr, kq, group_col_grad(role, dz, f4get(S, kq), f4get(p[j], kq), has_ex, exv));
                }
                acc[j] = first ? gr : f4add(acc[j], gr);
            }
            first = false;
            if (nxt != id) break;
            ++kk;
            slot = __ldg(sorted_slots + kk);
            nxt = (kk + 1 < n) ? __ldg(sorted_ids + kk + 1) : 0xffffffffu;
        }
        int stamp_in = step - 1;
        if (a.stamp_col >= 0) {
            float4 pc = p[0];
#pragma unroll
            for (int j = 1; j < CH; ++j)
                if (stamp_j == j) pc = p[j];
            stamp_in = __shfl_sync(pmask, __float_as_int(f4get(pc, a.stamp_col & 3)), stamp_src);
        }
#pragma unroll
        for (int j = 0; j < CH; ++j) {
            if (!live[j]) continue;
            if (a.stamp_col >= 0 && stamp_in < step - 1) P::replay4(p[j], m[j], v[j], stamp_in, step - 1, a.sched, a.h);
            P::apply4(p[j], m[j], v[j], acc[j], sc, a.h);
            embed_stamp(p[j], 4 * (h + 2 * j), a, step);
            st4(t.data + off + 8 * j, p[j]);
            st4(a.m + off + 8 * j, m[j]);
            if (P::TWO) st4(a.v + off + 8 * j, v[j]);
        }
    }
}

// block per long run: NSUB lane-groups stride the run, fixed-shape tree in shared memory
template <int LPR, int APPLY, bool GROUP = false, int NT = 256, class P = AdamStep>
__global__ void __launch_bounds__(NT)
rows_long_kernel(const uint32_t* __restrict__ sorted_ids, const uint32_t* __restrict__ sorted_slots, int64_t n,
                 const __grid_constant__ GradView g, TableView t, AdamView a, float* __restrict__ dense_grad,
                 const int32_t* __restrict__ long_count, const uint32_t* __restrict__ long_list) {
    constexpr int NSUB = NT / LPR;                       // a co-located record (LPR = 8) runs 512 threads: the 64 sub-groups -- and so
    GroupLane gl{};                                      // the partial sums and their tree -- of a stand-alone 16-float row (LPR = 4)
    if (GROUP) gl = group_lane(g, 4 * (int)(threadIdx.x % LPR));
    __shared__ float4 red[NT];
    __shared__ int64_t s_end;
    const int sub = threadIdx.x / LPR, c = threadIdx.x % LPR, col0 = 4 * c;
    const bool chunk_on = col0 < t.rs;
    const int nlong = *long_count;
    for (int li = blockIdx.x; li < nlong; li += gridDim.x) {
        const int64_t k = long_list[li];
        const uint32_t id = __ldg(sorted_ids + k);
        if (threadIdx.x == 0) {                          // upper bound of the run by bisection
            int64_t lo = k, hi = n;                      // ids[lo] == id, ids[hi] > id (or hi == n)
            while (hi - lo > 1) {
                int64_t mid = (lo + hi) >> 1;
                if (__ldg(sorted_ids + mid) == id) lo = mid; else hi = mid;
            }
            s_end = hi;
        }
        __syncthreads();
        const int64_t end = s_end;
        float4 p = f4zero(), acc = f4zero();
        int step = 0, stamp_in = 0;
        const bool staged = APPLY == 0 && a.stage != nullptr;
        const float* sp = staged ? a.stage + k * a.stage_pitch + col0 : nullptr;
        if (chunk_on) {
            p = (staged && col0 < a.stage_pitch / 3) ? ldg4(sp) : ld4(t.data + (int64_t)id * t.pitch + col0);
            for (int64_t kk = k + sub; kk < end; kk += NSUB)
                acc = f4add(acc, rowgrad_any<GROUP>(g, gl, __ldg(sorted_slots + kk), col0, p, t));
            if (APPLY == 0 && sub == 0) {
                step = __ldg(a.step) + 1;
                if (is_lazy(a) && !staged) stamp_in = load_stamp(t, a, id);
            }
        }
        red[threadIdx.x] = acc;
        __syncthreads();
        for (int half = NSUB / 2; half > 0; half >>= 1) {
            if (sub < half) red[threadIdx.x] = f4add(red[threadIdx.x], red[threadIdx.x + half * LPR]);
            __syncthreads();
        }
        if (sub == 0 && chunk_on) {
            if (P::TWO && staged) {                      // (the staging array is Adam's)
                if (col0 < a.stage_pitch / 3) {          // padding chunks carry no parameters: they are never touched
                    const int blk = a.stage_pitch / 3;
                    const float4 m0 = ldg4(sp + blk), v0 = ldg4(sp + 2 * blk);
                    finish_row<APPLY, P>(id, col0, p, red[threadIdx.x], t, a, dense_grad, step, stamp_in, &m0, &v0);
                } else {                                  // whole 64 B blocks (see rows_short_kernel)
                    const int64_t off = (int64_t)id * t.pitch + col0;
                    st4(t.data + off, f4zero()); st4(a.m + off, f4zero()); st4(a.v + off, f4zero());
                }
            } else {
                finish_row<APPLY, P>(id, col0, p, red[threadIdx.x], t, a, dense_grad, step, stamp_in);
            }
        }
        __syncthreads();
        if (APPLY == 0 && a.stamp && threadIdx.x == 0) a.stamp[id] = __ldg(a.step) + 1;
    }
}

// Heavy hitters of a WIDE co-located record (rlctr_group_rows_adam: more than one line, or members whose stand-alone rows are wider
// than 16 floats): block per long run, thread = (chunk, sub-group).  Chunk c sums the run in the sub-groups of its member's
// stand-alone update and pairs them in that kernel's tree: 64 sub-groups for a 16-float row (rows_long_kernel<4>), 32 for 20..32
// floats (rows_long_kernel<8>), one walked in slot order for 36 floats (rows_wide_kernel).  Same per-column arithmetic
// (group_col_grad) and the same Adam step: bit-identical to each member's stand-alone update.
template <class P = AdamStep>
__global__ void __launch_bounds__(256)
group_long_wide_kernel(const uint32_t* __restrict__ sorted_ids, const uint32_t* __restrict__ sorted_slots, int64_t n,
                       const __grid_constant__ GradView g, const __grid_constant__ TableView t, const __grid_constant__ AdamView a,
                       const int32_t* __restrict__ long_count, const uint32_t* __restrict__ long_list) {
    constexpr int SUBS = 64, C = RLCTR_GROUP_CHUNKS, PER = SUBS * C / 256;   // (sub-group, chunk) pairs per thread
    __shared__ float4 red[SUBS * C];
    __shared__ int64_t s_end;
    const int c = threadIdx.x % C, s0 = threadIdx.x / C, col0 = 4 * c;
    const bool chunk_on = c < ((t.used + 3) >> 2);
    const GroupLane gl = group_lane(g, col0);
    int form = 4;                                        // a chunk without latent columns (LR's own): the 16-float form
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (gl.role[k] >= 2) form = g.grp.lpr[gl.mem[k]];
    const int nsub = form == 4 ? 64 : (form == 8 ? 32 : 1);
    const int nlong = *long_count;
    for (int li = blockIdx.x; li < nlong; li += gridDim.x) {
        const int64_t k = long_list[li];
        const uint32_t id = __ldg(sorted_ids + k);
        if (threadIdx.x == 0) {                          // upper bound of the run by bisection
            int64_t lo = k, hi = n;
            while (hi - lo > 1) {
                int64_t mid = (lo + hi) >> 1;
                if (__ldg(sorted_ids + mid) == id) lo = mid; else hi = mid;
            }
            s_end = hi;
        }
        __syncthreads();
        const int64_t end = s_end;
        const float4 p = chunk_on ? ld4(t.data + (int64_t)id * t.pitch + col0) : f4zero();
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            const int sub = s0 + j * (256 / C);
            float4 acc = f4zero();
            if (chunk_on && sub < nsub)
                for (int64_t kk = k + sub; kk < end; kk += nsub) acc = f4add(acc, rowgrad_group(g, gl, __ldg(sorted_slots + kk), col0, p, t));
            red[sub * C + c] = acc;
        }
        const int step = __ldg(a.step) + 1;
        int stamp_in = 0;
        if (s0 == 0 && chunk_on && is_lazy(a)) stamp_in = load_stamp(t, a, id);
        __syncthreads();
        for (int half = SUBS / 2; half > 0; half >>= 1) {
#pragma unroll
            for (int j = 0; j < PER; ++j) {
                const int sub = s0 + j * (256 / C);
                if (sub < half && half < nsub) red[sub * C + c] = f4add(red[sub * C + c], red[(sub + half) * C + c]);
            }
            __syncthreads();
        }
        if (s0 == 0 && chunk_on) finish_row<0, P>(id, col0, p, red[c], t, a, nullptr, step, stamp_in);
        __syncthreads();
        if (a.stamp && threadIdx.x == 0) a.stamp[id] = step;      // a separate stamp array (the in-record stamp rides in p)
    }
}

// wide rows (row_stride > 32 floats: the interleaved FFM table, 36-float FM rows): one WARP per sorted position,
// lanes stride the float4 chunks of the row (WCH chunks per lane); runs are walked sequentially
// in slot order so the sum is bit-identical from run to run.  WCH = 2: rows up to 256 floats; WCH = 4: up to 512
// (FFM at F = 15, D = 18..33).
constexpr int WCH_MAX = 4;
template <int APPLY, int WCH, class P = AdamStep>
__global__ void __launch_bounds__(256)
rows_wide_kernel(const uint32_t* __restrict__ sorted_ids, const uint32_t* __restrict__ sorted_slots, int64_t n,
                 GradView g, TableView t, AdamView a, float* __restrict__ dense_grad) {
    const int lane = threadIdx.x & 31;
    const int64_t k = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (k >= n) return;
    const uint32_t id = __ldg(sorted_ids + k);
    if (id >= (uint64_t)t.n_rows || (k > 0 && __ldg(sorted_ids + k - 1) == id)) return;   // warp-uniform
    const int chunks = t.rs >> 2;
    float4 p[WCH], acc[WCH];
#pragma unroll
    for (int u = 0; u < WCH; ++u) {
        const int c = lane + 32 * u;
        acc[u] = f4zero();
        p[u] = c < chunks ? ld4(t.data + (int64_t)id * t.pitch + 4 * c) : f4zero();
    }
    int64_t kk = k;
    uint32_t nxt = id;
    while (nxt == id) {
        const uint32_t slot = __ldg(sorted_slots + kk);
        ++kk;
        nxt = (kk < n) ? __ldg(sorted_ids + kk) : 0xffffffffu;
#pragma unroll
        for (int u = 0; u < WCH; ++u) {
            const int c = lane + 32 * u;
            if (c < chunks) acc[u] = f4add(acc[u], rowgrad_chunk(g, slot, 4 * c, p[u], t));
        }
    }
    int step = 0, stamp_in = 0;
    if (APPLY == 0) {
        step = __ldg(a.step) + 1;
        if (is_lazy(a)) stamp_in = load_stamp(t, a, id);
        __syncwarp();
    }
#pragma unroll
    for (int u = 0; u < WCH; ++u) {
        const int c = lane + 32 * u;
        if (c < chunks) finish_row<APPLY, P>(id, 4 * c, p[u], acc[u], t, a, dense_grad, step, stamp_in);
    }
    if (APPLY == 0 && a.stamp) {
        __syncwarp();
        if (lane == 0) a.stamp[id] = step;
    }
}
// ---- replay kernels (lazy-exact mode) -------------------------------------------------------------------
// Work items are 16-byte row chunks; every item needs a DIFFERENT number of replay steps (its row's
// staleness), so a one-item-per-thread mapping leaves most lanes of a warp idle while the stalest one
// finishes.  Here each LANE walks its own queue of items: it replays one step per loop iteration and, the
// moment its item is done, stores it and switches to the next one, which was prefetched into registers
// while the current one was being replayed.  Lanes never wait for each other's items.
struct ReplayItem {
    float4 p, m, v;
    int64_t off;         // float offset of the chunk (-1: nothing to do)
    int t;               // steps already applied
};
// FLUSH: items are all chunks of rows [r0, r1).  CATCHUP: items are (sorted position, chunk); only run heads count.
template <bool CATCHUP, class P = AdamStep>
__device__ __forceinline__ void replay_fetch(ReplayItem& it, int64_t k, int c, int64_t n_items, const TableView& t,
                                             const AdamView& a, int64_t r0, const uint32_t* __restrict__ sorted_ids,
                                             int upto) {
    it.off = -1;
    it.t = upto;
    if (k >= n_items) return;
    int64_t row;
    if (CATCHUP) {
        const uint32_t id = __ldg(sorted_ids + k);
        if (id >= (uint64_t)t.n_rows || (k > 0 && __ldg(sorted_ids + k - 1) == id)) return;
        row = id;
    } else {
        row = r0 + k;
    }
    const int st = __ldg(a.stamp + row);
    if (st >= upto) return;
    it.t = st;
    it.off = row * t.pitch + 4 * c;
    it.p = ld4(t.data + it.off);
    it.m = ld4(a.m + it.off);
    it.v = P::TWO ? ld4(a.v + it.off) : f4zero();
}
template <bool CATCHUP, class P = AdamStep>
__global__ void __launch_bounds__(256)
replay_kernel(TableView t, AdamView a, int64_t r0, int64_t n_items, const uint32_t* __restrict__ sorted_ids) {
    const int chunks = (t.used + 3) >> 2;                 // trailing all-padding chunks are never touched
    const uint32_t stride = gridDim.x * blockDim.x;       // items (chunks) between two items of one lane
    const uint32_t dk = stride / chunks, dc = stride % chunks;
    const int upto = __ldg(a.step);
    const uint32_t i0 = blockIdx.x * blockDim.x + threadIdx.x;
    int64_t k = i0 / chunks;                              // (k, c) = item index / chunks, % chunks, advanced incrementally
    int c = (int)(i0 % chunks);
    ReplayItem cur, nxt;
    replay_fetch<CATCHUP, P>(cur, k, c, n_items, t, a, r0, sorted_ids, upto);
    bool cur_real = k < n_items;
    k += dk; c += dc; if (c >= chunks) { c -= chunks; ++k; }
    replay_fetch<CATCHUP, P>(nxt, k, c, n_items, t, a, r0, sorted_ids, upto);
    while (true) {
        if (cur.t >= upto) {                             // current item finished (or was nothing to do): switch
            if (cur.off >= 0) {
                st4(t.data + cur.off, cur.p);
                st4(a.m + cur.off, cur.m);
                if (P::TWO) st4(a.v + cur.off, cur.v);
            }
            if (!cur_real) break;                        // ran past the end of the queue: this lane is done
            cur = nxt;
            cur_real = k < n_items;
            k += dk; c += dc; if (c >= chunks) { c -= chunks; ++k; }
            replay_fetch<CATCHUP, P>(nxt, k, c, n_items, t, a, r0, sorted_ids, upto);
            continue;
        }
        ++cur.t;
        P::l2_step4(cur.p, cur.m, cur.v, P::coef(a.sched, cur.t), a.h);
    }
}
// In-record stamps (stamp_col >= 0): the stamp is part of the record, so ONE lane owns a whole row (all of its
// CH active chunks): it reads the stamp with the data, replays, and writes the new stamp with the data -- no
// separate stamp array, no second random access per row, no ordering problem between the chunks of a row.
template <int CH>
struct ReplayRow {
    float4 p[CH], m[CH], v[CH];
    int64_t off;
    int t;
    uint32_t lost;                                       // UNSORTED: another occurrence of the id claimed the record first
};
// UNSORTED catch-up (rlctr_rows_catchup_ids): the work items are the batch's ids in BATCH order -- no sorted view needed, so the
// sort leaves the critical path of the step.  Every occurrence requests its record; the occurrences of one id are told apart by a
// claim bit per table row (atomicOr on a bitmap zeroed by the call: the first to arrive replays, the others drop the item).
// The result does not depend on who wins: the replay is a function of the record alone.
__device__ __forceinline__ int64_t replay_row_unsorted(int64_t k, int64_t n_items, const int64_t* __restrict__ ids, int64_t n_rows) {
    if (k >= n_items) return -2;
    const int64_t id = __ldg(ids + k);
    return (id >= 0 && id < n_rows) ? id : -1;         // out-of-range ids own no record
}
// row of work item k: FLUSH -> r0 + k; CATCHUP -> the id at sorted position k if that position is a run head
// (-1: nothing to do at this position; -2: past the end -- of the items, or of the ids this table owns: out-of-range and,
// for a sharded table, non-owned ids sort last as sentinels and may outnumber the real ones G-1 to 1).
// The loads it issues are only consumed one item later (software prefetch of the id stream).
template <bool CATCHUP>
__device__ __forceinline__ int64_t replay_row_of(int64_t k, int64_t n_items, int64_t r0, const uint32_t* __restrict__ sorted_ids,
                                                 int64_t n_rows) {
    if (k >= n_items) return -2;
    if (!CATCHUP) return r0 + k;
    const uint32_t id = __ldg(sorted_ids + k);
    const uint32_t prev = k > 0 ? __ldg(sorted_ids + k - 1) : 0xffffffffu;
    if (id >= (uint64_t)n_rows) return -2;             // sentinel: keys are sorted, so nothing but sentinels follows
    return prev != id ? (int64_t)id : -1;
}
// issue the loads of a whole record WITHOUT looking at its stamp first: one DRAM round trip instead of two, and
// nothing in the caller depends on the data until the item becomes current (a full replay of another row later).
// LPRR lanes share a row (co-located records of 5..32 chunks): lane slice h owns chunks h*CH .. h*CH+CH-1, `live` of them active
// (none for the last slices of a record that does not fill them).
template <int CH, bool UNSORTED = false, class P = AdamStep>
__device__ __forceinline__ void replay_row_issue(ReplayRow<CH>& it, int64_t row, const TableView& t, const AdamView& a, int first_col,
                                                 int live, uint32_t* __restrict__ claim = nullptr, bool claimer = false) {
    it.off = row < 0 ? row : row * t.pitch + first_col;
    it.lost = 0;
    if (row >= 0) {
        if (UNSORTED && claimer) {                       // one lane per row; its answer is consumed a whole item later
            const uint32_t bit = 1u << (row & 31);
            it.lost = atomicOr(claim + (row >> 5), bit) & bit;
        }
#pragma unroll
        for (int c = 0; c < CH; ++c) {
            if (c < live) {
                it.p[c] = ld4(t.data + it.off + 4 * c);
                it.m[c] = ld4(a.m + it.off + 4 * c);
                it.v[c] = P::TWO ? ld4(a.v + it.off + 4 * c) : f4zero();
            } else {
                it.p[c] = f4zero(); it.m[c] = f4zero(); it.v[c] = f4zero();
            }
        }
    }
}
// the item becomes current: read the in-record stamp out of the data that has landed; up-to-date rows are dropped
template <int CH, int LPRR, bool UNSORTED = false>
__device__ __forceinline__ void replay_row_arm(ReplayRow<CH>& it, const AdamView& a, int upto, int h) {
    it.t = upto;
    if (it.off < 0) return;                              // the same for every lane of a row
    if (UNSORTED) {
        uint32_t lost = it.lost;
        if (LPRR > 1) {                                  // slice 0 of the row asked
            const int lane = threadIdx.x & 31;
            const unsigned mask = ((1u << LPRR) - 1u) << (lane & ~(LPRR - 1));
            lost = __shfl_sync(mask, lost, lane & ~(LPRR - 1));
        }
        if (lost) { it.off = -1; return; }
    }
    int st;
    if (LPRR == 1) {
        // the in-record stamp sits in the first padding column (= `used`, tables.Geometry.stamp_col), i.e. always in the
        // LAST active chunk: a compile-time register, only the element inside it is a run-time select
        st = __float_as_int(f4get(it.p[CH - 1], a.stamp_col & 3));
    } else {
        // the lane whose slice holds the stamp's chunk hands it to the row's other lanes (they took the same path here: the
        // lanes of a row always have the same staleness, so they switch rows in the same iteration)
        const int sc = a.stamp_col >> 2, hs = sc / CH, lc = sc - hs * CH;
        float4 pc = it.p[0];
#pragma unroll
        for (int c = 1; c < CH; ++c)
            if (lc == c) pc = it.p[c];
        const int lane = threadIdx.x & 31;
        const unsigned mask = ((1u << LPRR) - 1u) << (lane & ~(LPRR - 1));
        st = __shfl_sync(mask, __float_as_int(f4get(pc, a.stamp_col & 3)), (lane & ~(LPRR - 1)) + hs);
    }
    if (st >= upto) it.off = -1; else it.t = st;
}
template <int CH, int LPRR, bool CATCHUP, bool UNSORTED = false, class P = AdamStep>
__global__ void __launch_bounds__(128, (LPRR > 2 ? (CH == 3 ? 3 : 2) : (CH == 3 ? 4 : 3)))   // wide records (LPRR 4, 8): no spills
replay_rows_kernel(TableView t, AdamView a, int64_t r0, int64_t n_items, const uint32_t* __restrict__ sorted_ids,
                   const int64_t* __restrict__ ids64 = nullptr, uint32_t* __restrict__ claim = nullptr) {
    const int64_t stride = ((int64_t)gridDim.x * blockDim.x) / LPRR;  // rows between two items of one lane
    const int64_t gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int h = (int)(gt % LPRR);
    const int first_col = 4 * CH * h;
    int live = CH;
    if (LPRR > 1) { live = ((t.used + 3) >> 2) - CH * h; live = live > CH ? CH : live; }
    const int upto = __ldg(a.step);
    int64_t kc = gt / LPRR;                                           // index of the current item
    if (kc >= n_items) return;
    ReplayRow<CH> cur, nxt;
    auto row_of = [&](int64_t k) -> int64_t {
        return UNSORTED ? replay_row_unsorted(k, n_items, ids64, t.n_rows) : replay_row_of<CATCHUP>(k, n_items, r0, sorted_ids, t.n_rows);
    };
    replay_row_issue<CH, UNSORTED, P>(cur, row_of(kc), t, a, first_col, live, claim, h == 0);
    replay_row_issue<CH, UNSORTED, P>(nxt, row_of(kc + stride), t, a, first_col, live, claim, h == 0);
    int64_t row2 = row_of(kc + 2 * stride);
    if (cur.off == -2) return;
    replay_row_arm<CH, LPRR, UNSORTED>(cur, a, upto, h);
    while (true) {
        if (cur.t >= upto) {                             // current item finished (or had nothing to do): switch
            if (cur.off >= 0) {
#pragma unroll
                for (int c = 0; c < CH; ++c) {
                    if (c < live) {
                        embed_stamp(cur.p[c], first_col + 4 * c, a, upto);
                        st4(t.data + cur.off + 4 * c, cur.p[c]);
                        st4(a.m + cur.off + 4 * c, cur.m[c]);
                        if (P::TWO) st4(a.v + cur.off + 4 * c, cur.v[c]);
                    }
                }
            }
            kc += stride;
            if (kc >= n_items || nxt.off == -2) break;   // end of the queue, or of the ids this table owns
            cur = nxt;                                   // its loads were issued one whole item ago
            replay_row_issue<CH, UNSORTED, P>(nxt, row2, t, a, first_col, live, claim, h == 0);   // row2's id was fetched one item ago: no dependent wait here
            row2 = row_of(kc + 2 * stride);
            replay_row_arm<CH, LPRR, UNSORTED>(cur, a, upto, h);
            continue;
        }
        ++cur.t;
        const float2 sc = P::coef(a.sched, cur.t);
#pragma unroll
        for (int c = 0; c < CH; ++c) P::l2_step4(cur.p[c], cur.m[c], cur.v[c], sc, a.h);
    }
}
template <bool CATCHUP, class P = AdamStep>
static int launch_replay_rows(const TableView& t, const AdamView& a, int64_t r0, int64_t n_items,
                              const uint32_t* sorted_ids, cudaStream_t st, const int64_t* ids64 = nullptr, uint32_t* claim = nullptr) {
    const int ch = (t.used + 3) >> 2;
    const int lprr = ch > 16 ? 8 : (ch > 8 ? 4 : (ch > 4 ? 2 : 1));   // co-located records (5..32 chunks): 2, 4 or 8 lanes per row
    if (a.stamp_col >> 2 != ch - 1) return RLCTR_EUNSUPPORTED;        // the stamp rides in the last active chunk
    int64_t blocks = (n_items * lprr + 127) / 128;
    static int rgrid_env = -1;
    if (rgrid_env < 0) { const char* e = getenv("RLCTR_REPLAY_GRID"); rgrid_env = e ? atoi(e) : 8; }
    const int cap = RLCTR_SMS * (rgrid_env > 0 ? rgrid_env : 8);
    const int grid = (int)(blocks < cap ? (blocks < 1 ? 1 : blocks) : cap);
    if (CATCHUP && ids64) {                              // batch-order ids + claim bits (the co-located records: 5..8 chunks)
        switch (ch) {
            case 5: case 6: replay_rows_kernel<3, 2, true, true><<<grid, 128, 0, st>>>(t, a, r0, n_items, nullptr, ids64, claim); break;
            case 7: case 8: replay_rows_kernel<4, 2, true, true><<<grid, 128, 0, st>>>(t, a, r0, n_items, nullptr, ids64, claim); break;
            default: return RLCTR_EUNSUPPORTED;
        }
        RLCTR_LAUNCH_CHECK();
        return RLCTR_OK;
    }
    switch (ch) {
        case 1: replay_rows_kernel<1, 1, CATCHUP, false, P><<<grid, 128, 0, st>>>(t, a, r0, n_items, sorted_ids); break;
        case 2: replay_rows_kernel<2, 1, CATCHUP, false, P><<<grid, 128, 0, st>>>(t, a, r0, n_items, sorted_ids); break;
        case 3: replay_rows_kernel<3, 1, CATCHUP, false, P><<<grid, 128, 0, st>>>(t, a, r0, n_items, sorted_ids); break;
        case 4: replay_rows_kernel<4, 1, CATCHUP, false, P><<<grid, 128, 0, st>>>(t, a, r0, n_items, sorted_ids); break;
        case 5: case 6: replay_rows_kernel<3, 2, CATCHUP, false, P><<<grid, 128, 0, st>>>(t, a, r0, n_items, sorted_ids); break;
        case 7: case 8: replay_rows_kernel<4, 2, CATCHUP, false, P><<<grid, 128, 0, st>>>(t, a, r0, n_items, sorted_ids); break;
        case 9: case 10: case 11: case 12: replay_rows_kernel<3, 4, CATCHUP, false, P><<<grid, 128, 0, st>>>(t, a, r0, n_items, sorted_ids); break;
        case 13: case 14: case 15: case 16: replay_rows_kernel<4, 4, CATCHUP, false, P><<<grid, 128, 0, st>>>(t, a, r0, n_items, sorted_ids); break;
        default:
            if (ch > 32) return RLCTR_EUNSUPPORTED;      // wider than four lines
            if (ch <= 24) replay_rows_kernel<3, 8, CATCHUP, false, P><<<grid, 128, 0, st>>>(t, a, r0, n_items, sorted_ids);
            else replay_rows_kernel<4, 8, CATCHUP, false, P><<<grid, 128, 0, st>>>(t, a, r0, n_items, sorted_ids);
            break;
    }
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

// ---- rlctr_rows_lookup: the owner-side pass of the lazy-exact step ---------------------------------------------------------
// One pass over the sorted view replaces "catch-up (read + WRITE every touched record), then gather the rows again by id":
//   * every run head reads its record once (the only random DRAM access of the forward side), replays the L2-only steps the
//     row missed IN REGISTERS (per-lane queues as in replay_rows_kernel: no lane waits for another row's staleness),
//   * leaves (p | m | v), current through *step, in the staging array at its sorted position k -- the update kernel reads that
//     (coalesced) instead of the table record, so nothing is replayed twice and the table is written once per step, and
//   * PUSHES the current row to every sample that asked for it: gathered[src rank][slot] (for a sharded table a posted NVLink
//     write into the requester's buffer: the lookup exchange).  The forward then streams its samples' rows from `gathered`.
struct LookupView {
    float* stage;
    float* gathered[RLCTR_MAX_WORLD];
    int world;
    uint32_t n_per_rank;
    int rs;              // floats per gathered row
};
__device__ __forceinline__ float* gathered_row(const LookupView& lk, uint32_t gslot) {
    if (lk.world <= 1) return lk.gathered[0] + (int64_t)gslot * lk.rs;
    const uint32_t src = gslot / lk.n_per_rank;
    return lk.gathered[src] + (int64_t)(gslot - src * lk.n_per_rank) * lk.rs;
}
// One LANE GROUP (4 lanes, a 16-byte chunk of p, m and v each) owns a queue of sorted positions g, g + G, g + 2G ...: every access
// of a record, a staged row or a gathered row is one coalesced 48 / 64-byte request per group.  The groups of a warp advance
// through their queues independently (a group that finishes a row hands it out and switches to the next one, whose record was
// requested a whole row earlier), so no group waits for another row's staleness and the replay loop runs with all groups busy.
struct LookupItem {
    float4 p, m, v;
    int64_t off;         // float offset of this lane's chunk of the record; -1: nothing at this position; -2: end of the owned ids
    uint32_t id, slot0, next_id, far_id;
};
__device__ __forceinline__ void lookup_issue(LookupItem& it, int64_t row, int64_t k, int64_t n, int col0, bool chunk_on, const TableView& t,
                                             const AdamView& a, const uint32_t* __restrict__ sorted_ids,
                                             const uint32_t* __restrict__ sorted_slots) {
    it.off = row < 0 ? row : row * t.pitch + col0;
    it.p = f4zero(); it.m = f4zero(); it.v = f4zero();
    if (row >= 0) {
        it.id = (uint32_t)row;
        it.slot0 = __ldg(sorted_slots + k);
        it.next_id = (k + 1 < n) ? __ldg(sorted_ids + k + 1) : 0xffffffffu;
        it.far_id = (k + LONG_RUN < n) ? __ldg(sorted_ids + k + LONG_RUN) : 0xffffffffu;
        if (chunk_on) {
            it.p = ld4(t.data + it.off);
            it.m = ld4(a.m + it.off);
            it.v = ld4(a.v + it.off);
        }
    }
}
template <int CH>
__global__ void __launch_bounds__(256, 4)
lookup_rows_kernel(const __grid_constant__ TableView t, const __grid_constant__ AdamView a, const __grid_constant__ LookupView lk, int64_t n,
                   const uint32_t* __restrict__ sorted_ids, const uint32_t* __restrict__ sorted_slots,
                   int32_t* __restrict__ long_count, uint32_t* __restrict__ long_list) {
    constexpr int LPR = 4;
    const int lane = threadIdx.x & 31;
    const int c = lane & (LPR - 1), col0 = 4 * c;
    const bool chunk_on = c < CH;
    const unsigned gmask = 0xfu << (lane & ~(LPR - 1));                 // the four lanes of this group (always converged)
    const int stamp_lane = (lane & ~(LPR - 1)) + (a.stamp_col >= 0 ? (a.stamp_col >> 2) : 0);
    const int64_t stride = ((int64_t)gridDim.x * blockDim.x) / LPR;     // groups in the grid
    const int upto = __ldg(a.step);
    const bool lazy = a.stamp_col >= 0;
    int64_t kc = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / LPR;
    if (kc >= n) return;
    LookupItem cur, nxt;
    lookup_issue(cur, replay_row_of<true>(kc, n, 0, sorted_ids, t.n_rows), kc, n, col0, chunk_on, t, a, sorted_ids, sorted_slots);
    lookup_issue(nxt, replay_row_of<true>(kc + stride, n, 0, sorted_ids, t.n_rows), kc + stride, n, col0, chunk_on, t, a, sorted_ids,
                 sorted_slots);
    int64_t row2 = replay_row_of<true>(kc + 2 * stride, n, 0, sorted_ids, t.n_rows);
    if (cur.off == -2) return;
    int cur_t = upto;
    if (lazy) {
        const int st = __shfl_sync(gmask, __float_as_int(f4get(cur.p, a.stamp_col & 3)), stamp_lane);
        if (cur.off >= 0) cur_t = st;
    }
    while (true) {
        if (cur_t >= upto) {                             // the row is up to date: hand it out, switch to the next one
            if (cur.off >= 0) {
                if (chunk_on) {
                    float* sp = lk.stage + kc * (12 * CH) + col0;
                    st4(sp, cur.p);
                    st4(sp + 4 * CH, cur.m);
                    st4(sp + 8 * CH, cur.v);
                }
                if (lazy && c == (a.stamp_col >> 2)) f4set(cur.p, a.stamp_col & 3, 0.f);      // clean padding column for the samples
                if (cur.far_id == cur.id) {              // heavy-hitter id: its occurrences are served by lookup_long_kernel
                    if (c == 0) long_list[atomicAdd(long_count, 1)] = (uint32_t)kc;
                } else {
                    uint32_t slot = cur.slot0, nid = cur.next_id;
                    int64_t kk = kc;
                    while (true) {
                        if (col0 < lk.rs) st4(gathered_row(lk, slot) + col0, cur.p);          // whole row: padding chunks are zero
                        if (nid != cur.id) break;
                        ++kk;
                        slot = __ldg(sorted_slots + kk);
                        nid = (kk + 1 < n) ? __ldg(sorted_ids + kk + 1) : 0xffffffffu;
                    }
                }
            }
            kc += stride;
            if (kc >= n || nxt.off == -2) break;
            cur = nxt;
            lookup_issue(nxt, row2, kc + stride, n, col0, chunk_on, t, a, sorted_ids, sorted_slots);
            row2 = replay_row_of<true>(kc + 2 * stride, n, 0, sorted_ids, t.n_rows);
            cur_t = upto;
            if (lazy) {
                const int st = __shfl_sync(gmask, __float_as_int(f4get(cur.p, a.stamp_col & 3)), stamp_lane);
                if (cur.off >= 0) cur_t = st;
            }
            continue;
        }
        ++cur_t;
        adam_l2_step4(cur.p, cur.m, cur.v, __ldg(&a.sched[cur_t]), a.h);
    }
}
// block per heavy-hitter run: every occurrence gets the staged (current) row
template <int CH>
__global__ void __launch_bounds__(256)
lookup_long_kernel(const __grid_constant__ LookupView lk, int64_t n, const uint32_t* __restrict__ sorted_ids,
                   const uint32_t* __restrict__ sorted_slots, const int32_t* __restrict__ long_count,
                   const uint32_t* __restrict__ long_list, int stamp_col) {
    __shared__ int64_t s_end;
    __shared__ float4 s_p[CH];
    const int nlong = *long_count;
    for (int li = blockIdx.x; li < nlong; li += gridDim.x) {
        const int64_t k = long_list[li];
        const uint32_t id = __ldg(sorted_ids + k);
        if (threadIdx.x == 0) {
            int64_t lo = k, hi = n;
            while (hi - lo > 1) {
                int64_t mid = (lo + hi) >> 1;
                if (__ldg(sorted_ids + mid) == id) lo = mid; else hi = mid;
            }
            s_end = hi;
        }
        if (threadIdx.x < CH) {
            float4 p = ld4(lk.stage + k * (12 * CH) + 4 * threadIdx.x);
            if (stamp_col >= 0 && (stamp_col >> 2) == (int)threadIdx.x) f4set(p, stamp_col & 3, 0.f);
            s_p[threadIdx.x] = p;
        }
        __syncthreads();
        const int rch = lk.rs >> 2;                          // whole rows (padding chunks zero)
        const int64_t items = (s_end - k) * rch;
        for (int64_t i = threadIdx.x; i < items; i += blockDim.x) {
            const int64_t kk = k + i / rch;
            const int c = (int)(i % rch);
            st4(gathered_row(lk, __ldg(sorted_slots + kk)) + 4 * c, c < CH ? s_p[c] : f4zero());
        }
        __syncthreads();
    }
}
// LR records [w | m | v | stamp]: one lane per sorted position
__global__ void __launch_bounds__(256)
lookup_scalar_kernel(TableView t, AdamView a, const __grid_constant__ LookupView lk, int64_t n, const uint32_t* __restrict__ sorted_ids,
                     const uint32_t* __restrict__ sorted_slots, int32_t* __restrict__ long_count, uint32_t* __restrict__ long_list) {
    const int upto = __ldg(a.step);
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t id = __ldg(sorted_ids + k);
        if (id >= (uint64_t)t.n_rows) return;              // sentinel tail
        if (k > 0 && __ldg(sorted_ids + k - 1) == id) continue;
        const uint32_t slot0 = __ldg(sorted_slots + k);
        const uint32_t next_id = (k + 1 < n) ? __ldg(sorted_ids + k + 1) : 0xffffffffu;
        const uint32_t far_id = (k + LONG_RUN < n) ? __ldg(sorted_ids + k + LONG_RUN) : 0xffffffffu;
        const int64_t o = (int64_t)id * t.pitch;
        float p = t.data[o], m = a.m[o], v = a.v[o];
        if (is_lazy(a)) adam_replay1(p, m, v, load_stamp(t, a, id), upto, a.sched, a.h);
        st4(lk.stage + 4 * k, make_float4(p, m, v, 0.f));
        if (far_id == id) { long_list[atomicAdd(long_count, 1)] = (uint32_t)k; continue; }
        uint32_t slot = slot0, nid = next_id;
        int64_t kk = k;
        while (true) {
            *gathered_row(lk, slot) = p;
            if (nid != id) break;
            ++kk;
            slot = __ldg(sorted_slots + kk);
            nid = (kk + 1 < n) ? __ldg(sorted_ids + kk + 1) : 0xffffffffu;
        }
    }
}
__global__ void __launch_bounds__(256)
lookup_long_scalar_kernel(const __grid_constant__ LookupView lk, int64_t n, const uint32_t* __restrict__ sorted_ids,
                          const uint32_t* __restrict__ sorted_slots, const int32_t* __restrict__ long_count,
                          const uint32_t* __restrict__ long_list) {
    __shared__ int64_t s_end;
    const int nlong = *long_count;
    for (int li = blockIdx.x; li < nlong; li += gridDim.x) {
        const int64_t k = long_list[li];
        const uint32_t id = __ldg(sorted_ids + k);
        if (threadIdx.x == 0) {
            int64_t lo = k, hi = n;
            while (hi - lo > 1) {
                int64_t mid = (lo + hi) >> 1;
                if (__ldg(sorted_ids + mid) == id) lo = mid; else hi = mid;
            }
            s_end = hi;
        }
        __syncthreads();
        const float p = lk.stage[4 * k];
        for (int64_t kk = k + threadIdx.x; kk < s_end; kk += blockDim.x) *gathered_row(lk, __ldg(sorted_slots + kk)) = p;
        __syncthreads();
    }
}

// stamps are written after the replay kernel has completed (the chunks of one row are replayed by
// different threads, each of which reads the row's stamp)
__global__ void __launch_bounds__(256)
catchup_stamp_kernel(const uint32_t* __restrict__ sorted_ids, int64_t n, int64_t n_rows, int32_t* __restrict__ stamp,
                     const int32_t* __restrict__ step) {
    const int upto = __ldg(step);
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t id = __ldg(sorted_ids + k);
        if (id < (uint64_t)n_rows && (k == 0 || __ldg(sorted_ids + k - 1) != id)) stamp[id] = upto;
    }
}
template <class P = AdamStep>
__global__ void __launch_bounds__(256)
adam_flush_scalar_kernel(TableView t, AdamView a, int64_t r0, int64_t r1) {   // row_stride == 1 (LR)
    const int upto = __ldg(a.step);
    for (int64_t row = r0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < r1; row += (int64_t)gridDim.x * blockDim.x) {
        const int st = load_stamp(t, a, row);
        if (st >= upto) continue;
        const int64_t o = row * t.pitch;
        float p = t.data[o], m = a.m[o], v = P::TWO ? a.v[o] : 0.f;
        P::replay1(p, m, v, st, upto, a.sched, a.h);
        t.data[o] = p; a.m[o] = m; if (P::TWO) a.v[o] = v;
        if (a.stamp_col >= 0) t.data[o + a.stamp_col] = __int_as_float(upto); else a.stamp[row] = upto;
    }
}
__global__ void __launch_bounds__(256)
stamp_fill_kernel(int32_t* __restrict__ stamp, const int32_t* __restrict__ step, int64_t r0, int64_t r1) {
    const int upto = __ldg(step);
    for (int64_t row = r0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < r1; row += (int64_t)gridDim.x * blockDim.x)
        stamp[row] = upto;
}

// row_stride == 1 (the LR table): one lane per sorted position
template <int APPLY, class P = AdamStep>
__global__ void __launch_bounds__(256)
rows_scalar_kernel(const uint32_t* __restrict__ sorted_ids, const uint32_t* __restrict__ sorted_slots, int64_t n,
                   GradView g, TableView t, AdamView a, float* __restrict__ dense_grad) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t id = __ldg(sorted_ids + k);
    if (id >= (uint64_t)t.n_rows) return;                 // sentinel tail: nothing for this thread here or further on
    if (k > 0 && __ldg(sorted_ids + k - 1) == id) continue;
    float acc = 0.f;
    int64_t kk = k;
    uint32_t nxt = id;
    while (nxt == id) {                                   // LR runs: sequential, slot order
        const uint32_t slot = __ldg(sorted_slots + kk);
        ++kk;
        nxt = (kk < n) ? __ldg(sorted_ids + kk) : 0xffffffffu;
        const GradSrc q = grad_src(g, slot);
        float gsl = q.staged ? __ldg(q.staged + q.slot) : 0.f;
        if (q.dlogit) gsl += __ldg(q.dlogit + q.slot / (uint32_t)g.fields);
        acc += gsl;
    }
    if (APPLY == 1) { dense_grad[id] = acc; continue; }
    const int step = __ldg(a.step) + 1;
    const int64_t o = (int64_t)id * t.pitch;
    float p, m, v = 0.f;
    if (P::TWO && a.stage) {                               // [w, m, v, 0] of this position, replayed by rlctr_rows_lookup
        const float4 r = ldg4(a.stage + 4 * k);
        p = r.x; m = r.y; v = r.z;
    } else {
        p = t.data[o]; m = a.m[o]; if (P::TWO) v = a.v[o];
    }
    if (is_lazy(a)) {
        if (!a.stage) P::replay1(p, m, v, load_stamp(t, a, id), step - 1, a.sched, a.h);
        if (a.stamp_col >= 0) t.data[o + a.stamp_col] = __int_as_float(step); else a.stamp[id] = step;
    }
    P::apply1(p, m, v, acc, P::coef(a.sched, step), a.h);
    t.data[o] = p; a.m[o] = m; if (P::TWO) a.v[o] = v;
    }
}
template <class P = AdamStep>
__global__ void __launch_bounds__(256)
rows_catchup_scalar_kernel(const uint32_t* __restrict__ sorted_ids, int64_t n, TableView t, AdamView a) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const uint32_t id = __ldg(sorted_ids + k);
    if (id >= (uint64_t)t.n_rows || (k > 0 && __ldg(sorted_ids + k - 1) == id)) return;
    const int upto = __ldg(a.step);
    const int st = load_stamp(t, a, id);
    if (st >= upto) return;
    const int64_t o = (int64_t)id * t.pitch;
    float p = t.data[o], m = a.m[o], v = P::TWO ? a.v[o] : 0.f;
    P::replay1(p, m, v, st, upto, a.sched, a.h);
    t.data[o] = p; a.m[o] = m; if (P::TWO) a.v[o] = v;
    if (a.stamp_col >= 0) t.data[o + a.stamp_col] = __int_as_float(upto); else a.stamp[id] = upto;
}

__global__ void __launch_bounds__(256)
dense_adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                  int64_t n, const float2* __restrict__ sched, const int32_t* __restrict__ step, AdamHyper h) {
    const float2 sc = __ldg(&sched[__ldg(step) + 1]);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float pp = p[i], mm = m[i], vv = v[i];
        adam_elem(pp, mm, vv, g[i], h, sc.x, sc.y);
        p[i] = pp; m[i] = mm; v[i] = vv;
    }
}
__global__ void step_advance_kernel(int32_t* step, int32_t delta) { *step += delta; }
struct StepList { int index[RLCTR_DENSE_MAX]; int count; };
__global__ void steps_advance_kernel(int32_t* steps, const __grid_constant__ StepList list) {
    if ((int)threadIdx.x < list.count) steps[list.index[threadIdx.x]] += 1;
}

// All replicated dense parameters of a model in ONE launch (the reference's foreach Adam; nine launches of a few microseconds
// each for DeepFM otherwise).  Block b belongs to tensor t with first_block[t] <= b < first_block[t+1].
struct DenseGroup {
    float* p[RLCTR_DENSE_MAX];
    const float* g[RLCTR_DENSE_MAX];
    float* m[RLCTR_DENSE_MAX];
    float* v[RLCTR_DENSE_MAX];
    int64_t n[RLCTR_DENSE_MAX];
    int first_block[RLCTR_DENSE_MAX + 1];
    int step_index[RLCTR_DENSE_MAX];     // torch keeps one step counter per parameter: steps[step_index[t]] = completed steps of tensor t
    int count;
};
__global__ void __launch_bounds__(256)
dense_adam_multi_kernel(const __grid_constant__ DenseGroup grp, const float2* __restrict__ sched, const int32_t* __restrict__ steps,
                        AdamHyper h) {
    int t = 0;
    while (t + 1 < grp.count && (int)blockIdx.x >= grp.first_block[t + 1]) ++t;
    const float2 sc = __ldg(&sched[__ldg(steps + grp.step_index[t]) + 1]);
    const int nb = grp.first_block[t + 1] - grp.first_block[t];
    float* __restrict__ p = grp.p[t];
    const float* __restrict__ g = grp.g[t];
    float* __restrict__ m = grp.m[t];
    float* __restrict__ v = grp.v[t];
    for (int64_t i = (int64_t)(blockIdx.x - grp.first_block[t]) * blockDim.x + threadIdx.x; i < grp.n[t]; i += (int64_t)nb * blockDim.x) {
        float pp = p[i], mm = m[i], vv = v[i];
        adam_elem(pp, mm, vv, g[i], h, sc.x, sc.y);
        p[i] = pp; m[i] = mm; v[i] = vv;
    }
}
// torch.optim.Adagrad for the replicated dense parameters (DenseGroup.m = state sums, .v unused), IEEE sqrt and division:
// grad.add(param, alpha=wd); state_sum.addcmul_(grad, grad); param.addcdiv_(grad, state_sum.sqrt().add_(eps), value=-clr)
__global__ void __launch_bounds__(256)
dense_adagrad_multi_kernel(const __grid_constant__ DenseGroup grp, const float* __restrict__ clr_tab, const int32_t* __restrict__ steps,
                           float eps, float wd) {
    int t = 0;
    while (t + 1 < grp.count && (int)blockIdx.x >= grp.first_block[t + 1]) ++t;
    const float clr = __ldg(&clr_tab[__ldg(steps + grp.step_index[t]) + 1]);
    const int nb = grp.first_block[t + 1] - grp.first_block[t];
    float* __restrict__ p = grp.p[t];
    const float* __restrict__ g = grp.g[t];
    float* __restrict__ s = grp.m[t];
    for (int64_t i = (int64_t)(blockIdx.x - grp.first_block[t]) * blockDim.x + threadIdx.x; i < grp.n[t]; i += (int64_t)nb * blockDim.x) {
        float pp = p[i], gg = g[i];
        if (wd != 0.f) gg = __fadd_rn(gg, __fmul_rn(wd, pp));
        const float ss = __fadd_rn(s[i], __fmul_rn(gg, gg));
        const float std = __fadd_rn(__fsqrt_rn(ss), eps);
        p[i] = __fadd_rn(pp, __fdiv_rn(__fmul_rn(-clr, gg), std));
        s[i] = ss;
    }
}

static inline int grid_1d(int64_t threads, int cap_blocks) {
    int64_t blocks = (threads + 255) / 256;
    if (blocks < 1) blocks = 1;
    return (int)(blocks < cap_blocks ? blocks : cap_blocks);
}
static inline int key_bits(int64_t n_rows) {     // bits needed for keys 0..n_rows (sentinel included)
    int b = 1;
    while (b < 32 && ((int64_t)1 << b) <= n_rows) ++b;
    return b;
}
struct RowsWs {
    int32_t* long_count;
    uint32_t* long_list;
};
static inline size_t rows_ws_bytes(int64_t n) { return 16 + sizeof(uint32_t) * (size_t)(n / LONG_RUN + 1); }

// Sharded table: an owner meets ~1/world of the n gathered positions (the rest are sentinels at the end of the sorted view), so
// the grid covers 1.25/world of them + a margin and the kernels stride: any excess (skewed ownership) takes another trip.
static inline unsigned capped_blocks(int64_t full, int world) {
    if (world <= 1) return (unsigned)full;
    int64_t cap = full / world + full / (4 * world) + 2 * RLCTR_SMS;
    return (unsigned)(cap < full ? cap : full);
}

// Persistent grid of the row-update kernels: exactly the resident blocks (148 SMs x 5), each striding the positions -- the
// co-located update takes 245 us against 289 us with one block per 32 positions (30,720 blocks whose slots are only refilled when
// their slowest row is done).  RLCTR_ROWS_GRID = m: m x 740 blocks; 0: one block per group of positions.
static inline int rows_grid_env() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("RLCTR_ROWS_GRID"); v = e ? atoi(e) : 1; }
    return v;
}

// the optimizer structs of the C ABI: the pointers every update needs, and the AdamView the kernels take (see AdamStep / AdagradStep)
static inline bool opt_ok(const rlctr_adam* o) { return o && o->exp_avg && o->exp_avg_sq && o->sched && o->step; }
static inline bool opt_ok(const rlctr_adagrad* o) { return o && o->state_sum && o->clr && o->step; }
static inline AdamView view_of(const rlctr_adagrad* o, const TableView& t) {
    return AdamView{o->state_sum, nullptr, o->stamp_col >= 0 ? nullptr : o->stamp, o->stamp_col >= 0 ? o->stamp_col : -1,
                    reinterpret_cast<const float2*>(o->clr), o->step, AdamHyper{0.f, 0.f, 0.f, (float)o->eps, (float)o->weight_decay},
                    nullptr, stage_pitch_of(t)};
}

template <int APPLY, class P = AdamStep, class O = rlctr_adam>
static int launch_rows(const uint32_t* sorted_ids, const uint32_t* sorted_slots, int64_t n, const rlctr_rowgrad* grad,
                       const rlctr_table* table, const O* opt, float* dense_grad, void* ws, size_t ws_bytes,
                       cudaStream_t st) {
    if (!sorted_ids || !sorted_slots || !grad || !table || !table->data || n < 0) return RLCTR_EINVAL;
    if (APPLY == 0 && !opt_ok(opt)) return RLCTR_EINVAL;
    if (APPLY == 0 && opt->stamp_col >= (table->row_pitch > 0 ? table->row_pitch : table->row_stride)) return RLCTR_EINVAL;
    if (APPLY == 0 && opt->stamp_col >= 0 && table->row_stride > 32) return RLCTR_EUNSUPPORTED;   // wide rows: separate stamps
    if (APPLY == 1 && !dense_grad) return RLCTR_EINVAL;
    if ((grad->dlogit || grad->extra) && grad->fields <= 0) return RLCTR_EINVAL;
    if (n == 0) return RLCTR_OK;
    TableView t = view_of(table);
    AdamView a = APPLY == 0 ? view_of(opt, t) : AdamView{};
    if (grad->world > RLCTR_MAX_WORLD || (grad->world > 1 && grad->n_per_rank == 0)) return RLCTR_EINVAL;
    GradView g = grad_view_of(grad);
    if ((g.flags & RLCTR_STAGED_PARTNER) && (!g.staged || !g.dlogit || g.fields <= 0)) return RLCTR_EINVAL;
    if ((g.flags & RLCTR_DZ_IN_SUMS) && (t.rs <= t.used || !g.sums)) return RLCTR_EINVAL;
    if (t.rs == 1) {
        if (grad->extra || grad->sums) return RLCTR_EUNSUPPORTED;
        rows_scalar_kernel<APPLY, P><<<capped_blocks((n + 255) / 256, grad->world), 256, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a,
                                                                                              dense_grad);
        RLCTR_LAUNCH_CHECK();
        return RLCTR_OK;
    }
    if (t.rs % 4 != 0 || t.rs > 128 * WCH_MAX) return RLCTR_EUNSUPPORTED;
    if (t.rs > 32) {
        if (t.rs <= 256)
            rows_wide_kernel<APPLY, 2, P><<<(unsigned)((n + 7) / 8), 256, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, dense_grad);
        else
            rows_wide_kernel<APPLY, 4, P><<<(unsigned)((n + 7) / 8), 256, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, dense_grad);
        RLCTR_LAUNCH_CHECK();
        return RLCTR_OK;
    }
    if (ws_bytes < rows_ws_bytes(n) || !ws) return RLCTR_EWORKSPACE;
    RowsWs w{reinterpret_cast<int32_t*>(ws), reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(ws) + 16)};
    RLCTR_CUDA(cudaMemsetAsync(w.long_count, 0, sizeof(int32_t), st));
    const int lpr = rlctr_lanes_per_row(t.rs);
    unsigned blocks = capped_blocks((n * lpr + 255) / 256, grad->world);
    if (rows_grid_env() > 0 && blocks > (unsigned)(RLCTR_SMS * 5 * rows_grid_env())) blocks = RLCTR_SMS * 5 * rows_grid_env();
#define LAUNCH_ROWS(L)                                                                                              \
    rows_short_kernel<L, APPLY, false, P><<<blocks, 256, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, dense_grad, \
                                                        w.long_count, w.long_list);                                \
    rows_long_kernel<L, APPLY, false, 256, P><<<RLCTR_SMS, 256, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, dense_grad, \
                                                          w.long_count, w.long_list)
    if (P::TWO && APPLY == 0 && a.stage && a.stamp == nullptr && lpr <= 4) {
        // the lookup's staging array feeds the update: phased kernel (R rows per lane group in flight), then the heavy hitters
        static int r_env = -1;
        if (r_env < 0) { const char* e = getenv("RLCTR_ROWS_R"); r_env = e ? atoi(e) : 0; }
        if (r_env == 0 && lpr == 4) {                    // default: the double-buffered tile pipeline
            const int ch = (t.used + 3) >> 2;
            const int64_t tiles = capped_blocks((n + tile::TT - 1) / tile::TT, grad->world);
            const unsigned tb = (unsigned)(tiles < RLCTR_SMS * 3 ? tiles : RLCTR_SMS * 3);
#define LAUNCH_TILE(C)                                                                                                \
            { const size_t sm = 2 * sizeof(tile::Buf<C>);                                                             \
              RLCTR_CUDA(cudaFuncSetAttribute(rows_staged_tile_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm)); \
              rows_staged_tile_kernel<C><<<tb, 256, sm, st>>>(sorted_ids, sorted_slots, n, g, t, a, w.long_count, w.long_list); }
            switch (ch) {
                case 1: LAUNCH_TILE(1); break;
                case 2: LAUNCH_TILE(2); break;
                case 3: LAUNCH_TILE(3); break;
                default: LAUNCH_TILE(4); break;
            }
#undef LAUNCH_TILE
            RLCTR_LAUNCH_CHECK();
            rows_long_kernel<4, 0><<<RLCTR_SMS, 256, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, dense_grad, w.long_count, w.long_list);
            RLCTR_LAUNCH_CHECK();
            return RLCTR_OK;
        }
        const int R = r_env == 2 ? 2 : 4;
        const int64_t per_block = (256 / lpr) * R;
        int64_t want = (n + per_block - 1) / per_block;
        want = capped_blocks(want, grad->world);
        const int64_t cap = (int64_t)RLCTR_SMS * (R > 2 ? 2 : 3) * 4;     // a few trips per resident block
        const unsigned sblocks = (unsigned)(want < cap ? want : cap);
#define LAUNCH_STAGED(L)                                                                                              \
        if (R == 2) rows_staged_kernel<L, 2><<<sblocks, 256, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, w.long_count, w.long_list); \
        else rows_staged_kernel<L, 4><<<sblocks, 256, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, w.long_count, w.long_list);       \
        rows_long_kernel<L, 0><<<RLCTR_SMS, 256, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, dense_grad, w.long_count, w.long_list)
        switch (lpr) {
            case 1: LAUNCH_STAGED(1); break;
            case 2: LAUNCH_STAGED(2); break;
            default: LAUNCH_STAGED(4); break;
        }
#undef LAUNCH_STAGED
        RLCTR_COUNT_LAUNCH(1);
        RLCTR_LAUNCH_CHECK();
        return RLCTR_OK;
    }
    switch (lpr) {
        case 1: LAUNCH_ROWS(1); break;
        case 2: LAUNCH_ROWS(2); break;
        case 4: LAUNCH_ROWS(4); break;
        default: LAUNCH_ROWS(8); break;
    }
#undef LAUNCH_ROWS
    RLCTR_COUNT_LAUNCH(1);                              // two kernels, one check
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

}  // namespace rlctr

using namespace rlctr;

extern "C" size_t rlctr_sort_ws_bytes(int64_t n, int64_t n_rows) {
    if (n <= 0) return 16;
    size_t temp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, temp, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                    (const uint32_t*)nullptr, (uint32_t*)nullptr, n, 0, key_bits(n_rows));
    size_t arr = ((size_t)n * sizeof(uint32_t) + 255) & ~(size_t)255;
    return 2 * arr + temp + 256;
}

extern "C" int rlctr_sort_ids(const int64_t* ids, int64_t n, int64_t n_rows, uint32_t* sorted_ids,
                              uint32_t* sorted_slots, void* ws, size_t ws_bytes, rlctr_stream_t stream) {
    if (!ids || !sorted_ids || !sorted_slots || !ws || n < 0 || n_rows <= 0) return RLCTR_EINVAL;
    if (n >= ((int64_t)1 << 32) || n_rows >= ((int64_t)1 << 32) - 1) return RLCTR_EUNSUPPORTED;
    if (n == 0) return RLCTR_OK;
    cudaStream_t st = (cudaStream_t)stream;
    size_t arr = ((size_t)n * sizeof(uint32_t) + 255) & ~(size_t)255;
    if (ws_bytes < 2 * arr + 256) return RLCTR_EWORKSPACE;
    uint32_t* keys = reinterpret_cast<uint32_t*>(ws);
    uint32_t* vals = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(ws) + arr);
    void* temp = reinterpret_cast<char*>(ws) + 2 * arr;
    size_t temp_bytes = ws_bytes - 2 * arr;
    sort_prep_kernel<<<grid_1d(n, RLCTR_SMS * 8), 256, 0, st>>>(ids, n, n_rows, keys, vals);
    RLCTR_LAUNCH_CHECK();
    cudaError_t e = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys, sorted_ids, vals, sorted_slots, n, 0,
                                                    key_bits(n_rows), st);
    if (e != cudaSuccess) return (int)e;
    RLCTR_COUNT_LAUNCH(2 + (key_bits(n_rows) + 7) / 8);   // cub onesweep: histogram, scan, one kernel per 8-bit digit
    return RLCTR_OK;
}

extern "C" int rlctr_sort_ids_sharded(const uint32_t* ids_all, int64_t n_all, int32_t world, int32_t rank, int64_t n_rows_global,
                                      uint32_t* sorted_rows, uint32_t* sorted_slots, void* ws, size_t ws_bytes,
                                      rlctr_stream_t stream) {
    if (!ids_all || !sorted_rows || !sorted_slots || !ws || n_all < 0 || n_rows_global <= 0) return RLCTR_EINVAL;
    if (world != 1 && world != 2 && world != 4 && world != 8) return RLCTR_EUNSUPPORTED;
    if (rank < 0 || rank >= world) return RLCTR_EINVAL;
    if (n_all >= ((int64_t)1 << 32) || n_rows_global >= ((int64_t)1 << 32) - 1) return RLCTR_EUNSUPPORTED;
    if (n_all == 0) return RLCTR_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int shift = 0;
    while ((1 << shift) < world) ++shift;
    const int64_t n_local = (n_rows_global - rank + world - 1) / world;         // rows of this rank's shard
    size_t arr = ((size_t)n_all * sizeof(uint32_t) + 255) & ~(size_t)255;
    if (ws_bytes < 2 * arr + 256) return RLCTR_EWORKSPACE;
    uint32_t* keys = reinterpret_cast<uint32_t*>(ws);
    uint32_t* vals = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(ws) + arr);
    void* temp = reinterpret_cast<char*>(ws) + 2 * arr;
    size_t temp_bytes = ws_bytes - 2 * arr;
    sort_prep_sharded_kernel<<<grid_1d(n_all, RLCTR_SMS * 8), 256, 0, st>>>(ids_all, n_all, n_rows_global, shift, (uint32_t)(world - 1),
                                                                             (uint32_t)rank, (uint32_t)n_local, keys, vals);
    RLCTR_LAUNCH_CHECK();
    cudaError_t e = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys, sorted_rows, vals, sorted_slots, n_all, 0,
                                                    key_bits(n_local), st);
    if (e != cudaSuccess) return (int)e;
    RLCTR_COUNT_LAUNCH(2 + (key_bits(n_local) + 7) / 8);
    return RLCTR_OK;
}

extern "C" size_t rlctr_rows_ws_bytes(int64_t n) { return rows_ws_bytes(n < 0 ? 0 : n); }

extern "C" int rlctr_rows_adam(const uint32_t* sorted_ids, const uint32_t* sorted_slots, int64_t n,
                               const rlctr_rowgrad* grad, const rlctr_table* table, const rlctr_adam* opt, void* ws,
                               size_t ws_bytes, rlctr_stream_t stream) {
    return launch_rows<0>(sorted_ids, sorted_slots, n, grad, table, opt, nullptr, ws, ws_bytes, (cudaStream_t)stream);
}

static inline const float* stage_of(const rlctr_adam* o) { return o->stage; }
static inline const float* stage_of(const rlctr_adagrad*) { return nullptr; }
template <class P, class O>
static int group_rows(const uint32_t* sorted_ids, const uint32_t* sorted_slots, int64_t n, const rlctr_table* table, const O* opt,
                      const rlctr_member* members, int32_t n_members, const float* sums, int32_t sums_pitch, int32_t fields,
                      int32_t world, const uint32_t* slot_of, void* ws, size_t ws_bytes, rlctr_stream_t stream) {
    if (!sorted_ids || !sorted_slots || !table || !table->data || !opt_ok(opt) || !members || !sums || n < 0 || fields <= 0)
        return RLCTR_EINVAL;
    if (n_members < 1 || n_members > RLCTR_GROUP_MAX) return RLCTR_EINVAL;
    if (table->world > 1 || stage_of(opt)) return RLCTR_EUNSUPPORTED;
    if (n == 0) return RLCTR_OK;
    cudaStream_t st = (cudaStream_t)stream;
    TableView t = view_of(table);
    AdamView a = view_of(opt, t);
    if (t.rs % 4 != 0 || t.rs <= 8 || t.rs > RLCTR_GROUP_MAX_FLOATS) return RLCTR_EUNSUPPORTED;
    if (opt->stamp_col >= t.pitch) return RLCTR_EINVAL;
    if (!rlctr_aligned16(sums)) return RLCTR_EALIGN;
    if (sums_pitch == 0) sums_pitch = t.rs;
    if (sums_pitch < t.rs || sums_pitch % 4 != 0 || world < 0 || world > RLCTR_MAX_WORLD) return RLCTR_EINVAL;
    GradView g{};
    g.sums = sums; g.fields = fields; g.world = 0;
    g.grp.n = n_members;
    g.grp.sums_pitch = sums_pitch;
    g.grp.slot_of = slot_of;
    for (int col = 0; col < RLCTR_GROUP_MAX_FLOATS; ++col) { g.grp.member[col] = -1; g.grp.role[col] = 0; }
    // one line and every vector member a 16-float stand-alone row: the one-line kernels; anything else: the wide ones
    bool wide = t.rs > 32;
    for (int m = 0; m < n_members; ++m) {
        const rlctr_member& mm = members[m];
        if (mm.dim < 0 || mm.emb_col < 0 || mm.emb_col + mm.dim > t.rs || mm.lin_col >= t.rs) return RLCTR_EINVAL;
        if (mm.extra_pitch != 0 && (mm.extra_pitch < mm.dim || mm.extra_pitch > INT32_MAX)) return RLCTR_EINVAL;
        const bool uses_dz = mm.lin_col >= 0 || ((mm.flags & RLCTR_FM_TERM) && mm.dim > 0);
        if (uses_dz && !mm.dlogit && sums_pitch - RLCTR_GROUP_MAX < t.rs) return RLCTR_EINVAL;   // no room for dL/dlogit in the sums rows
        if (uses_dz) g.grp.dz_used |= 1 << m;
        g.grp.dz[m] = mm.dlogit; g.grp.extra[m] = mm.extra; g.grp.emb_col[m] = mm.emb_col; g.grp.dim[m] = mm.dim;
        g.grp.ex_pitch[m] = mm.extra_pitch ? (int)mm.extra_pitch : mm.dim;
        g.grp.lpr[m] = (signed char)(mm.dim > 0 ? rlctr_member_lpr(mm.lin_col, mm.emb_col, mm.dim) : 4);
        if (g.grp.lpr[m] == 0) return RLCTR_EUNSUPPORTED;                // stand-alone rows of at most 36 floats
        if (g.grp.lpr[m] != 4) wide = true;
        if (mm.lin_col >= 0) {
            if (g.grp.member[mm.lin_col] >= 0) return RLCTR_EINVAL;              // two members claim one column
            g.grp.member[mm.lin_col] = (signed char)m; g.grp.role[mm.lin_col] = 1;
        }
        for (int d = 0; d < mm.dim; ++d) {
            const int col = mm.emb_col + d;
            if (g.grp.member[col] >= 0) return RLCTR_EINVAL;
            g.grp.member[col] = (signed char)m; g.grp.role[col] = (mm.flags & RLCTR_FM_TERM) ? 2 : 3;
        }
    }
    if (opt->stamp_col >= 0 && opt->stamp_col < RLCTR_GROUP_MAX_FLOATS && g.grp.member[opt->stamp_col] >= 0) return RLCTR_EINVAL;
    if (ws_bytes < rows_ws_bytes(n) || !ws) return RLCTR_EWORKSPACE;
    RowsWs w{reinterpret_cast<int32_t*>(ws), reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(ws) + 16)};
    RLCTR_CUDA(cudaMemsetAsync(w.long_count, 0, sizeof(int32_t), st));
    if (wide) {
        // short runs: a lane per chunk walks the occurrences in slot order (the order of every stand-alone form), 16 or 32 lanes per
        // record; long runs: each chunk in its member's stand-alone tree (group_long_wide_kernel)
        const int lanes = t.rs <= 64 ? 16 : 32;
        unsigned blocks = capped_blocks((n * lanes + 255) / 256, world);
        if (rows_grid_env() > 0 && blocks > (unsigned)(RLCTR_SMS * 5 * rows_grid_env())) blocks = RLCTR_SMS * 5 * rows_grid_env();
        if (lanes == 16) rows_short_kernel<16, 0, true, P><<<blocks, 256, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, nullptr, w.long_count, w.long_list);
        else rows_short_kernel<32, 0, true, P><<<blocks, 256, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, nullptr, w.long_count, w.long_list);
        group_long_wide_kernel<P><<<RLCTR_SMS, 256, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, w.long_count, w.long_list);
        RLCTR_COUNT_LAUNCH(1);                          // two kernels, one check
        RLCTR_LAUNCH_CHECK();
        return RLCTR_OK;
    }
    const int lpr = rlctr_lanes_per_row(t.rs);
    // RLCTR_GROUP_ROWS2=0: the eight-lanes-per-record kernel.  Both take ~250 us for 936 K records at B = 65536 (read per call: the
    // tests switch it): 2.5x fewer instructions and 1.7x more records in flight buy nothing, because the update already runs at the
    // memory system's random-access rate -- 3 lines read + 3 written per record + the dense-tail rows = ~27 G line operations/s
    const char* r2e = getenv("RLCTR_GROUP_ROWS2");
    const int rows2_env = r2e ? atoi(r2e) : 1;
    bool one_member_per_chunk = true;                    // group_rows2_kernel keeps ONE dense-tail pointer per 16-byte chunk
    for (int ch = 0; ch < 8; ++ch) {
        int owner = -1;
        for (int q = 0; q < 4; ++q) {
            const int col = 4 * ch + q;
            if (g.grp.role[col] >= 2) {
                if (owner >= 0 && owner != g.grp.member[col]) one_member_per_chunk = false;
                owner = g.grp.member[col];
            }
        }
    }
    if (rows2_env && one_member_per_chunk && !opt->stamp && (t.used + 3) / 4 <= 8 && lpr == 8) {
        // two lanes per record on a persistent grid (2 resident blocks per SM), then the heavy hitters
        int64_t want = capped_blocks((2 * n + 255) / 256, world);
        const int64_t cap = (int64_t)RLCTR_SMS * 2 * (rows_grid_env() > 0 ? rows_grid_env() : 64);
        const unsigned b2 = (unsigned)(want < cap ? want : cap);
        if ((t.used + 3) / 4 <= 6) group_rows2_kernel<3, P><<<b2, 256, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, w.long_count, w.long_list);
        else group_rows2_kernel<4, P><<<b2, 256, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, w.long_count, w.long_list);
        rows_long_kernel<8, 0, true, 512, P><<<RLCTR_SMS, 512, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, nullptr, w.long_count, w.long_list);
        RLCTR_COUNT_LAUNCH(1);
        RLCTR_LAUNCH_CHECK();
        return RLCTR_OK;
    }
    unsigned blocks = capped_blocks((n * lpr + 255) / 256, world);
    if (rows_grid_env() > 0 && blocks > (unsigned)(RLCTR_SMS * 5 * rows_grid_env())) blocks = RLCTR_SMS * 5 * rows_grid_env();
    if (lpr == 4) {
        rows_short_kernel<4, 0, true, P><<<blocks, 256, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, nullptr, w.long_count, w.long_list);
        rows_long_kernel<4, 0, true, 256, P><<<RLCTR_SMS, 256, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, nullptr, w.long_count, w.long_list);
    } else {
        rows_short_kernel<8, 0, true, P><<<blocks, 256, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, nullptr, w.long_count, w.long_list);
        rows_long_kernel<8, 0, true, 512, P><<<RLCTR_SMS, 512, 0, st>>>(sorted_ids, sorted_slots, n, g, t, a, nullptr, w.long_count, w.long_list);
    }
    RLCTR_COUNT_LAUNCH(1);                              // two kernels, one check
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

extern "C" int rlctr_group_rows_adam(const uint32_t* sorted_ids, const uint32_t* sorted_slots, int64_t n, const rlctr_table* table,
                                     const rlctr_adam* opt, const rlctr_member* members, int32_t n_members, const float* sums,
                                     int32_t sums_pitch, int32_t fields, int32_t world, const uint32_t* slot_of, void* ws,
                                     size_t ws_bytes, rlctr_stream_t stream) {
    return group_rows<AdamStep>(sorted_ids, sorted_slots, n, table, opt, members, n_members, sums, sums_pitch, fields, world, slot_of,
                                ws, ws_bytes, stream);
}

extern "C" int rlctr_rows_grad_dense(const uint32_t* sorted_ids, const uint32_t* sorted_slots, int64_t n,
                                     const rlctr_rowgrad* grad, const rlctr_table* table, float* dense_grad, void* ws,
                                     size_t ws_bytes, rlctr_stream_t stream) {
    return launch_rows<1>(sorted_ids, sorted_slots, n, grad, table, (const rlctr_adam*)nullptr, dense_grad, ws, ws_bytes,
                          (cudaStream_t)stream);
}

extern "C" int64_t rlctr_lookup_stage_floats(const rlctr_table* table) {
    if (!table) return 0;
    return stage_pitch_of(view_of(table));
}

extern "C" int rlctr_rows_lookup(const uint32_t* sorted_ids, const uint32_t* sorted_slots, int64_t n, const rlctr_table* table,
                                 const rlctr_adam* opt, const rlctr_lookup* lookup, void* ws, size_t ws_bytes,
                                 rlctr_stream_t stream) {
    if (!sorted_ids || !sorted_slots || !table || !table->data || !opt || !opt->exp_avg || !opt->exp_avg_sq || !opt->sched ||
        !opt->step || !lookup || !lookup->stage || n < 0)
        return RLCTR_EINVAL;
    if (lookup->world > RLCTR_MAX_WORLD || (lookup->world > 1 && lookup->n_per_rank == 0)) return RLCTR_EINVAL;
    if (n == 0) return RLCTR_OK;
    cudaStream_t st = (cudaStream_t)stream;
    TableView t = view_of(table);
    AdamView a = view_of(opt, t);
    LookupView lk{};
    lk.stage = lookup->stage; lk.world = lookup->world; lk.n_per_rank = lookup->n_per_rank; lk.rs = t.rs;
    const int peers = lookup->world > 1 ? lookup->world : 1;
    for (int r = 0; r < peers; ++r) {
        if (!lookup->gathered[r]) return RLCTR_EINVAL;
        lk.gathered[r] = lookup->gathered[r];
    }
    if (ws_bytes < rows_ws_bytes(n) || !ws) return RLCTR_EWORKSPACE;
    RowsWs w{reinterpret_cast<int32_t*>(ws), reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(ws) + 16)};
    RLCTR_CUDA(cudaMemsetAsync(w.long_count, 0, sizeof(int32_t), st));
    if (t.rs == 1) {
        lookup_scalar_kernel<<<capped_blocks((n + 255) / 256, lookup->world), 256, 0, st>>>(t, a, lk, n, sorted_ids, sorted_slots,
                                                                                            w.long_count, w.long_list);
        RLCTR_LAUNCH_CHECK();
        lookup_long_scalar_kernel<<<RLCTR_SMS, 256, 0, st>>>(lk, n, sorted_ids, sorted_slots, w.long_count, w.long_list);
        RLCTR_LAUNCH_CHECK();
        return RLCTR_OK;
    }
    // vector rows: the per-lane replay queues need the stamp inside the record (or no lazy state at all)
    if (t.rs % 4 != 0 || t.rs > 16 || (opt->stamp && opt->stamp_col < 0)) return RLCTR_EUNSUPPORTED;
    if (a.stamp_col >= 0 && (a.stamp_col >> 2) != ((t.used + 3) >> 2) - 1) return RLCTR_EUNSUPPORTED;
    if (!rlctr_aligned16(lookup->stage)) return RLCTR_EALIGN;
    const int ch = (t.used + 3) >> 2;
    int64_t blocks = (n * 4 + 255) / 256;               // one 4-lane group per position, queues of a few rows per group
    blocks = capped_blocks(blocks, lookup->world);
    const int grid = (int)(blocks < RLCTR_SMS * 4 ? (blocks < 1 ? 1 : blocks) : RLCTR_SMS * 4);
#define LAUNCH_LOOKUP(C)                                                                                                     \
    lookup_rows_kernel<C><<<grid, 256, 0, st>>>(t, a, lk, n, sorted_ids, sorted_slots, w.long_count, w.long_list);           \
    lookup_long_kernel<C><<<RLCTR_SMS, 256, 0, st>>>(lk, n, sorted_ids, sorted_slots, w.long_count, w.long_list, a.stamp_col)
    switch (ch) {
        case 1: LAUNCH_LOOKUP(1); break;
        case 2: LAUNCH_LOOKUP(2); break;
        case 3: LAUNCH_LOOKUP(3); break;
        case 4: LAUNCH_LOOKUP(4); break;
        default: return RLCTR_EUNSUPPORTED;
    }
#undef LAUNCH_LOOKUP
    RLCTR_COUNT_LAUNCH(1);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

static inline const void* sched_of(const rlctr_adam* o) { return o->sched; }
static inline const void* sched_of(const rlctr_adagrad* o) { return o->clr; }
template <class P, class O>
static int rows_catchup(const uint32_t* sorted_ids, int64_t n, const rlctr_table* table, const O* opt, rlctr_stream_t stream) {
    if (!sorted_ids || !table || !table->data || !opt || (!opt->stamp && opt->stamp_col < 0) || !sched_of(opt) || !opt->step ||
        n < 0)
        return RLCTR_EINVAL;
    if (n == 0) return RLCTR_OK;
    cudaStream_t st = (cudaStream_t)stream;
    TableView t = view_of(table);
    AdamView a = view_of(opt, t);
    if (t.rs == 1) {
        rows_catchup_scalar_kernel<P><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(sorted_ids, n, t, a);
        RLCTR_LAUNCH_CHECK();
        return RLCTR_OK;
    }
    if (t.rs % 4 != 0) return RLCTR_EUNSUPPORTED;
    if (a.stamp_col >= 0) return launch_replay_rows<true, P>(t, a, 0, n, sorted_ids, st);
    replay_kernel<true, P><<<grid_1d(n * ((t.used + 3) / 4), RLCTR_SMS * 8), 256, 0, st>>>(t, a, 0, n, sorted_ids);
    RLCTR_LAUNCH_CHECK();
    catchup_stamp_kernel<<<grid_1d(n, RLCTR_SMS * 8), 256, 0, st>>>(sorted_ids, n, t.n_rows, a.stamp, a.step);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}
extern "C" int rlctr_rows_catchup(const uint32_t* sorted_ids, int64_t n, const rlctr_table* table,
                                  const rlctr_adam* opt, rlctr_stream_t stream) {
    return rows_catchup<AdamStep>(sorted_ids, n, table, opt, stream);
}

extern "C" size_t rlctr_rows_claim_bytes(int64_t n_rows) {
    return n_rows > 0 ? (size_t)((n_rows + 31) / 32) * sizeof(uint32_t) : 0;
}
extern "C" int rlctr_rows_catchup_ids(const int64_t* ids, int64_t n, const rlctr_table* table, const rlctr_adam* opt, void* claim,
                                      size_t claim_bytes, rlctr_stream_t stream) {
    if (!ids || !table || !table->data || !opt || !opt->sched || !opt->step || n < 0) return RLCTR_EINVAL;
    if (opt->stamp_col < 0) return RLCTR_EUNSUPPORTED;                // in-record stamps only (the joint records)
    if (n == 0) return RLCTR_OK;
    if (!claim || claim_bytes < rlctr_rows_claim_bytes(table->n_rows)) return RLCTR_EWORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    TableView t = view_of(table);
    AdamView a = view_of(opt, t);
    if (t.rs % 4 != 0 || ((t.used + 3) >> 2) < 5 || ((t.used + 3) >> 2) > 8) return RLCTR_EUNSUPPORTED;   // records of 5..8 chunks
    RLCTR_CUDA(cudaMemsetAsync(claim, 0, rlctr_rows_claim_bytes(table->n_rows), st));
    return launch_replay_rows<true>(t, a, 0, n, nullptr, st, ids, reinterpret_cast<uint32_t*>(claim));
}

template <class P, class O>
static int rows_flush(const rlctr_table* table, const O* opt, int64_t row_begin, int64_t row_end, rlctr_stream_t stream) {
    if (!table || !table->data || !opt || (!opt->stamp && opt->stamp_col < 0) || !sched_of(opt) || !opt->step) return RLCTR_EINVAL;
    if (row_begin < 0 || row_end > table->n_rows || row_begin > row_end) return RLCTR_EINVAL;
    if (row_begin == row_end) return RLCTR_OK;
    cudaStream_t st = (cudaStream_t)stream;
    TableView t = view_of(table);
    AdamView a = view_of(opt, t);
    if (t.rs == 1) {
        adam_flush_scalar_kernel<P><<<grid_1d(row_end - row_begin, RLCTR_SMS * 8), 256, 0, st>>>(t, a, row_begin, row_end);
        RLCTR_LAUNCH_CHECK();
        return RLCTR_OK;
    }
    if (t.rs % 4 != 0) return RLCTR_EUNSUPPORTED;
    if (a.stamp_col >= 0) return launch_replay_rows<false, P>(t, a, row_begin, row_end - row_begin, nullptr, st);
    replay_kernel<false, P><<<grid_1d((row_end - row_begin) * ((t.used + 3) / 4), RLCTR_SMS * 8), 256, 0, st>>>(
        t, a, row_begin, row_end - row_begin, nullptr);
    RLCTR_LAUNCH_CHECK();
    stamp_fill_kernel<<<grid_1d(row_end - row_begin, RLCTR_SMS * 8), 256, 0, st>>>(a.stamp, a.step, row_begin, row_end);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}
extern "C" int rlctr_adam_flush(const rlctr_table* table, const rlctr_adam* opt, int64_t row_begin, int64_t row_end,
                                rlctr_stream_t stream) {
    return rows_flush<AdamStep>(table, opt, row_begin, row_end, stream);
}

extern "C" int rlctr_dense_adam(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                                const float* sched, const int32_t* step, double beta1, double beta2, double eps,
                                double weight_decay, rlctr_stream_t stream) {
    if (!param || !grad || !exp_avg || !exp_avg_sq || !sched || !step || n < 0) return RLCTR_EINVAL;
    if (n == 0) return RLCTR_OK;
    dense_adam_kernel<<<grid_1d(n, RLCTR_SMS * 8), 256, 0, (cudaStream_t)stream>>>(
        param, grad, exp_avg, exp_avg_sq, n, reinterpret_cast<const float2*>(sched), step,
        adam_hyper(beta1, beta2, eps, weight_decay));
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

extern "C" int rlctr_dense_adam_multi(float* const* params, const float* const* grads, float* const* exp_avgs,
                                      float* const* exp_avg_sqs, const int64_t* sizes, int32_t count, const float* sched,
                                      const int32_t* steps, const int32_t* step_index, double beta1, double beta2, double eps,
                                      double weight_decay, rlctr_stream_t stream) {
    if (!params || !grads || !exp_avgs || !exp_avg_sqs || !sizes || !sched || !steps || count < 0) return RLCTR_EINVAL;
    if (count > RLCTR_DENSE_MAX) return RLCTR_EUNSUPPORTED;
    if (count == 0) return RLCTR_OK;
    DenseGroup grp;
    grp.count = count;
    int blocks = 0;
    for (int t = 0; t < count; ++t) {
        if (!params[t] || !grads[t] || !exp_avgs[t] || !exp_avg_sqs[t] || sizes[t] < 0) return RLCTR_EINVAL;
        grp.p[t] = params[t]; grp.g[t] = grads[t]; grp.m[t] = exp_avgs[t]; grp.v[t] = exp_avg_sqs[t]; grp.n[t] = sizes[t];
        grp.step_index[t] = step_index ? step_index[t] : 0;
        if (grp.step_index[t] < 0) return RLCTR_EINVAL;
        grp.first_block[t] = blocks;
        blocks += grid_1d(sizes[t], RLCTR_SMS * 2);
    }
    grp.first_block[count] = blocks;
    dense_adam_multi_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(grp, reinterpret_cast<const float2*>(sched), steps,
                                                                     adam_hyper(beta1, beta2, eps, weight_decay));
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

extern "C" int rlctr_steps_advance(int32_t* steps, const int32_t* step_index, int32_t count, rlctr_stream_t stream) {
    if (!steps || !step_index || count < 0) return RLCTR_EINVAL;
    if (count > RLCTR_DENSE_MAX) return RLCTR_EUNSUPPORTED;
    if (count == 0) return RLCTR_OK;
    StepList list;
    list.count = count;
    for (int t = 0; t < count; ++t) {
        if (step_index[t] < 0) return RLCTR_EINVAL;
        list.index[t] = step_index[t];
    }
    steps_advance_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(steps, list);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

extern "C" int rlctr_step_advance(int32_t* step, int32_t delta, rlctr_stream_t stream) {
    if (!step) return RLCTR_EINVAL;
    step_advance_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(step, delta);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

// ---- torch.optim.Adagrad (include/rlctr.h): the Adam calls' gradient side and launch shapes with AdagradStep ------------------
extern "C" int rlctr_rows_adagrad(const uint32_t* sorted_ids, const uint32_t* sorted_slots, int64_t n, const rlctr_rowgrad* grad,
                                  const rlctr_table* table, const rlctr_adagrad* opt, void* ws, size_t ws_bytes,
                                  rlctr_stream_t stream) {
    return launch_rows<0, AdagradStep>(sorted_ids, sorted_slots, n, grad, table, opt, nullptr, ws, ws_bytes, (cudaStream_t)stream);
}

extern "C" int rlctr_group_rows_adagrad(const uint32_t* sorted_ids, const uint32_t* sorted_slots, int64_t n, const rlctr_table* table,
                                        const rlctr_adagrad* opt, const rlctr_member* members, int32_t n_members, const float* sums,
                                        int32_t sums_pitch, int32_t fields, int32_t world, const uint32_t* slot_of, void* ws,
                                        size_t ws_bytes, rlctr_stream_t stream) {
    return group_rows<AdagradStep>(sorted_ids, sorted_slots, n, table, opt, members, n_members, sums, sums_pitch, fields, world,
                                   slot_of, ws, ws_bytes, stream);
}

extern "C" int rlctr_adagrad_catchup(const uint32_t* sorted_ids, int64_t n, const rlctr_table* table, const rlctr_adagrad* opt,
                                     rlctr_stream_t stream) {
    return rows_catchup<AdagradStep>(sorted_ids, n, table, opt, stream);
}

extern "C" int rlctr_adagrad_flush(const rlctr_table* table, const rlctr_adagrad* opt, int64_t row_begin, int64_t row_end,
                                   rlctr_stream_t stream) {
    return rows_flush<AdagradStep>(table, opt, row_begin, row_end, stream);
}

extern "C" int rlctr_dense_adagrad_multi(float* const* params, const float* const* grads, float* const* state_sums,
                                         const int64_t* sizes, int32_t count, const float* clr, const int32_t* steps,
                                         const int32_t* step_index, double eps, double weight_decay, rlctr_stream_t stream) {
    if (!params || !grads || !state_sums || !sizes || !clr || !steps || count < 0) return RLCTR_EINVAL;
    if (count > RLCTR_DENSE_MAX) return RLCTR_EUNSUPPORTED;
    if (count == 0) return RLCTR_OK;
    DenseGroup grp;
    grp.count = count;
    int blocks = 0;
    for (int t = 0; t < count; ++t) {
        if (!params[t] || !grads[t] || !state_sums[t] || sizes[t] < 0) return RLCTR_EINVAL;
        grp.p[t] = params[t]; grp.g[t] = grads[t]; grp.m[t] = state_sums[t]; grp.v[t] = nullptr; grp.n[t] = sizes[t];
        grp.step_index[t] = step_index ? step_index[t] : 0;
        if (grp.step_index[t] < 0) return RLCTR_EINVAL;
        grp.first_block[t] = blocks;
        blocks += grid_1d(sizes[t], RLCTR_SMS * 2);
    }
    grp.first_block[count] = blocks;
    dense_adagrad_multi_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(grp, clr, steps, (float)eps, (float)weight_decay);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}
