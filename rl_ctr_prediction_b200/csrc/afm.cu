// afm.cu -- the AFM attention tail (p_model.py:438-485) over already-gathered rows, forward and backward.
//
//     ip_p   = v_i (.) v_j                         p = (i < j), the reference's row/col order (:452-455)
//     a_p    = relu(W_a ip_p + b_a)                attention_net  (:474)
//     s_p    = <w_s, a_p> + b_s                    attention_softmax (:475)
//     score  = softmax_p(s)                        over the P pairs of one sample
//     sd_p   = score_p * m1_p                      F.dropout(p=0.2) -- ALWAYS on, also in eval() (:477; SURVEY N6)
//     attn_d = sum_p sd_p * ip_p[d]                (:478)
//     y      = <fc_w, attn (.) m2> + fc_b          second F.dropout (:479), fc (:481)
//
// The reference materialises [B, P, D] temporaries for ip, a and the products (4.2 KB per sample each, six of them with
// autograd's copies); here a warp owns a sample, keeps the 15 rows in shared memory and each lane walks its pairs with
// ip / a in registers, so nothing but the rows is read and one float per sample is written.  The backward recomputes the
// forward (no saved activations) and regenerates the dropout masks from the (seed, counter) snapshot of the forward.
// Parameter gradients are accumulated in registers over the whole grid-stride loop (the D x D attention weight distributed by
// entry over the lanes, the small vectors per lane and summed over the warp once at the end) and written as per-warp partials;
// a fixed-order pass reduces them, so results are bit-identical run to run.
//
// params / dparams (packed, NP = D*D + 3*D + 2 floats):  [W_a (D x D, row k = output k) | b_a | w_s | b_s | fc_w | fc_b]
// masks (optional, tests): float [batch, P + D] multipliers (0 or 1/(1-p)) used instead of the hash -- mask-as-input parity.
#include <math.h>
#include "common.cuh"

namespace rlctr {

constexpr int AFM_WARPS = 4;

__device__ __forceinline__ float afm_warp_sum(float x) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) x += __shfl_xor_sync(RLCTR_FULL, x, off);
    return x;
}
__device__ __forceinline__ float afm_warp_max(float x) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) x = fmaxf(x, __shfl_xor_sync(RLCTR_FULL, x, off));
    return x;
}

struct AfmDrop {
    const float* masks;          // [batch, npair + D] or nullptr
    const uint64_t* rng;         // (seed, counter) in device memory or nullptr
    uint32_t thresh;
    float scale;                 // 1 / (1 - p)
};
__device__ __forceinline__ float afm_mask(const AfmDrop& dr, uint64_t seed, uint64_t ctr, int64_t b, int width, int col) {
    if (dr.masks) return __ldg(dr.masks + b * width + col);
    if (!dr.rng) return 1.f;
    return dropout_keep(seed, ctr + (uint64_t)(b * width + col), dr.thresh) ? dr.scale : 0.f;
}

template <int D>
struct AfmSmem {
    static constexpr int DP = (D + 3) / 4 * 4;
    static constexpr int PAR = D * DP + 3 * DP + 4;     // Wa rows padded to DP | ba | ws | fcw | (bs, fcb, -, -)
    static __device__ __forceinline__ void load(float* par, const float* __restrict__ params) {
        for (int i = threadIdx.x; i < PAR; i += blockDim.x) par[i] = 0.f;
        __syncthreads();
        for (int i = threadIdx.x; i < D * D; i += blockDim.x) par[(i / D) * DP + (i % D)] = __ldg(params + i);
        for (int i = threadIdx.x; i < D; i += blockDim.x) {
            par[D * DP + i] = __ldg(params + D * D + i);                      // b_a
            par[D * DP + DP + i] = __ldg(params + D * D + D + i);             // w_s
            par[D * DP + 2 * DP + i] = __ldg(params + D * D + 2 * D + 1 + i); // fc_w
        }
        if (threadIdx.x == 0) {
            par[D * DP + 3 * DP] = __ldg(params + D * D + 2 * D);             // b_s
            par[D * DP + 3 * DP + 1] = __ldg(params + D * D + 3 * D + 1);     // fc_b
        }
    }
};

// scores of one sample: sc[p] <- exp(s_p - max), returns sum_p exp(s_p - max).  stage = the sample's rows in smem.
template <int D>
__device__ __forceinline__ float afm_scores(const float* __restrict__ stage, const float* __restrict__ par,
                                            const unsigned char* __restrict__ pi, const unsigned char* __restrict__ pj,
                                            float* __restrict__ sc, int npair, int lane) {
    constexpr int DP = AfmSmem<D>::DP;
    const float* ba = par + D * DP;
    const float* ws = ba + DP;
    const float bs = par[D * DP + 3 * DP];
    float mx = -INFINITY;
    for (int p = lane; p < npair; p += 32) {
        const float* vi = stage + pi[p] * D;
        const float* vj = stage + pj[p] * D;
        float ip[D];
#pragma unroll
        for (int d = 0; d < D; ++d) ip[d] = vi[d] * vj[d];
        float s = bs;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            float a = ba[k];
#pragma unroll
            for (int d = 0; d < D; ++d) a = fmaf(par[k * DP + d], ip[d], a);
            s = fmaf(ws[k], fmaxf(a, 0.f), s);
        }
        sc[p] = s;
        mx = fmaxf(mx, s);
    }
    mx = afm_warp_max(mx);
    float sum = 0.f;
    for (int p = lane; p < npair; p += 32) {
        const float e = expf(sc[p] - mx);
        sc[p] = e;
        sum += e;
    }
    return afm_warp_sum(sum);
}

__device__ __forceinline__ void afm_pair_tables(unsigned char* pi, unsigned char* pj, unsigned char* pidx, int fields) {
    for (int i = threadIdx.x; i < fields; i += blockDim.x) {
        const int base = i * fields - i * (i + 1) / 2;
        for (int j = i + 1; j < fields; ++j) {
            const int p = base + j - i - 1;
            pi[p] = (unsigned char)i; pj[p] = (unsigned char)j;
            if (pidx) { pidx[i * fields + j] = (unsigned char)p; pidx[j * fields + i] = (unsigned char)p; }
        }
    }
}

// dynamic smem: PAR floats | AFM_WARPS * (fd + npair_pad) floats | 2 * npair bytes
template <int D>
__global__ void __launch_bounds__(AFM_WARPS * 32)
afm_fwd_kernel(const float* __restrict__ rows, int64_t ld_rows, const float* __restrict__ params, AfmDrop dr,
               float* __restrict__ out, int64_t batch, int fields) {
    extern __shared__ __align__(16) float smem[];
    constexpr int DP = AfmSmem<D>::DP;
    constexpr int PAR = AfmSmem<D>::PAR;
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int fd = fields * D, npair = fields * (fields - 1) / 2, npp = (npair + 3) / 4 * 4;
    float* par = smem;
    float* stage = smem + PAR + wib * (fd + npp);
    float* sc = stage + fd;
    unsigned char* pi = reinterpret_cast<unsigned char*>(smem + PAR + AFM_WARPS * (fd + npp));
    unsigned char* pj = pi + npair;
    AfmSmem<D>::load(par, params);
    for (int i = threadIdx.x; i < fields; i += blockDim.x) {
        const int base = i * fields - i * (i + 1) / 2;
        for (int j = i + 1; j < fields; ++j) { pi[base + j - i - 1] = (unsigned char)i; pj[base + j - i - 1] = (unsigned char)j; }
    }
    __syncthreads();
    uint64_t seed = 0, ctr = 0;
    if (dr.rng && !dr.masks) { seed = dr.rng[0]; ctr = dr.rng[1]; }
    const float* fcw = par + D * DP + 2 * DP;
    const float fcb = par[D * DP + 3 * DP + 1];
    const int width = npair + D;
    for (int64_t b = (int64_t)blockIdx.x * AFM_WARPS + wib; b < batch; b += (int64_t)gridDim.x * AFM_WARPS) {
        const float* r = rows + b * ld_rows;
        for (int i = lane; i < fd; i += 32) stage[i] = __ldg(r + i);
        __syncwarp();
        const float sum = afm_scores<D>(stage, par, pi, pj, sc, npair, lane);
        float acc[D];
#pragma unroll
        for (int d = 0; d < D; ++d) acc[d] = 0.f;
        for (int p = lane; p < npair; p += 32) {
            const float sd = sc[p] / sum * afm_mask(dr, seed, ctr, b, width, p);
            const float* vi = stage + pi[p] * D;
            const float* vj = stage + pj[p] * D;
#pragma unroll
            for (int d = 0; d < D; ++d) acc[d] = fmaf(sd, vi[d] * vj[d], acc[d]);
        }
        float y = fcb;
#pragma unroll
        for (int d = 0; d < D; ++d) {
            const float o = afm_warp_sum(acc[d]) * afm_mask(dr, seed, ctr, b, width, npair + d);
            y = fmaf(fcw[d], o, y);
        }
        if (lane == 0) out[b] = y;
        __syncwarp();
    }
}

// dynamic smem: PAR | AFM_WARPS * (fd + 2 * npair_pad + 3 * npair * DP) floats | 2 * npair + fields * fields bytes
//
// Parameter gradients: the D x D gradient of the attention weight is an outer-product sum over pairs,
// dW_a[k][d] = sum_p da_p[k] * ip_p[d].  Accumulating it per lane over the lane's own pairs needs D*D registers per lane (the
// first version: 255 registers, two warps per scheduler, latency-bound at ~6x its issue-rate estimate).  Instead every pair's
// da_p and ip_p are staged in shared memory and the D*D entries are DISTRIBUTED over the lanes: lane l owns entries l, l+32, ...
// (at most ENT = ceil(D*D/32)) and sums over all pairs of the sample.  The small vectors (db_a, dw_s, db_s, dfc) stay per lane.
template <int D>
__global__ void __launch_bounds__(AFM_WARPS * 32, 3)          // <= 168 registers: keeps the compiler from parking all of W_a in registers
afm_bwd_kernel(const float* __restrict__ rows, int64_t ld_rows, const float* __restrict__ params, AfmDrop dr,
               const float* __restrict__ gout, float* __restrict__ grows, int64_t ld_grows, float* __restrict__ part,
               int64_t batch, int fields) {
    extern __shared__ __align__(16) float smem[];
    constexpr int DP = AfmSmem<D>::DP;
    constexpr int PAR = AfmSmem<D>::PAR;
    constexpr int NP = D * D + 3 * D + 2;
    constexpr int CHK = DP / 4;                         // float4 chunks of a (padded) row of D values
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int fd = fields * D, npair = fields * (fields - 1) / 2, npp = (npair + 3) / 4 * 4;
    const int fdp = (fd + 3) & ~3;                  // every per-warp array starts on a 16-byte boundary
    const int per_warp = fdp + 2 * npp + 3 * npair * DP;
    float* par = smem;
    float* stage = smem + PAR + wib * per_warp;
    float* sc = stage + fdp;                // exp(s_p - max)
    float* dsc = sc + npp;                  // d L / d score_p
    float* dipS = dsc + npp;                // d L / d ip_p   [npair, DP]   (rows padded to DP floats: 128-bit accesses)
    float* daS = dipS + npair * DP;         // d L / d (pre-ReLU attention activation) [npair, DP]
    float* ipS = daS + npair * DP;          // ip_p           [npair, DP]
    unsigned char* pi = reinterpret_cast<unsigned char*>(smem + PAR + AFM_WARPS * per_warp);
    unsigned char* pj = pi + npair;
    unsigned char* pidx = pj + npair;
    static_assert(PAR % 4 == 0, "the per-warp arrays follow the parameters at a 16-byte boundary");
    static_assert(D * CHK <= 32, "one dW_a chunk per lane: D <= 10 (afm_bwd_wide_kernel serves larger D)");
    AfmSmem<D>::load(par, params);
    afm_pair_tables(pi, pj, pidx, fields);
    __syncthreads();
    uint64_t seed = 0, ctr = 0;
    if (dr.rng && !dr.masks) { seed = dr.rng[0]; ctr = dr.rng[1]; }
    const float* ba = par + D * DP;
    const float* ws = ba + DP;
    const float* fcw = ws + DP;
    const int width = npair + D;

    // dW_a: lane l < D * CHK owns row k = l / CHK, columns 4 (l % CHK) .. +3 -- one scalar (da_p[k]) and one 128-bit (ip_p chunk)
    // shared-memory read per pair instead of two scalar reads per ENTRY (the first layout: entries l, l + 32, ...)
    float dba[D], dws[D], dfcw[D], dbs = 0.f, dfcb = 0.f;
    float4 dWa4 = f4zero();
    const bool wa_on = lane < D * CHK;
    const int wk = wa_on ? lane / CHK : 0, wc = wa_on ? lane % CHK : 0;
#pragma unroll
    for (int k = 0; k < D; ++k) { dba[k] = 0.f; dws[k] = 0.f; dfcw[k] = 0.f; }

    for (int64_t b = (int64_t)blockIdx.x * AFM_WARPS + wib; b < batch; b += (int64_t)gridDim.x * AFM_WARPS) {
        const float* r = rows + b * ld_rows;
        for (int i = lane; i < fd; i += 32) stage[i] = __ldg(r + i);
        __syncwarp();
        const float sum = afm_scores<D>(stage, par, pi, pj, sc, npair, lane);
        // attention output (needed for d fc_w) -- as in the forward; ip_p is staged for the later passes
        float acc[D];
#pragma unroll
        for (int d = 0; d < D; ++d) acc[d] = 0.f;
        for (int p = lane; p < npair; p += 32) {
            const float sd = sc[p] / sum * afm_mask(dr, seed, ctr, b, width, p);
            const float* vi = stage + pi[p] * D;
            const float* vj = stage + pj[p] * D;
#pragma unroll
            for (int d = 0; d < D; ++d) {
                const float ipd = vi[d] * vj[d];
                ipS[p * DP + d] = ipd;
                acc[d] = fmaf(sd, ipd, acc[d]);
            }
        }
        const float g = __ldg(gout + b);
        float dattn[D];
#pragma unroll
        for (int d = 0; d < D; ++d) {
            const float m2 = afm_mask(dr, seed, ctr, b, width, npair + d);
            const float o = afm_warp_sum(acc[d]) * m2;
            dfcw[d] = fmaf(g, o, dfcw[d]);             // identical in every lane: lane 0's copy is the one written
            dattn[d] = g * fcw[d] * m2;
        }
        dfcb += g;
        // d score_p and the softmax's inner product
        float dot = 0.f;
        for (int p = lane; p < npair; p += 32) {
            float t = 0.f;
#pragma unroll
            for (int d = 0; d < D; ++d) t = fmaf(dattn[d], ipS[p * DP + d], t);
            t *= afm_mask(dr, seed, ctr, b, width, p);
            dsc[p] = t;
            dot = fmaf(sc[p] / sum, t, dot);
        }
        dot = afm_warp_sum(dot);
        for (int p = lane; p < npair; p += 32) {
            const float score = sc[p] / sum;
            const float dsp = score * (dsc[p] - dot);                      // d L / d s_p
            const float sd = score * afm_mask(dr, seed, ctr, b, width, p);
            float ip[D], dip[D];
#pragma unroll
            for (int d = 0; d < D; ++d) { ip[d] = ipS[p * DP + d]; dip[d] = sd * dattn[d]; }
            dbs += dsp;
#pragma unroll
            for (int k = 0; k < D; ++k) {
                float a = ba[k];
#pragma unroll
                for (int d = 0; d < D; ++d) a = fmaf(par[k * DP + d], ip[d], a);
                const float da = a > 0.f ? dsp * ws[k] : 0.f;
                dws[k] = fmaf(dsp, fmaxf(a, 0.f), dws[k]);
                dba[k] += da;
                daS[p * DP + k] = da;
#pragma unroll
                for (int d = 0; d < D; ++d) dip[d] = fmaf(par[k * DP + d], da, dip[d]);
            }
#pragma unroll
            for (int d = 0; d < D; ++d) dipS[p * DP + d] = dip[d];
        }
        __syncwarp();
        // dW_a chunk of this lane: sum over the pairs of the sample, in pair order (two chains: even / odd pairs)
        if (wa_on) {
            float4 a0 = f4zero(), a1 = f4zero();
            int p = 0;
            for (; p + 1 < npair; p += 2) {
                const float d0 = daS[p * DP + wk], d1 = daS[(p + 1) * DP + wk];
                const float4 i0 = *reinterpret_cast<const float4*>(ipS + p * DP + 4 * wc);
                const float4 i1 = *reinterpret_cast<const float4*>(ipS + (p + 1) * DP + 4 * wc);
                a0.x = fmaf(d0, i0.x, a0.x); a0.y = fmaf(d0, i0.y, a0.y); a0.z = fmaf(d0, i0.z, a0.z); a0.w = fmaf(d0, i0.w, a0.w);
                a1.x = fmaf(d1, i1.x, a1.x); a1.y = fmaf(d1, i1.y, a1.y); a1.z = fmaf(d1, i1.z, a1.z); a1.w = fmaf(d1, i1.w, a1.w);
            }
            if (p < npair) {
                const float d0 = daS[p * DP + wk];
                const float4 i0 = *reinterpret_cast<const float4*>(ipS + p * DP + 4 * wc);
                a0.x = fmaf(d0, i0.x, a0.x); a0.y = fmaf(d0, i0.y, a0.y); a0.z = fmaf(d0, i0.z, a0.z); a0.w = fmaf(d0, i0.w, a0.w);
            }
            dWa4.x += a0.x + a1.x; dWa4.y += a0.y + a1.y; dWa4.z += a0.z + a1.z; dWa4.w += a0.w + a1.w;
        }
        // d v_i[d] = sum_{j != i} d ip_{pair(i,j)}[d] * v_j[d], j in order
        for (int t = lane; t < fd; t += 32) {
            const int i = t / D, d = t - i * D;
            const unsigned char* prow = pidx + i * fields;
            float a0 = 0.f, a1 = 0.f;                                      // two chains: the loop is a string of dependent LDS -> FMA
            int j = 0;
            for (; j + 1 < fields; j += 2) {
                if (j != i) a0 = fmaf(dipS[prow[j] * DP + d], stage[j * D + d], a0);
                if (j + 1 != i) a1 = fmaf(dipS[prow[j + 1] * DP + d], stage[(j + 1) * D + d], a1);
            }
            if (j < fields && j != i) a0 = fmaf(dipS[prow[j] * DP + d], stage[j * D + d], a0);
            grows[b * ld_grows + t] = a0 + a1;
        }
        __syncwarp();
    }
    // per-warp partials, one row of NP floats per warp of the grid: dW_a entries are already whole-warp sums of their lane
    float* mine = part + ((int64_t)blockIdx.x * AFM_WARPS + wib) * NP;
    if (wa_on) {
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (4 * wc + q < D) mine[wk * D + 4 * wc + q] = f4get(dWa4, q);
    }
#pragma unroll
    for (int k = 0; k < D; ++k) {
        const float sb = afm_warp_sum(dba[k]);
        const float sw = afm_warp_sum(dws[k]);
        if (lane == 0) {
            mine[D * D + k] = sb;
            mine[D * D + D + k] = sw;
            mine[D * D + 2 * D + 1 + k] = dfcw[k];
        }
    }
    const float sbs = afm_warp_sum(dbs);
    if (lane == 0) { mine[D * D + 2 * D] = sbs; mine[D * D + 3 * D + 1] = dfcb; }
}

// D = 11..32.  The per-lane layout above keeps ip_p, the attention output and its gradient as D floats per lane and lets the
// compiler keep W_a in registers; past D = 10 that spills.  Here every pass that touches the D x D attention weight is turned
// around: a lane OWNS one output unit k (one input dimension d) and walks all pairs of the sample, reading v_i, v_j, d a_p ... as
// shared-memory broadcasts.  A lane keeps three D-float vectors (row k and column d of W_a, its row of d W_a) and nothing else
// of size D:
//     scores  (lane = k):     a_p[k] = b_a[k] + <W_a[k, :], ip_p>   staged [P, AP];  then lane = pair: s_p = b_s + <w_s, relu(a_p)>
//     forward (lane = d):     attn_d = sum_p sd_p ip_p[d];  y = fc_b + sum over lanes of fc_w[d] attn_d m2_d
//     pass A  (lane = k):     d a_p[k], d W_a[k, :] += d a_p[k] ip_p,  d a_p overwrites a_p
//     pass B  (lane = d):     d ip_p[d] = sd_p d attn[d] + sum_k W_a[k][d] d a_p[k],  overwrites d a_p once every lane has read it
// The staged rows have an odd pitch AP, so the pair-per-lane reads are free of bank conflicts.  Every sum has a fixed order and
// the per-warp partials are reduced by the fixed-order pass: bit-identical from run to run.  The dropout masks are the same
// (seed, counter) indices as the other kernels, or the given `masks`.
template <int D>
struct AfmWide {
    static constexpr int AP = D | 1;                      // floats per staged pair row
};
// exp(s_p - max) of one sample into sc (and a_p into aS); returns sum_p exp(s_p - max).  wrow / ba_k: lane k's row of W_a, b_a[k]
template <int D>
__device__ __forceinline__ float afm_scores_wide(const float* __restrict__ stage, const float* __restrict__ par, const float (&wrow)[D],
                                                 float ba_k, const unsigned char* __restrict__ pi, const unsigned char* __restrict__ pj,
                                                 float* __restrict__ aS, float* __restrict__ sc, int npair, int lane) {
    constexpr int DP = AfmSmem<D>::DP, AP = AfmWide<D>::AP;
    for (int p = 0; p < npair; ++p) {
        const float* vi = stage + pi[p] * D;
        const float* vj = stage + pj[p] * D;
        float a = ba_k;
#pragma unroll
        for (int d = 0; d < D; ++d) a = fmaf(wrow[d], vi[d] * vj[d], a);
        if (lane < D) aS[p * AP + lane] = a;
    }
    __syncwarp();
    const float* ws = par + D * DP + DP;
    const float bs = par[D * DP + 3 * DP];
    float mx = -INFINITY;
    for (int p = lane; p < npair; p += 32) {
        float s = bs;
        for (int k = 0; k < D; ++k) s = fmaf(ws[k], fmaxf(aS[p * AP + k], 0.f), s);
        sc[p] = s;
        mx = fmaxf(mx, s);
    }
    mx = afm_warp_max(mx);
    float sum = 0.f;
    for (int p = lane; p < npair; p += 32) {
        const float e = expf(sc[p] - mx);
        sc[p] = e;
        sum += e;
    }
    return afm_warp_sum(sum);
}

// dynamic smem: PAR | nw * (fd_pad + npair_pad + npair * AP) floats | 2 * npair bytes
template <int D>
__global__ void __launch_bounds__(AFM_WARPS * 32)
afm_fwd_wide_kernel(const float* __restrict__ rows, int64_t ld_rows, const float* __restrict__ params, AfmDrop dr,
                    float* __restrict__ out, int64_t batch, int fields) {
    extern __shared__ __align__(16) float smem[];
    constexpr int DP = AfmSmem<D>::DP, PAR = AfmSmem<D>::PAR, AP = AfmWide<D>::AP;
    static_assert(D <= 32, "one lane per output unit");
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int fd = fields * D, npair = fields * (fields - 1) / 2, npp = (npair + 3) / 4 * 4;
    const int per_warp = ((fd + 3) & ~3) + npp + npair * AP;
    float* par = smem;
    float* stage = smem + PAR + wib * per_warp;
    float* sc = stage + ((fd + 3) & ~3);
    float* aS = sc + npp;
    unsigned char* pi = reinterpret_cast<unsigned char*>(smem + PAR + nw * per_warp);
    unsigned char* pj = pi + npair;
    AfmSmem<D>::load(par, params);
    afm_pair_tables(pi, pj, nullptr, fields);
    __syncthreads();
    uint64_t seed = 0, ctr = 0;
    if (dr.rng && !dr.masks) { seed = dr.rng[0]; ctr = dr.rng[1]; }
    const bool own = lane < D;
    float wrow[D];
#pragma unroll
    for (int d = 0; d < D; ++d) wrow[d] = own ? par[lane * DP + d] : 0.f;
    const float ba_k = own ? par[D * DP + lane] : 0.f;
    const float fcw_d = own ? par[D * DP + 2 * DP + lane] : 0.f;
    const float fcb = par[D * DP + 3 * DP + 1];
    const int width = npair + D;
    for (int64_t b = (int64_t)blockIdx.x * nw + wib; b < batch; b += (int64_t)gridDim.x * nw) {
        const float* r = rows + b * ld_rows;
        for (int i = lane; i < fd; i += 32) stage[i] = __ldg(r + i);
        __syncwarp();
        const float sum = afm_scores_wide<D>(stage, par, wrow, ba_k, pi, pj, aS, sc, npair, lane);
        for (int p = lane; p < npair; p += 32) sc[p] = sc[p] / sum * afm_mask(dr, seed, ctr, b, width, p);     // sd_p
        __syncwarp();
        float y = 0.f;
        if (own) {
            float at = 0.f;
            for (int p = 0; p < npair; ++p) at = fmaf(sc[p], stage[pi[p] * D + lane] * stage[pj[p] * D + lane], at);
            y = fcw_d * (at * afm_mask(dr, seed, ctr, b, width, npair + lane));
        }
        y = afm_warp_sum(y);
        if (lane == 0) out[b] = fcb + y;
        __syncwarp();
    }
}

// dynamic smem: PAR | nw * (fd_pad + 2 * npair_pad + DP + npair * AP) floats | 2 * npair + fields * fields bytes
template <int D>
__global__ void __launch_bounds__(AFM_WARPS * 32)
afm_bwd_wide_kernel(const float* __restrict__ rows, int64_t ld_rows, const float* __restrict__ params, AfmDrop dr,
                    const float* __restrict__ gout, float* __restrict__ grows, int64_t ld_grows, float* __restrict__ part,
                    int64_t batch, int fields) {
    extern __shared__ __align__(16) float smem[];
    constexpr int DP = AfmSmem<D>::DP, PAR = AfmSmem<D>::PAR, AP = AfmWide<D>::AP;
    constexpr int NP = D * D + 3 * D + 2;
    static_assert(D <= 32, "one lane per output unit");
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int fd = fields * D, npair = fields * (fields - 1) / 2, npp = (npair + 3) / 4 * 4;
    const int fdp = (fd + 3) & ~3;
    const int per_warp = fdp + 2 * npp + DP + npair * AP;
    float* par = smem;
    float* stage = smem + PAR + wib * per_warp;
    float* sc = stage + fdp;                // exp(s_p - max) -> score_p -> sd_p = score_p m1_p
    float* dsc = sc + npp;                  // sd_p -> d L / d(score_p m1_p) -> d L / d s_p
    float* dat = dsc + npp;                 // d L / d attn  [D]
    float* aS = dat + DP;                   // a_p -> d a_p -> d ip_p   [npair, AP]
    unsigned char* pi = reinterpret_cast<unsigned char*>(smem + PAR + nw * per_warp);
    unsigned char* pj = pi + npair;
    unsigned char* pidx = pj + npair;
    AfmSmem<D>::load(par, params);
    afm_pair_tables(pi, pj, pidx, fields);
    __syncthreads();
    uint64_t seed = 0, ctr = 0;
    if (dr.rng && !dr.masks) { seed = dr.rng[0]; ctr = dr.rng[1]; }
    const int width = npair + D;
    const bool own = lane < D;
    float wrow[D], wcol[D], dwa[D];
#pragma unroll
    for (int d = 0; d < D; ++d) {
        wrow[d] = own ? par[lane * DP + d] : 0.f;
        wcol[d] = own ? par[d * DP + lane] : 0.f;
        dwa[d] = 0.f;
    }
    const float ba_k = own ? par[D * DP + lane] : 0.f;
    const float ws_k = own ? par[D * DP + DP + lane] : 0.f;
    const float fcw_d = own ? par[D * DP + 2 * DP + lane] : 0.f;
    float dba_k = 0.f, dws_k = 0.f, dfcw_d = 0.f, dbs = 0.f, dfcb = 0.f;

    for (int64_t b = (int64_t)blockIdx.x * nw + wib; b < batch; b += (int64_t)gridDim.x * nw) {
        const float* r = rows + b * ld_rows;
        for (int i = lane; i < fd; i += 32) stage[i] = __ldg(r + i);
        __syncwarp();
        const float sum = afm_scores_wide<D>(stage, par, wrow, ba_k, pi, pj, aS, sc, npair, lane);
        for (int p = lane; p < npair; p += 32) {
            const float score = sc[p] / sum;
            sc[p] = score;
            dsc[p] = score * afm_mask(dr, seed, ctr, b, width, p);
        }
        __syncwarp();
        // lane d: attention output, d fc_w, d attn
        const float g = __ldg(gout + b);
        if (own) {
            float at = 0.f;
            for (int p = 0; p < npair; ++p) at = fmaf(dsc[p], stage[pi[p] * D + lane] * stage[pj[p] * D + lane], at);
            const float m2 = afm_mask(dr, seed, ctr, b, width, npair + lane);
            dfcw_d = fmaf(g, at * m2, dfcw_d);
            dat[lane] = g * fcw_d * m2;
        }
        dfcb += g;
        __syncwarp();
        // lane = pair: d L / d s_p = score_p (t_p - sum_q score_q t_q),  t_p = <d attn, ip_p> m1_p
        float dot = 0.f;
        for (int p = lane; p < npair; p += 32) {
            const float* vi = stage + pi[p] * D;
            const float* vj = stage + pj[p] * D;
            float t = 0.f;
            for (int d = 0; d < D; ++d) t = fmaf(dat[d], vi[d] * vj[d], t);
            t *= afm_mask(dr, seed, ctr, b, width, p);
            dsc[p] = t;
            dot = fmaf(sc[p], t, dot);
        }
        dot = afm_warp_sum(dot);
        for (int p = lane; p < npair; p += 32) {
            const float score = sc[p];
            const float dsp = score * (dsc[p] - dot);
            dbs += dsp;
            dsc[p] = dsp;
            sc[p] = score * afm_mask(dr, seed, ctr, b, width, p);
        }
        __syncwarp();
        // pass A: lane k
        for (int p = 0; p < npair; ++p) {
            const float* vi = stage + pi[p] * D;
            const float* vj = stage + pj[p] * D;
            const float a = own ? aS[p * AP + lane] : 0.f;
            const float dsp = dsc[p];
            const float da = a > 0.f ? dsp * ws_k : 0.f;
            dws_k = fmaf(dsp, fmaxf(a, 0.f), dws_k);
            dba_k += da;
#pragma unroll
            for (int d = 0; d < D; ++d) dwa[d] = fmaf(da, vi[d] * vj[d], dwa[d]);
            if (own) aS[p * AP + lane] = da;
        }
        __syncwarp();
        // pass B: lane d; every lane reads row p of d a before it is overwritten by d ip_p
        const float my_dat = own ? dat[lane] : 0.f;
        for (int p = 0; p < npair; ++p) {
            float dip = sc[p] * my_dat;
#pragma unroll
            for (int k = 0; k < D; ++k) dip = fmaf(wcol[k], aS[p * AP + k], dip);
            __syncwarp();
            if (own) aS[p * AP + lane] = dip;
        }
        __syncwarp();
        // d v_i[d] = sum_{j != i} d ip_{pair(i,j)}[d] * v_j[d], j in order (as afm_bwd_kernel)
        for (int t = lane; t < fd; t += 32) {
            const int i = t / D, d = t - i * D;
            const unsigned char* prow = pidx + i * fields;
            float a0 = 0.f, a1 = 0.f;
            int j = 0;
            for (; j + 1 < fields; j += 2) {
                if (j != i) a0 = fmaf(aS[prow[j] * AP + d], stage[j * D + d], a0);
                if (j + 1 != i) a1 = fmaf(aS[prow[j + 1] * AP + d], stage[(j + 1) * D + d], a1);
            }
            if (j < fields && j != i) a0 = fmaf(aS[prow[j] * AP + d], stage[j * D + d], a0);
            grows[b * ld_grows + t] = a0 + a1;
        }
        __syncwarp();
    }
    float* mine = part + ((int64_t)blockIdx.x * nw + wib) * NP;
    if (own) {
#pragma unroll
        for (int d = 0; d < D; ++d) mine[lane * D + d] = dwa[d];
        mine[D * D + lane] = dba_k;
        mine[D * D + D + lane] = dws_k;
        mine[D * D + 2 * D + 1 + lane] = dfcw_d;
    }
    const float sbs = afm_warp_sum(dbs);
    if (lane == 0) { mine[D * D + 2 * D] = sbs; mine[D * D + 3 * D + 1] = dfcb; }
}

static int afm_blocks(int64_t batch, int per_sm) {
    int64_t want = (batch + AFM_WARPS - 1) / AFM_WARPS;
    const int64_t cap = (int64_t)RLCTR_SMS * per_sm;
    return (int)(want < cap ? (want < 1 ? 1 : want) : cap);
}

template <int D>
static int afm_fwd_launch(const float* rows, int64_t ld_rows, const float* params, const AfmDrop& dr, float* out, int64_t batch,
                          int fields, cudaStream_t st) {
    const int fd = fields * D, npair = fields * (fields - 1) / 2, npp = (npair + 3) / 4 * 4;
    const size_t smem = (size_t)(AfmSmem<D>::PAR + AFM_WARPS * (fd + npp)) * sizeof(float) + 2 * (size_t)npair;
    if (smem > 48 * 1024) return RLCTR_EUNSUPPORTED;
    afm_fwd_kernel<D><<<afm_blocks(batch, 8), AFM_WARPS * 32, smem, st>>>(rows, ld_rows, params, dr, out, batch, fields);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

template <int D>
static int afm_bwd_launch(const float* rows, int64_t ld_rows, const float* params, const AfmDrop& dr, const float* gout,
                          float* grows, int64_t ld_grows, float* dparams, float* part, int64_t batch, int fields, cudaStream_t st) {
    const int fd = fields * D, npair = fields * (fields - 1) / 2, npp = (npair + 3) / 4 * 4;
    const size_t smem = (size_t)(AfmSmem<D>::PAR + AFM_WARPS * (((fd + 3) & ~3) + 2 * npp + 3 * npair * AfmSmem<D>::DP)) * sizeof(float) + 2 * (size_t)npair +
                        (size_t)fields * fields;
    if (smem > 200 * 1024) return RLCTR_EUNSUPPORTED;
    if (smem > 48 * 1024)
        RLCTR_CUDA(cudaFuncSetAttribute(afm_bwd_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int blocks = afm_blocks(batch, 3);
    constexpr int NP = D * D + 3 * D + 2;
    afm_bwd_kernel<D><<<blocks, AFM_WARPS * 32, smem, st>>>(rows, ld_rows, params, dr, gout, grows, ld_grows, part, batch, fields);
    RLCTR_LAUNCH_CHECK();
    colsum_parts_kernel<<<colsum_parts_grid(NP), 256, 0, st>>>(part, dparams, nullptr, NP, 0, NP, blocks * AFM_WARPS);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

// D <= 10: the per-lane kernels; above that the wide kernels, with AFM_WARPS warps per block or fewer when their staging does not
// fit (F = 23 at D = 32 takes two in the backward).  The partials never outnumber rlctr_afm_ws_bytes' blocks * AFM_WARPS.
constexpr int AFM_LANE_MAX_D = 10;
static int afm_wide_warps(size_t fixed, size_t per_warp, size_t* smem) {
    int nw = AFM_WARPS;
    while (nw > 1 && fixed + nw * per_warp > 200 * 1024) nw >>= 1;
    *smem = fixed + nw * per_warp;
    return *smem > 200 * 1024 ? 0 : nw;
}
template <int D>
static int afm_fwd_dispatch(const float* rows, int64_t ld_rows, const float* params, const AfmDrop& dr, float* out, int64_t batch,
                            int fields, cudaStream_t st) {
    if constexpr (D <= AFM_LANE_MAX_D) {
        return afm_fwd_launch<D>(rows, ld_rows, params, dr, out, batch, fields, st);
    } else {
        const int fd = fields * D, npair = fields * (fields - 1) / 2, npp = (npair + 3) / 4 * 4;
        size_t smem;
        const int nw = afm_wide_warps((size_t)AfmSmem<D>::PAR * sizeof(float) + 2 * (size_t)npair,
                                      (size_t)(((fd + 3) & ~3) + npp + npair * AfmWide<D>::AP) * sizeof(float), &smem);
        if (!nw) return RLCTR_EUNSUPPORTED;
        if (smem > 48 * 1024)
            RLCTR_CUDA(cudaFuncSetAttribute(afm_fwd_wide_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int64_t want = (batch + nw - 1) / nw;
        const int64_t cap = (int64_t)RLCTR_SMS * 8;
        afm_fwd_wide_kernel<D><<<(int)(want < cap ? want : cap), nw * 32, smem, st>>>(rows, ld_rows, params, dr, out, batch, fields);
        RLCTR_LAUNCH_CHECK();
        return RLCTR_OK;
    }
}
template <int D>
static int afm_bwd_dispatch(const float* rows, int64_t ld_rows, const float* params, const AfmDrop& dr, const float* gout,
                            float* grows, int64_t ld_grows, float* dparams, float* part, int64_t batch, int fields, cudaStream_t st) {
    if constexpr (D <= AFM_LANE_MAX_D) {
        return afm_bwd_launch<D>(rows, ld_rows, params, dr, gout, grows, ld_grows, dparams, part, batch, fields, st);
    } else {
        const int fd = fields * D, npair = fields * (fields - 1) / 2, npp = (npair + 3) / 4 * 4;
        size_t smem;
        const int nw = afm_wide_warps((size_t)AfmSmem<D>::PAR * sizeof(float) + 2 * (size_t)npair + (size_t)fields * fields,
                                      (size_t)(((fd + 3) & ~3) + 2 * npp + AfmSmem<D>::DP + npair * AfmWide<D>::AP) * sizeof(float),
                                      &smem);
        if (!nw) return RLCTR_EUNSUPPORTED;
        if (smem > 48 * 1024)
            RLCTR_CUDA(cudaFuncSetAttribute(afm_bwd_wide_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const int blocks = afm_blocks(batch, 3);
        constexpr int NP = D * D + 3 * D + 2;
        afm_bwd_wide_kernel<D><<<blocks, nw * 32, smem, st>>>(rows, ld_rows, params, dr, gout, grows, ld_grows, part, batch, fields);
        RLCTR_LAUNCH_CHECK();
        colsum_parts_kernel<<<colsum_parts_grid(NP), 256, 0, st>>>(part, dparams, nullptr, NP, 0, NP, blocks * nw);
        RLCTR_LAUNCH_CHECK();
        return RLCTR_OK;
    }
}

#define AFM_DIMS(X) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(16) \
                    X(17) X(18) X(19) X(20) X(21) X(22) X(23) X(24) X(25) X(26) X(27) X(28) X(29) X(30) X(31) X(32)
constexpr int AFM_MAX_D = 32;

}  // namespace rlctr

using namespace rlctr;

extern "C" size_t rlctr_afm_ws_bytes(int64_t batch, int32_t dim) {
    if (batch <= 0 || dim <= 0) return 256;
    return (size_t)afm_blocks(batch, 3) * AFM_WARPS * (dim * dim + 3 * dim + 2) * sizeof(float) + 256;
}

static int afm_drop(AfmDrop* dr, float dropout_p, const uint64_t* rng_state, const float* masks) {
    if (dropout_p < 0.f || dropout_p >= 1.f) return RLCTR_EINVAL;
    dr->masks = masks;
    dr->rng = (dropout_p > 0.f && !masks) ? rng_state : nullptr;
    if (dropout_p > 0.f && !masks && !rng_state) return RLCTR_EINVAL;
    dr->thresh = dropout_thresh(dropout_p);
    dr->scale = 1.0f / (1.0f - dropout_p);
    return RLCTR_OK;
}

extern "C" int rlctr_afm_fwd(const float* rows, int64_t ld_rows, const float* params, float* out, int64_t batch, int32_t fields,
                             int32_t dim, float dropout_p, const uint64_t* rng_state, const float* masks, rlctr_stream_t stream) {
    if (!rows || !params || !out || batch < 0 || fields < 2 || dim <= 0) return RLCTR_EINVAL;
    if (fields > 23 || dim > AFM_MAX_D) return RLCTR_EUNSUPPORTED;
    if (ld_rows < (int64_t)fields * dim) return RLCTR_EINVAL;
    AfmDrop dr;
    int rc = afm_drop(&dr, dropout_p, rng_state, masks);
    if (rc) return rc;
    if (batch == 0) return RLCTR_OK;
    cudaStream_t st = (cudaStream_t)stream;
    switch (dim) {
#define AFM_FWD_CASE(DD) case DD: return afm_fwd_dispatch<DD>(rows, ld_rows, params, dr, out, batch, fields, st);
        AFM_DIMS(AFM_FWD_CASE)
#undef AFM_FWD_CASE
        default: return RLCTR_EUNSUPPORTED;
    }
}

extern "C" int rlctr_afm_bwd(const float* rows, int64_t ld_rows, const float* params, const float* gout, float* grows,
                             int64_t ld_grows, float* dparams, int64_t batch, int32_t fields, int32_t dim, float dropout_p,
                             const uint64_t* rng_state, const float* masks, void* ws, size_t ws_bytes, rlctr_stream_t stream) {
    if (!rows || !params || !gout || !grows || !dparams || batch <= 0 || fields < 2 || dim <= 0) return RLCTR_EINVAL;
    if (fields > 23 || dim > AFM_MAX_D) return RLCTR_EUNSUPPORTED;
    if (ld_rows < (int64_t)fields * dim || ld_grows < (int64_t)fields * dim) return RLCTR_EINVAL;
    if (!ws || ws_bytes < rlctr_afm_ws_bytes(batch, dim)) return RLCTR_EWORKSPACE;
    AfmDrop dr;
    int rc = afm_drop(&dr, dropout_p, rng_state, masks);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    float* part = reinterpret_cast<float*>(ws);
    switch (dim) {
#define AFM_BWD_CASE(DD) \
        case DD: return afm_bwd_dispatch<DD>(rows, ld_rows, params, dr, gout, grows, ld_grows, dparams, part, batch, fields, st);
        AFM_DIMS(AFM_BWD_CASE)
#undef AFM_BWD_CASE
        default: return RLCTR_EUNSUPPORTED;
    }
}
