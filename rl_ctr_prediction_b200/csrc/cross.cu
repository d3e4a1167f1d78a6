// cross.cu -- the DCN cross network (p_model.py:408-419,423-428) over already-gathered rows, forward and backward.
//
//     x_{l+1} = x_0 * <x_l, w_l> + b_l + x_l,     l = 0 .. L-1,     x_0 = concat_f v_f  (F*D floats per sample)
//
// The reference runs 4 ATen kernels per layer over [B, F*D] temporaries (Linear(F*D, 1), mul, two adds) and autograd
// replays them; here a warp owns a sample, keeps x_0 and x_l in registers (C columns per lane), takes the dot product
// with a butterfly sum and writes x_L once.  Only the L scalars s_l = <x_l, w_l> are saved: the backward recomputes the
// x_l from them.  Parameter gradients (dw_l = sum_b ds_l * x_l, db_l = sum_b g_{l+1}) are accumulated per warp in
// registers, combined per block through shared memory in a fixed order and written as per-block partials, which a
// fixed-order pass (colsum_parts_kernel) reduces: bit-identical from run to run.
//
// C columns per lane: C = 8 serves F*D <= 256, C = 16 serves F*D <= 512 (D up to 32 at F = 15).  At C = 16 the 2*L*C gradient
// accumulators (160 floats at L = 5) no longer fit beside x_l in registers: each lane accumulates them in its own columns of the
// warp's shared-memory slice instead -- the same per-element fma sequence, so the same numbers.
#include "common.cuh"

namespace rlctr {

constexpr int CROSS_MAX_L = 8;         // layers
constexpr int CROSS_C = 8;             // columns per lane: F*D <= 256
constexpr int CROSS_C_WIDE = 16;       // F*D <= 512
constexpr int CROSS_WARPS = 4;

__device__ __forceinline__ float warp_sum(float x) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) x += __shfl_xor_sync(RLCTR_FULL, x, off);
    return x;
}

template <int C>
__global__ void __launch_bounds__(CROSS_WARPS * 32)
cross_fwd_kernel(const float* __restrict__ x0, int64_t ldx, const float* __restrict__ w, const float* __restrict__ b, int layers,
                 float* __restrict__ out, int64_t ld_out, float* __restrict__ s_saved, int64_t batch, int dim) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (int64_t)blockIdx.x * CROSS_WARPS + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * CROSS_WARPS;
    for (int64_t r = warp0; r < batch; r += nwarps) {
        float a0[C], a[C];
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const int k = lane + 32 * c;
            a0[c] = k < dim ? __ldg(x0 + r * ldx + k) : 0.f;
            a[c] = a0[c];
        }
        for (int l = 0; l < layers; ++l) {
            float d = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const int k = lane + 32 * c;
                if (k < dim) d = fmaf(a[c], __ldg(w + l * dim + k), d);
            }
            const float s = warp_sum(d);
            if (lane == 0 && s_saved) s_saved[r * layers + l] = s;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const int k = lane + 32 * c;
                if (k < dim) a[c] = a0[c] * s + __ldg(b + l * dim + k) + a[c];      // (x0 * s + b) + x, the reference's order
            }
        }
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const int k = lane + 32 * c;
            if (k < dim) out[r * ld_out + k] = a[c];
        }
    }
}

// dynamic smem: CROSS_WARPS * 2 * layers * dim floats (per-warp dw | db partials)
template <int L, int C>
__global__ void __launch_bounds__(CROSS_WARPS * 32)
cross_bwd_kernel(const float* __restrict__ x0, int64_t ldx, const float* __restrict__ w, const float* __restrict__ b,
                 const float* __restrict__ s_saved, const float* __restrict__ gout, int64_t ld_g, float* __restrict__ gx0,
                 int64_t ld_gx, float* __restrict__ dw_part, float* __restrict__ db_part, int64_t batch, int dim) {
    extern __shared__ float red[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t warp0 = (int64_t)blockIdx.x * CROSS_WARPS + wib;
    const int64_t nwarps = (int64_t)gridDim.x * CROSS_WARPS;
    constexpr bool REG = C <= CROSS_C;                                     // gradient accumulators in registers, or in `mine`
    float* mine = red + (size_t)wib * 2 * L * dim;
    float dw[REG ? L : 1][C], db[REG ? L : 1][C];
#pragma unroll
    for (int l = 0; l < (REG ? L : 1); ++l)
#pragma unroll
        for (int c = 0; c < C; ++c) { dw[l][c] = 0.f; db[l][c] = 0.f; }
    if (!REG) {
        for (int i = lane; i < 2 * L * dim; i += 32) mine[i] = 0.f;
        __syncwarp();
    }
    for (int64_t r = warp0; r < batch; r += nwarps) {
        float a0[C], xl[L][C], g[C], g0[C], s[L];
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const int k = lane + 32 * c;
            a0[c] = k < dim ? __ldg(x0 + r * ldx + k) : 0.f;
            g[c] = k < dim ? __ldg(gout + r * ld_g + k) : 0.f;
            g0[c] = 0.f;
            xl[0][c] = a0[c];
        }
#pragma unroll
        for (int l = 0; l < L; ++l) s[l] = __ldg(s_saved + r * L + l);
        // recompute x_1 .. x_{L-1} from the saved scalars (x_L itself is not needed)
#pragma unroll
        for (int l = 0; l + 1 < L; ++l)
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const int k = lane + 32 * c;
                xl[l + 1][c] = k < dim ? a0[c] * s[l] + __ldg(b + l * dim + k) + xl[l][c] : 0.f;
            }
#pragma unroll
        for (int l = L - 1; l >= 0; --l) {
            float d = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) d = fmaf(g[c], a0[c], d);
            const float ds = warp_sum(d);                                  // dL/ds_l = <g_{l+1}, x_0>
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const int k = lane + 32 * c;
                if constexpr (REG) {
                    db[l][c] += g[c];                                      // dL/db_l
                    dw[l][c] = fmaf(ds, xl[l][c], dw[l][c]);               // dL/dw_l
                } else if (k < dim) {                                      // lane-private columns: no race
                    mine[(L + l) * dim + k] += g[c];
                    mine[l * dim + k] = fmaf(ds, xl[l][c], mine[l * dim + k]);
                }
                g0[c] = fmaf(g[c], s[l], g0[c]);                           // dL/dx_0 through the explicit x_0 factor
                if (k < dim) g[c] = fmaf(ds, __ldg(w + l * dim + k), g[c]);    // g_l = g_{l+1} + ds * w_l
            }
        }
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const int k = lane + 32 * c;
            if (k < dim) gx0[r * ld_gx + k] = g0[c] + g[c];                // + g_0 (x_0 is also the first x_l)
        }
    }
    // block partials: warps in a fixed order
    if constexpr (REG) {
#pragma unroll
        for (int l = 0; l < L; ++l)
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const int k = lane + 32 * c;
                if (k < dim) { mine[l * dim + k] = dw[l][c]; mine[(L + l) * dim + k] = db[l][c]; }
            }
    }
    __syncthreads();
    const int per = L * dim;
    for (int i = threadIdx.x; i < per; i += blockDim.x) {
        float sw = 0.f, sb = 0.f;
        for (int q = 0; q < CROSS_WARPS; ++q) { sw += red[(size_t)q * 2 * per + i]; sb += red[(size_t)q * 2 * per + per + i]; }
        dw_part[(int64_t)blockIdx.x * per + i] = sw;
        db_part[(int64_t)blockIdx.x * per + i] = sb;
    }
}

static int cross_blocks(int64_t batch) {
    int64_t want = (batch + CROSS_WARPS - 1) / CROSS_WARPS;
    const int64_t cap = (int64_t)RLCTR_SMS * 4;
    return (int)(want < cap ? (want < 1 ? 1 : want) : cap);
}

}  // namespace rlctr

using namespace rlctr;

extern "C" size_t rlctr_cross_ws_bytes(int64_t batch, int32_t dim, int32_t layers) {
    if (batch <= 0 || dim <= 0 || layers <= 0) return 256;
    return (size_t)2 * cross_blocks(batch) * layers * dim * sizeof(float) + 256;
}

extern "C" int rlctr_cross_fwd(const float* x0, int64_t ldx, const float* w, const float* b, int32_t layers, float* out,
                               int64_t ld_out, float* s_saved, int64_t batch, int32_t dim, rlctr_stream_t stream) {
    if (!x0 || !w || !b || !out || batch < 0 || dim <= 0 || layers <= 0) return RLCTR_EINVAL;
    if (dim > 32 * CROSS_C_WIDE || layers > CROSS_MAX_L) return RLCTR_EUNSUPPORTED;
    if (ldx < dim || ld_out < dim) return RLCTR_EINVAL;
    if (batch == 0) return RLCTR_OK;
    if (dim <= 32 * CROSS_C)
        cross_fwd_kernel<CROSS_C><<<cross_blocks(batch), CROSS_WARPS * 32, 0, (cudaStream_t)stream>>>(x0, ldx, w, b, layers, out, ld_out,
                                                                                                     s_saved, batch, dim);
    else
        cross_fwd_kernel<CROSS_C_WIDE><<<cross_blocks(batch), CROSS_WARPS * 32, 0, (cudaStream_t)stream>>>(x0, ldx, w, b, layers, out,
                                                                                                          ld_out, s_saved, batch, dim);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

extern "C" int rlctr_cross_bwd(const float* x0, int64_t ldx, const float* w, const float* b, const float* s_saved, int32_t layers,
                               const float* gout, int64_t ld_g, float* gx0, int64_t ld_gx, float* dw, float* db, int64_t batch,
                               int32_t dim, void* ws, size_t ws_bytes, rlctr_stream_t stream) {
    if (!x0 || !w || !b || !s_saved || !gout || !gx0 || !dw || !db || batch <= 0 || dim <= 0) return RLCTR_EINVAL;
    if (dim > 32 * CROSS_C_WIDE) return RLCTR_EUNSUPPORTED;
    if (ldx < dim || ld_g < dim || ld_gx < dim) return RLCTR_EINVAL;
    if (!ws || ws_bytes < rlctr_cross_ws_bytes(batch, dim, layers)) return RLCTR_EWORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const int blocks = cross_blocks(batch);
    const int per = layers * dim;
    float* dw_part = reinterpret_cast<float*>(ws);
    float* db_part = dw_part + (size_t)blocks * per;
    const size_t smem = (size_t)CROSS_WARPS * 2 * per * sizeof(float);
    const bool wide = dim > 32 * CROSS_C;
    if (smem > (wide ? 128 : 48) * 1024) return RLCTR_EUNSUPPORTED;          // wide: 4 x 2 x 6 x 512 floats at most
#define LAUNCH_CROSS(LL)                                                                                                   \
    if (!wide) {                                                                                                           \
        cross_bwd_kernel<LL, CROSS_C><<<blocks, CROSS_WARPS * 32, smem, st>>>(x0, ldx, w, b, s_saved, gout, ld_g, gx0, ld_gx, dw_part, \
                                                                              db_part, batch, dim);                        \
    } else {                                                                                                               \
        if (smem > 48 * 1024)                                                                                              \
            RLCTR_CUDA(cudaFuncSetAttribute(cross_bwd_kernel<LL, CROSS_C_WIDE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        cross_bwd_kernel<LL, CROSS_C_WIDE><<<blocks, CROSS_WARPS * 32, smem, st>>>(x0, ldx, w, b, s_saved, gout, ld_g, gx0, ld_gx,  \
                                                                                   dw_part, db_part, batch, dim);          \
    }
    switch (layers) {
        case 1: LAUNCH_CROSS(1); break;
        case 2: LAUNCH_CROSS(2); break;
        case 3: LAUNCH_CROSS(3); break;
        case 4: LAUNCH_CROSS(4); break;
        case 5: LAUNCH_CROSS(5); break;
        case 6: LAUNCH_CROSS(6); break;
        default: return RLCTR_EUNSUPPORTED;
    }
#undef LAUNCH_CROSS
    RLCTR_LAUNCH_CHECK();
    colsum_parts_kernel<<<colsum_parts_grid(per), 256, 0, st>>>(dw_part, dw, nullptr, per, 0, per, blocks);
    RLCTR_LAUNCH_CHECK();
    colsum_parts_kernel<<<colsum_parts_grid(per), 256, 0, st>>>(db_part, db, nullptr, per, 0, per, blocks);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// OuterPNN product term (p_model.py:236,245-251).  The reference's kernel matrix is a constant torch.ones((D, D)) (not a
// parameter, not in the state_dict), so  sum_i (S_j * K[i,j]) * S_j  collapses to D copies of S_j^2, S = sum_f v_f:
//     out[b, :] = [ E (F*D) | cross (D) ],   cross[d] = sum_{i<D} (S_d * 1) * S_d   (summed in i order like torch.sum(dim=1))
//     d E[f, d] = g_E[f, d] + g_cross[d] * 2 * D * S_d
// Warp per sample; the row block is staged in shared memory.
// ------------------------------------------------------------------------------------------------------------------
namespace rlctr {

__global__ void __launch_bounds__(128)
fieldsq_fwd_kernel(const float* __restrict__ rows, int64_t ld_rows, float* __restrict__ out, int64_t ld_out, int64_t batch,
                   int fields, int dim) {
    extern __shared__ float smem[];
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int fd = fields * dim;
    float* stage = smem + wib * fd;
    for (int64_t b = (int64_t)blockIdx.x * nw + wib; b < batch; b += (int64_t)gridDim.x * nw) {
        const float* r = rows + b * ld_rows;
        float* o = out + b * ld_out;
        for (int i = lane; i < fd; i += 32) { const float v = __ldg(r + i); stage[i] = v; o[i] = v; }
        __syncwarp();
        for (int d = lane; d < dim; d += 32) {
            float s = 0.f;
            for (int f = 0; f < fields; ++f) s += stage[f * dim + d];
            const float sq = s * s;
            float acc = 0.f;
            for (int i = 0; i < dim; ++i) acc += sq;
            o[fd + d] = acc;
        }
        __syncwarp();
    }
}

__global__ void __launch_bounds__(128)
fieldsq_bwd_kernel(const float* __restrict__ rows, int64_t ld_rows, const float* __restrict__ gout, int64_t ld_g,
                   float* __restrict__ grows, int64_t ld_grows, int64_t batch, int fields, int dim) {
    extern __shared__ float smem[];
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int fd = fields * dim;
    float* stage = smem + wib * (fd + dim);
    float* coef = stage + fd;                          // g_cross[d] * 2 * D * S_d
    for (int64_t b = (int64_t)blockIdx.x * nw + wib; b < batch; b += (int64_t)gridDim.x * nw) {
        const float* r = rows + b * ld_rows;
        const float* g = gout + b * ld_g;
        for (int i = lane; i < fd; i += 32) stage[i] = __ldg(r + i);
        __syncwarp();
        for (int d = lane; d < dim; d += 32) {
            float s = 0.f;
            for (int f = 0; f < fields; ++f) s += stage[f * dim + d];
            coef[d] = __ldg(g + fd + d) * (2.f * (float)dim) * s;
        }
        __syncwarp();
        for (int t = lane; t < fd; t += 32) grows[b * ld_grows + t] = __ldg(g + t) + coef[t % dim];
        __syncwarp();
    }
}

}  // namespace rlctr

extern "C" int rlctr_fieldsq_fwd(const float* rows, int64_t ld_rows, float* out, int64_t ld_out, int64_t batch, int32_t fields,
                                 int32_t dim, rlctr_stream_t stream) {
    if (!rows || !out || batch < 0 || fields <= 0 || dim <= 0) return RLCTR_EINVAL;
    const int fd = fields * dim;
    if (ld_rows < fd || ld_out < fd + dim) return RLCTR_EINVAL;
    if (batch == 0) return RLCTR_OK;
    const int nw = 4;
    const size_t smem = (size_t)nw * fd * sizeof(float);
    if (smem > 48 * 1024) return RLCTR_EUNSUPPORTED;
    int64_t want = (batch + nw - 1) / nw;
    const int64_t cap = (int64_t)RLCTR_SMS * 16;
    fieldsq_fwd_kernel<<<(int)(want < cap ? want : cap), nw * 32, smem, (cudaStream_t)stream>>>(rows, ld_rows, out, ld_out, batch,
                                                                                               fields, dim);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

extern "C" int rlctr_fieldsq_bwd(const float* rows, int64_t ld_rows, const float* gout, int64_t ld_g, float* grows,
                                 int64_t ld_grows, int64_t batch, int32_t fields, int32_t dim, rlctr_stream_t stream) {
    if (!rows || !gout || !grows || batch < 0 || fields <= 0 || dim <= 0) return RLCTR_EINVAL;
    const int fd = fields * dim;
    if (ld_rows < fd || ld_g < fd + dim || ld_grows < fd) return RLCTR_EINVAL;
    if (batch == 0) return RLCTR_OK;
    const int nw = 4;
    const size_t smem = (size_t)nw * (fd + dim) * sizeof(float);
    if (smem > 48 * 1024) return RLCTR_EUNSUPPORTED;
    int64_t want = (batch + nw - 1) / nw;
    const int64_t cap = (int64_t)RLCTR_SMS * 16;
    fieldsq_bwd_kernel<<<(int)(want < cap ? want : cap), nw * 32, smem, (cudaStream_t)stream>>>(rows, ld_rows, gout, ld_g, grows,
                                                                                               ld_grows, batch, fields, dim);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}
