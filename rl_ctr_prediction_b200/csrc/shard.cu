// shard.cu -- multi-GPU row sharding: route the ids of a local batch to the ranks that own their rows.
//
// Tables are row-sharded over G ranks: owner(id) = id mod G, local_row(id) = id div G (modulo balances the
// Zipf heads of the real vocabularies; SURVEY section 8e).  rlctr_bucket_by_owner groups the n = B*F ids of
// the local batch by owner, STABLY (slot order inside a bucket), so that the owner-side segmented reduction
// sums the row gradients in a fixed order and the whole sharded step is bit-identical from run to run.
// The all-to-all itself is NCCL (torch.distributed) on the buffers this kernel lays out.
#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"

namespace rlctr {

__global__ void __launch_bounds__(256)
owner_keys_kernel(const int64_t* __restrict__ ids, int64_t n, int world, int64_t n_rows, uint32_t* __restrict__ keys,
                  uint32_t* __restrict__ vals) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t id = __ldg(ids + i);
        // out-of-range ids go to rank 0 with an out-of-range local row: gathered as a zero row, never updated
        keys[i] = ((uint64_t)id < (uint64_t)n_rows) ? (uint32_t)(id % world) : 0u;
        vals[i] = (uint32_t)i;
    }
}
__global__ void __launch_bounds__(256)
owner_pack_kernel(const int64_t* __restrict__ ids, int64_t n, int world, int64_t n_rows,
                  const uint32_t* __restrict__ sorted_owner, const uint32_t* __restrict__ sorted_slots,
                  int64_t* __restrict__ send_local, int64_t* __restrict__ pos_of_slot, int64_t* __restrict__ counts) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t slot = __ldg(sorted_slots + k);
        const int64_t id = __ldg(ids + slot);
        send_local[k] = ((uint64_t)id < (uint64_t)n_rows) ? id / world : (int64_t)-1;
        pos_of_slot[slot] = k;
        const uint32_t o = __ldg(sorted_owner + k);
        if (k == n - 1 || __ldg(sorted_owner + k + 1) != o) {          // last element of bucket o
            // bucket o ends at k+1; starts are recovered on the host side as a difference of ends
            counts[o] = k + 1;
        }
    }
}
static inline int bits_for(int world) {
    int b = 1;
    while ((1 << b) < world) ++b;
    return b;
}

}  // namespace rlctr

using namespace rlctr;

extern "C" size_t rlctr_bucket_ws_bytes(int64_t n, int32_t world) {
    if (n <= 0) return 256;
    size_t temp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, temp, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const uint32_t*)nullptr,
                                    (uint32_t*)nullptr, n, 0, bits_for(world));
    size_t arr = ((size_t)n * sizeof(uint32_t) + 255) & ~(size_t)255;
    return 3 * arr + temp + 256;
}

extern "C" int rlctr_bucket_by_owner(const int64_t* ids, int64_t n, int32_t world, int64_t n_rows, int64_t* send_local,
                                     int64_t* pos_of_slot, uint32_t* send_slots, int64_t* bucket_ends, void* ws,
                                     size_t ws_bytes, rlctr_stream_t stream) {
    if (!ids || !send_local || !pos_of_slot || !send_slots || !bucket_ends || !ws || n < 0 || world < 1 || n_rows <= 0)
        return RLCTR_EINVAL;
    if (n >= ((int64_t)1 << 32) || world > 1024) return RLCTR_EUNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    // bucket_ends[o] = end offset of bucket o in the send buffer; empty buckets are filled in by the caller
    // from the preceding end (initialise to -1 here)
    RLCTR_CUDA(cudaMemsetAsync(bucket_ends, 0xff, sizeof(int64_t) * world, st));
    if (n == 0) return RLCTR_OK;
    size_t arr = ((size_t)n * sizeof(uint32_t) + 255) & ~(size_t)255;
    if (ws_bytes < rlctr_bucket_ws_bytes(n, world)) return RLCTR_EWORKSPACE;
    uint32_t* keys = reinterpret_cast<uint32_t*>(ws);
    uint32_t* vals = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(ws) + arr);
    uint32_t* skeys = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(ws) + 2 * arr);
    void* temp = reinterpret_cast<char*>(ws) + 3 * arr;
    size_t temp_bytes = ws_bytes - 3 * arr;
    int64_t blocks = (n + 255) / 256;
    int grid = (int)(blocks < RLCTR_SMS * 8 ? blocks : RLCTR_SMS * 8);
    owner_keys_kernel<<<grid, 256, 0, st>>>(ids, n, world, n_rows, keys, vals);
    RLCTR_LAUNCH_CHECK();
    cudaError_t e = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys, skeys, vals, send_slots, n, 0, bits_for(world), st);
    if (e != cudaSuccess) return (int)e;
    RLCTR_COUNT_LAUNCH(3);
    owner_pack_kernel<<<grid, 256, 0, st>>>(ids, n, world, n_rows, skeys, send_slots, send_local, pos_of_slot, bucket_ends);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

// ---- gradient-side push: the source rank WRITES what an owner needs into the owner's memory ---------------------------------
// Owners used to PULL the per-occurrence gradient rows of remote samples inside the update kernel: 40-600 byte reads with a
// 2-3 us NVLink round trip each, on the dependent path of every row -- latency-bound (rows_adam 0.14 -> 0.36 ms at 8 GPUs).
// Remote WRITES are posted: the source streams row `slot` of its [n, width] array to recv[rank * n + slot] in the memory of
// owner(ids[slot]) and moves on; after the step's barrier the owner's kernel reads only local memory (peer_*[r] = recv + r*n*width).
namespace rlctr {

__global__ void __launch_bounds__(256)
push_rows_kernel(const int64_t* __restrict__ ids, int64_t n, int mask, int64_t n_rows, const float* __restrict__ src, int width,
                 ShardView recv, int64_t base) {
    const int vec = (width % 2 == 0) ? 2 : 1;
    const int per = width / vec;
    const int64_t total = n * per;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t slot = i / per;
        const int j = (int)(i - slot * per);
        const int64_t id = __ldg(ids + slot);
        if ((uint64_t)id >= (uint64_t)n_rows) continue;                      // out-of-range ids own nothing
        float* dst = const_cast<float*>(recv.peers[id & mask]) + (base + slot) * width;
        if (vec == 2) reinterpret_cast<float2*>(dst)[j] = __ldg(reinterpret_cast<const float2*>(src + slot * width) + j);
        else dst[j] = __ldg(src + slot * width + j);
    }
}

}  // namespace rlctr

extern "C" int rlctr_push_rows(const int64_t* ids, int64_t n, int32_t world, int32_t rank, int64_t n_rows_global, const float* src,
                               int32_t width, void* const* peer_recv, rlctr_stream_t stream) {
    if (!ids || !src || !peer_recv || n < 0 || width <= 0 || n_rows_global <= 0) return RLCTR_EINVAL;
    if (world != 2 && world != 4 && world != 8) return RLCTR_EUNSUPPORTED;
    if (rank < 0 || rank >= world) return RLCTR_EINVAL;
    if ((((uintptr_t)src) & 7u) != 0) return RLCTR_EALIGN;
    ShardView sv;
    sv.shift = 0; sv.mask = world - 1;
    for (int r = 0; r < RLCTR_MAX_WORLD; ++r) sv.peers[r] = nullptr;
    for (int r = 0; r < world; ++r) {
        if (!peer_recv[r] || (((uintptr_t)peer_recv[r]) & 7u) != 0) return RLCTR_EINVAL;
        sv.peers[r] = reinterpret_cast<const float*>(peer_recv[r]);
    }
    if (n == 0) return RLCTR_OK;
    const int per = width % 2 == 0 ? width / 2 : width;
    int64_t blocks = (n * per + 255) / 256;
    const int grid = (int)(blocks < RLCTR_SMS * 16 ? blocks : RLCTR_SMS * 16);
    push_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(ids, n, world - 1, n_rows_global, src, width, sv, (int64_t)rank * n);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}


// ---- owner routing of a batch's ids --------------------------------------------------------------------------------------
// The first sharded lookup all-gathered the ids of every rank and let every rank sort all G*n of them to find the ~n it owns
// (sort 0.09 -> 0.24 ms at 8 GPUs).  Here every SOURCE rank buckets its n ids by owner (stable: slot order inside a bucket) and
// WRITES (local row, global slot) of bucket o into its own fixed-capacity segment of owner o's receive buffer
//     keys[o][rank * cap + j], vals[o][rank * cap + j],  j < cap      (posted NVLink writes; unused slots get the sentinel key)
// so an owner sorts G * cap ~ 1.5 n pairs, whatever G is.  A bucket larger than `cap` (skewed ownership) raises the device
// flag `overflow` (checked by the host at flush time): the step is then wrong and must be rerun with a larger capacity.
namespace rlctr {

__global__ void __launch_bounds__(256)
route_keys_kernel(const int64_t* __restrict__ ids, int64_t n, uint32_t mask, uint32_t world, int64_t n_rows,
                  uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t id = __ldg(ids + i);
        keys[i] = ((uint64_t)id < (uint64_t)n_rows) ? ((uint32_t)id & mask) : world;        // out of range: routed nowhere
        vals[i] = (uint32_t)i;
    }
}
__global__ void route_bounds_kernel(const uint32_t* __restrict__ skeys, int64_t n, int world, int64_t cap,
                                    int64_t* __restrict__ starts, int32_t* __restrict__ overflow) {
    const int o = threadIdx.x;
    if (o > world) return;
    int64_t lo = 0, hi = n;                              // lower bound of key o
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(skeys + mid) < (uint32_t)o) lo = mid + 1; else hi = mid;
    }
    starts[o] = lo;
    __syncthreads();
    if (o < world && starts[o + 1] - starts[o] > cap) atomicOr(overflow, 1);
}
struct RoutePeers {
    uint32_t* keys[RLCTR_MAX_WORLD];
    uint32_t* vals[RLCTR_MAX_WORLD];
};
__global__ void __launch_bounds__(256)
route_write_kernel(const int64_t* __restrict__ ids, int64_t n, const uint32_t* __restrict__ skeys,
                   const uint32_t* __restrict__ sslots, const int64_t* __restrict__ starts, int world, int shift, int rank,
                   int64_t cap, const __grid_constant__ RoutePeers peers) {
    const int64_t total = n > (int64_t)world * cap ? n : (int64_t)world * cap;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        if (i < n) {
            const uint32_t o = __ldg(skeys + i);
            if (o < (uint32_t)world) {
                const int64_t j = i - starts[o];
                if (j < cap) {
                    const uint32_t slot = __ldg(sslots + i);
                    const int64_t id = __ldg(ids + slot);
                    peers.keys[o][(int64_t)rank * cap + j] = (uint32_t)(id >> shift);
                    peers.vals[o][(int64_t)rank * cap + j] = (uint32_t)((int64_t)rank * n + slot);
                }
            }
        }
        if (i < (int64_t)world * cap) {                  // sentinel keys behind the bucket's last element
            const int o = (int)(i / cap);
            const int64_t j = i - (int64_t)o * cap;
            if (j >= starts[o + 1] - starts[o]) peers.keys[o][(int64_t)rank * cap + j] = 0xffffffffu;
        }
    }
}

}  // namespace rlctr

extern "C" size_t rlctr_route_ws_bytes(int64_t n, int32_t world) {
    if (n <= 0) return 512;
    size_t temp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, temp, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const uint32_t*)nullptr,
                                    (uint32_t*)nullptr, n, 0, bits_for(world + 1));
    size_t arr = ((size_t)n * sizeof(uint32_t) + 255) & ~(size_t)255;
    return 4 * arr + temp + 512;
}

extern "C" int rlctr_route_ids(const int64_t* ids, int64_t n, int32_t world, int32_t rank, int64_t n_rows_global, int64_t cap,
                               void* const* peer_keys, void* const* peer_vals, int32_t* overflow, void* ws, size_t ws_bytes,
                               rlctr_stream_t stream) {
    if (!ids || !peer_keys || !peer_vals || !overflow || !ws || n < 0 || cap <= 0 || n_rows_global <= 0) return RLCTR_EINVAL;
    if (world != 2 && world != 4 && world != 8) return RLCTR_EUNSUPPORTED;
    if (rank < 0 || rank >= world) return RLCTR_EINVAL;
    if (n >= ((int64_t)1 << 32) / world) return RLCTR_EUNSUPPORTED;                 // global slots are 32-bit
    if (ws_bytes < rlctr_route_ws_bytes(n, world)) return RLCTR_EWORKSPACE;
    RoutePeers peers;
    for (int r = 0; r < world; ++r) {
        if (!peer_keys[r] || !peer_vals[r]) return RLCTR_EINVAL;
        peers.keys[r] = reinterpret_cast<uint32_t*>(peer_keys[r]);
        peers.vals[r] = reinterpret_cast<uint32_t*>(peer_vals[r]);
    }
    cudaStream_t st = (cudaStream_t)stream;
    int shift = 0;
    while ((1 << shift) < world) ++shift;
    size_t arr = ((size_t)(n > 0 ? n : 1) * sizeof(uint32_t) + 255) & ~(size_t)255;
    char* base = reinterpret_cast<char*>(ws);
    uint32_t* keys = reinterpret_cast<uint32_t*>(base);
    uint32_t* vals = reinterpret_cast<uint32_t*>(base + arr);
    uint32_t* skeys = reinterpret_cast<uint32_t*>(base + 2 * arr);
    uint32_t* sslots = reinterpret_cast<uint32_t*>(base + 3 * arr);
    int64_t* starts = reinterpret_cast<int64_t*>(base + 4 * arr);                    // world + 1 entries (256 bytes reserved)
    void* temp = base + 4 * arr + 256;
    size_t temp_bytes = ws_bytes - 4 * arr - 256;
    const int64_t total = n > (int64_t)world * cap ? n : (int64_t)world * cap;
    int64_t blocks = (total + 255) / 256;
    const int grid = (int)(blocks < RLCTR_SMS * 8 ? (blocks < 1 ? 1 : blocks) : RLCTR_SMS * 8);
    if (n > 0) {
        route_keys_kernel<<<grid, 256, 0, st>>>(ids, n, (uint32_t)(world - 1), (uint32_t)world, n_rows_global, keys, vals);
        RLCTR_LAUNCH_CHECK();
        cudaError_t e = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys, skeys, vals, sslots, n, 0, bits_for(world + 1), st);
        if (e != cudaSuccess) return (int)e;
        RLCTR_COUNT_LAUNCH(3);
    }
    route_bounds_kernel<<<1, 32, 0, st>>>(skeys, n, world, cap, starts, overflow);
    RLCTR_LAUNCH_CHECK();
    route_write_kernel<<<grid, 256, 0, st>>>(ids, n, skeys, sslots, starts, world, shift, rank, cap, peers);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

namespace rlctr {
__global__ void __launch_bounds__(256) iota_kernel(uint32_t* __restrict__ out, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = (uint32_t)i;
}
// rows of up to RLCTR_GROUP_MAX sources (src_s [n, width_s], widths even) in the bucket order rlctr_route_ids computed: occurrence
// sslots[i] goes to owner skeys[i] as ONE interleaved row at recv[owner][(rank * cap + i - starts[owner]) * pitch], source s at float
// offset off_s = sum_{t<s} width_t, pitch = sum_s width_s: consecutive threads write consecutive 8-byte pieces of an owner's segment
struct PushSrcs {
    const float* src[RLCTR_GROUP_MAX];
    int width[RLCTR_GROUP_MAX];
    int off[RLCTR_GROUP_MAX];
    int n_src;
};
__global__ void __launch_bounds__(256)
push_routed_kernel(const uint32_t* __restrict__ skeys, const uint32_t* __restrict__ sslots, const int64_t* __restrict__ starts,
                   int64_t n, int world, int64_t seg0, int64_t cap, const __grid_constant__ PushSrcs ps, int pitch,
                   const __grid_constant__ ShardView sv) {
    const int per = pitch >> 1;
    const int64_t total = n * per;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = t / per;
        const int j = (int)(t - i * per);
        const uint32_t o = __ldg(skeys + i);
        if (o >= (uint32_t)world) continue;
        const int64_t pos = i - starts[o];
        if (pos >= cap) continue;                                   // overflow: flagged by rlctr_route_ids
        const uint32_t slot = __ldg(sslots + i);
        int s = 0;                                                  // the source of piece j (n_src <= 4: a short scan)
#pragma unroll
        for (int q = 1; q < RLCTR_GROUP_MAX; ++q)
            if (q < ps.n_src && 2 * j >= ps.off[q]) s = q;
        const int c = 2 * j - ps.off[s];
        const float2 v = __ldg(reinterpret_cast<const float2*>(ps.src[s] + (int64_t)slot * ps.width[s] + c));
        float* dst = const_cast<float*>(sv.peers[o]) + (seg0 + pos) * pitch;
        reinterpret_cast<float2*>(dst)[j] = v;
    }
}
}  // namespace rlctr

extern "C" int rlctr_push_rows_routed_multi(const void* route_ws, int64_t n, int32_t world, int32_t rank, int64_t cap,
                                            const float* const* srcs, const int32_t* widths, int32_t n_src, void* const* peer_recv,
                                            rlctr_stream_t stream) {
    if (!route_ws || !srcs || !widths || !peer_recv || n < 0 || cap <= 0) return RLCTR_EINVAL;
    if (n_src < 1 || n_src > RLCTR_GROUP_MAX) return RLCTR_EINVAL;
    if (world != 2 && world != 4 && world != 8) return RLCTR_EUNSUPPORTED;
    if (rank < 0 || rank >= world) return RLCTR_EINVAL;
    PushSrcs ps;
    ps.n_src = n_src;
    int pitch = 0;
    for (int s = 0; s < RLCTR_GROUP_MAX; ++s) { ps.src[s] = nullptr; ps.width[s] = 0; ps.off[s] = 0; }
    for (int s = 0; s < n_src; ++s) {
        if (!srcs[s] || widths[s] <= 0 || widths[s] % 2 != 0) return RLCTR_EINVAL;
        if ((((uintptr_t)srcs[s]) & 7u) != 0) return RLCTR_EALIGN;
        ps.src[s] = srcs[s]; ps.width[s] = widths[s]; ps.off[s] = pitch;
        pitch += widths[s];
    }
    ShardView sv;
    sv.shift = 0; sv.mask = world - 1;
    for (int r = 0; r < RLCTR_MAX_WORLD; ++r) sv.peers[r] = nullptr;
    for (int r = 0; r < world; ++r) {
        if (!peer_recv[r] || (((uintptr_t)peer_recv[r]) & 7u) != 0) return RLCTR_EINVAL;
        sv.peers[r] = reinterpret_cast<const float*>(peer_recv[r]);
    }
    if (n == 0) return RLCTR_OK;
    // the layout rlctr_route_ids gave its workspace: keys | vals | sorted owner keys | sorted slots | bucket starts
    const size_t arr = ((size_t)n * sizeof(uint32_t) + 255) & ~(size_t)255;
    const char* base = reinterpret_cast<const char*>(route_ws);
    const uint32_t* skeys = reinterpret_cast<const uint32_t*>(base + 2 * arr);
    const uint32_t* sslots = reinterpret_cast<const uint32_t*>(base + 3 * arr);
    const int64_t* starts = reinterpret_cast<const int64_t*>(base + 4 * arr);
    int64_t blocks = (n * (pitch / 2) + 255) / 256;
    const int grid = (int)(blocks < RLCTR_SMS * 16 ? blocks : RLCTR_SMS * 16);
    push_routed_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(skeys, sslots, starts, n, world, (int64_t)rank * cap, cap, ps, pitch, sv);
    RLCTR_LAUNCH_CHECK();
    return RLCTR_OK;
}

// the one-source form: the same kernel, pitch = width (the same bytes in the same places as the multi call with n_src = 1)
extern "C" int rlctr_push_rows_routed(const void* route_ws, int64_t n, int32_t world, int32_t rank, int64_t cap, const float* src,
                                      int32_t width, void* const* peer_recv, rlctr_stream_t stream) {
    if (!src) return RLCTR_EINVAL;
    const float* srcs[1] = {src};
    const int32_t widths[1] = {width};
    return rlctr_push_rows_routed_multi(route_ws, n, world, rank, cap, srcs, widths, 1, peer_recv, stream);
}

extern "C" int rlctr_sort_routed_pos(const uint32_t* keys, int64_t n_in, int64_t n_rows_local, uint32_t* sorted_rows,
                                     uint32_t* sorted_pos, void* ws, size_t ws_bytes, rlctr_stream_t stream) {
    if (!keys || !sorted_rows || !sorted_pos || !ws || n_in < 0 || n_rows_local <= 0) return RLCTR_EINVAL;
    if (n_in == 0) return RLCTR_OK;
    const size_t arr = ((size_t)n_in * sizeof(uint32_t) + 255) & ~(size_t)255;
    if (ws_bytes < arr + 256) return RLCTR_EWORKSPACE;
    uint32_t* pos = reinterpret_cast<uint32_t*>(ws);
    int64_t blocks = (n_in + 255) / 256;
    iota_kernel<<<(int)(blocks < RLCTR_SMS * 8 ? blocks : RLCTR_SMS * 8), 256, 0, (cudaStream_t)stream>>>(pos, n_in);
    RLCTR_LAUNCH_CHECK();
    int bits = 1;
    while (bits < 32 && ((int64_t)1 << bits) <= n_rows_local) ++bits;               // the sentinel (all ones) sorts last
    size_t temp_bytes = ws_bytes - arr;
    cudaError_t e = cub::DeviceRadixSort::SortPairs(static_cast<void*>(reinterpret_cast<char*>(ws) + arr), temp_bytes, keys, sorted_rows,
                                                    static_cast<const uint32_t*>(pos), sorted_pos, n_in, 0, bits, (cudaStream_t)stream);
    if (e != cudaSuccess) return (int)e;
    RLCTR_COUNT_LAUNCH(2 + (bits + 7) / 8);
    return RLCTR_OK;
}

extern "C" int rlctr_sort_routed(const uint32_t* keys, const uint32_t* vals, int64_t n_in, int64_t n_rows_local,
                                 uint32_t* sorted_rows, uint32_t* sorted_slots, void* ws, size_t ws_bytes, rlctr_stream_t stream) {
    if (!keys || !vals || !sorted_rows || !sorted_slots || !ws || n_in < 0 || n_rows_local <= 0) return RLCTR_EINVAL;
    if (n_in == 0) return RLCTR_OK;
    int bits = 1;
    while (bits < 32 && ((int64_t)1 << bits) <= n_rows_local) ++bits;               // the sentinel (all ones) sorts last
    cudaError_t e = cub::DeviceRadixSort::SortPairs(ws, ws_bytes, keys, sorted_rows, vals, sorted_slots, n_in, 0, bits,
                                                    (cudaStream_t)stream);
    if (e != cudaSuccess) return (int)e;
    RLCTR_COUNT_LAUNCH(2 + (bits + 7) / 8);
    return RLCTR_OK;
}
