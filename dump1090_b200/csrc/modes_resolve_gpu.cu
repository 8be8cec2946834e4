// modes_resolve_gpu.cu — the sequential half of detectModeS() on the device (SURVEY.md §8(f) item 4).
//
// What is sequential in the reference — skip past a good message, retry otherwise
// (dump1090.c:1769-1791), the ICAO address cache (:898-983, :1183-1210), the statistics — is
// sequential only WITHIN a 131072-sample buffer as far as the skip state goes (:1593); across
// buffers the only carrier is the 1024-slot address cache.  So:
//   replay    one warp per reference buffer replays its candidates in order from a GUESS of the
//             cache at its start (modes_resolve_core.cuh, the same rules as the host resolve),
//             noting which slots it read before writing them (what its outcome depends on) and
//             which it wrote (what later buffers inherit);
//   hand-over one thread per cache slot walks the buffers: the cache at the start of buffer b is the
//             batch's starting cache overwritten by the last writer of each slot among buffers < b;
//             a buffer whose guess was wrong in a slot it read first is marked for another replay;
//   repeat    a fixed number of rounds (two suffice on real traffic: the first replays everything
//             from the batch's starting cache, the second with the inherited caches; a third run
//             is needed only when a changed verdict changes what a buffer itself writes); then
//   emit      a last replay writes the delivered messages (40-byte records: position, the evaluated
//             frame, crcok / phase_corrected / recovered address) at their final places, in stream
//             order, and adds up the statistics.
// The host then only builds struct modesMessage fields from 40-byte deliveries (in parallel); the
// 56-byte candidate records never leave the GPU (47 MB -> 17 MB per GiB of the dense capture).
// Exactness is checked on the CPU for the algorithm (tests/test_resolve_core_host.py) and on the
// GPU against the host resolver and the oracle (tests/test_gpu_resolve.py).
//
// A receiver pool (modes_pool.cpp) needs none of the guessing: its batch holds one buffer per receiver,
// so pool_resolve_kernel replays each from that receiver's resident cache and writes the cache back
// (count, resolve_offsets_kernel, emit); tests/test_pool_gpu_resolve.py.
#include <cstdint>
#include <cuda_runtime.h>
#include "modes_internal.h"
#include "modes_resolve_core.cuh"

namespace modes {
namespace {

constexpr int kWarpsPerCta = 8;

// The address cache of the buffer being replayed: values in shared memory, the written / read-first
// sets as one 32-bit word per lane (all lanes run the same code on the same slot).
struct WarpCache {
    uint32_t *c;                 // [1024] in shared memory
    uint32_t written, readfirst; // this lane's word of the two 1024-bit sets
    int lane;
    __device__ __forceinline__ uint32_t read(uint32_t s) {
        if (lane == (int)(s >> 5) && !((written >> (s & 31)) & 1u)) readfirst |= 1u << (s & 31);
        return c[s];
    }
    __device__ __forceinline__ void write(uint32_t s, uint32_t a) {
        __syncwarp();
        if (lane == 0) c[s] = a;
        if (lane == (int)(s >> 5)) written |= 1u << (s & 31);
        __syncwarp();
    }
};

// The address cache of a receiver pool's buffer: nothing to track, every buffer starts from the cache
// its receiver really has.
struct SharedCache {
    uint32_t *c;                 // [1024] in shared memory
    int lane;
    __device__ __forceinline__ uint32_t read(uint32_t s) { return c[s]; }
    __device__ __forceinline__ void write(uint32_t s, uint32_t a) {
        __syncwarp();
        if (lane == 0) c[s] = a;
        __syncwarp();
    }
};

__device__ __forceinline__ rcore::Attempt attempt_from_words(uint32_t e0, uint32_t e3, uint32_t e4, uint32_t e5) {
    rcore::Attempt a;
    a.meta = (e3 >> 16) | (e4 << 16);                   // msgtype, flags, errorbit, nfixed
    a.crc = e5;
    a.addr = __byte_perm(e0, 0u, 0x4123);               // msg[1] << 16 | msg[2] << 8 | msg[3]
    return a;
}

// One warp replays the candidates of buffer b of the batch (t >> 17 == b) in stream order and returns
// its delivery count.  kEmit: the deliveries are also written from out + out_base on (below `capacity`),
// with position t - t_shift.
template <bool kEmit, class Cache>
__device__ __forceinline__ uint32_t replay_buffer(Cache &wc, rcore::BufferState &st, const modes_candidate *__restrict__ records,
                                                  const modes_tile *__restrict__ tiles, uint32_t n_tiles, uint32_t b, int check_crc,
                                                  int lane, modes_delivery *out, uint32_t out_base, uint32_t capacity, uint64_t t_shift) {
    uint32_t n_out = 0;
    const uint64_t v_lo = (uint64_t)b * kBufSamples + 2, v_hi = (uint64_t)(b + 1) * kBufSamples + 1;
    uint32_t t_lo = (uint32_t)(v_lo / kTileSamples), t_hi = (uint32_t)(v_hi / kTileSamples);
    if (t_hi >= n_tiles) t_hi = n_tiles - 1;
    for (uint32_t ti = t_lo; ti <= t_hi; ti++) {
        const modes_tile tl = tiles[ti];
        for (uint32_t i0 = 0; i0 < tl.count; i0 += 32) {
            const uint32_t n_here = min(32u, tl.count - i0);
            // lane i holds candidate i0 + i of the tile: 14 words
            uint32_t w[14];
            if ((uint32_t)lane < n_here) {
                const uint2 *rp = reinterpret_cast<const uint2 *>(records + tl.offset + i0 + lane);
#pragma unroll
                for (int k = 0; k < 7; k++) { const uint2 v = rp[k]; w[2 * k] = v.x; w[2 * k + 1] = v.y; }
            } else {
#pragma unroll
                for (int k = 0; k < 14; k++) w[k] = 0;
            }
            for (uint32_t i = 0; i < n_here; i++) {
                const uint32_t t0 = __shfl_sync(0xffffffffu, w[0], i), t1 = __shfl_sync(0xffffffffu, w[1], i);
                const uint64_t t = ((uint64_t)t1 << 32) | t0;
                if ((t >> 17) != (uint64_t)b) continue;            // the tile straddles a buffer boundary
                const rcore::Attempt p1 = attempt_from_words(__shfl_sync(0xffffffffu, w[2], i), __shfl_sync(0xffffffffu, w[5], i),
                                                             __shfl_sync(0xffffffffu, w[6], i), __shfl_sync(0xffffffffu, w[7], i));
                const rcore::Attempt p2 = attempt_from_words(__shfl_sync(0xffffffffu, w[8], i), __shfl_sync(0xffffffffu, w[11], i),
                                                             __shfl_sync(0xffffffffu, w[12], i), __shfl_sync(0xffffffffu, w[13], i));
                rcore::Decision d[2];
                rcore::candidate(st, wc, (uint32_t)(t0 & (kBufSamples - 1)), p1, p2, check_crc, d);
#pragma unroll
                for (int p = 0; p < 2; p++) {
                    if (!d[p].deliver) continue;
                    if (kEmit && lane == (int)i && out_base + n_out < capacity) {
                        modes_delivery *o = out + out_base + n_out;
                        uint32_t *ow = reinterpret_cast<uint32_t *>(o);
                        const uint64_t tp = (((uint64_t)w[1] << 32) | w[0]) - t_shift;     // this lane's own t
                        ow[0] = (uint32_t)tp; ow[1] = (uint32_t)(tp >> 32);
#pragma unroll
                        for (int k = 0; k < 6; k++) ow[2 + k] = w[2 + 6 * p + k];
                        ow[8] = d[p].extra;
                        ow[9] = d[p].crcok | (d[p].phase_corrected << 8) | (d[p].extra_is_ap << 16);
                    }
                    n_out++;
                }
            }
        }
    }
    return n_out;
}

__global__ void __launch_bounds__(256)
resolve_init_kernel(GpuResolve g, uint32_t n_buffers) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < (uint64_t)n_buffers * 1024) g.start[i] = g.cache_in[i & 1023];
    if (i < n_buffers) g.rerun[i] = 1;
    if (i < 8) g.stats_out[i] = 0;
    if (i == 0) { g.flags[0] = 0; g.flags[1] = 0; }
}

// kEmit = false: replay the marked buffers, counting deliveries; kEmit = true: replay all buffers
// once more from their final caches and write the deliveries at offsets[b].
template <bool kEmit>
__global__ void __launch_bounds__(32 * kWarpsPerCta)
resolve_replay_kernel(GpuResolve g, const modes_candidate *__restrict__ records, const modes_tile *__restrict__ tiles,
                      uint32_t n_tiles, uint32_t n_buffers, int check_crc) {
    __shared__ uint32_t s_cache[kWarpsPerCta][1024];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t *cache = s_cache[warp];
    for (uint32_t b = blockIdx.x * kWarpsPerCta + warp; b < n_buffers; b += gridDim.x * kWarpsPerCta) {
        if (!kEmit && !g.rerun[b]) continue;
        __syncwarp();
#pragma unroll
        for (int k = 0; k < 8; k++)
            reinterpret_cast<uint4 *>(cache)[32 * k + lane] = reinterpret_cast<const uint4 *>(g.start + (size_t)b * 1024)[32 * k + lane];
        __syncwarp();
        WarpCache wc{cache, 0u, 0u, lane};
        rcore::BufferState st;
        st.next_j = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) st.stats[k] = 0;
        const uint32_t out_base = kEmit ? g.offsets[b] : 0u;
        const uint32_t n_out = replay_buffer<kEmit>(wc, st, records, tiles, n_tiles, b, check_crc, lane, g.out, out_base, g.capacity, 0);
        __syncwarp();
        if (!kEmit) {
#pragma unroll
            for (int k = 0; k < 8; k++)
                reinterpret_cast<uint4 *>(g.end + (size_t)b * 1024)[32 * k + lane] = reinterpret_cast<const uint4 *>(cache)[32 * k + lane];
            g.written[(size_t)b * 32 + lane] = wc.written;
            g.readfirst[(size_t)b * 32 + lane] = wc.readfirst;
            if (lane == 0) { g.n_deliv[b] = n_out; g.rerun[b] = 0; }
        } else if (lane < 8) {
            atomicAdd(reinterpret_cast<unsigned long long *>(g.stats_out) + lane, (unsigned long long)st.stats[lane]);
        }
    }
}

// One thread per cache slot: hand the caches from buffer to buffer (last writer of the slot wins),
// mark the buffers whose guess was wrong in a slot they read before writing.  The loads of an
// iteration do not depend on the previous one, so they pipeline.
__global__ void __launch_bounds__(128)
resolve_handover_kernel(GpuResolve g, uint32_t n_buffers) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;          // 0 .. 1023
    const uint32_t word = s >> 5, bit = 1u << (s & 31);
    uint32_t cur = g.cache_in[s];
    uint32_t pending = 0;
#pragma unroll 8
    for (uint32_t b = 0; b < n_buffers; b++) {
        const size_t o = (size_t)b * 1024 + s;
        const uint32_t had = g.start[o];
        const uint32_t rf = g.readfirst[(size_t)b * 32 + word], wr = g.written[(size_t)b * 32 + word];
        const uint32_t e = g.end[o];
        if (had != cur) {
            g.start[o] = cur;
            if (rf & bit) { g.rerun[b] = 1; pending = 1; }
        }
        if (wr & bit) cur = e;
    }
    g.cache_out[s] = cur;
    if (pending) g.flags[0] = 1;                                       // somebody has to run again
}

// Exclusive prefix sum of the per-buffer delivery counts (one CTA).
__global__ void __launch_bounds__(1024)
resolve_offsets_kernel(GpuResolve g, uint32_t n_buffers, uint32_t capacity) {
    __shared__ uint32_t s_part[1024];
    const uint32_t per = (n_buffers + 1023) / 1024;
    const uint32_t lo = threadIdx.x * per, hi = min(n_buffers, lo + per);
    uint32_t sum = 0;
    for (uint32_t b = lo; b < hi; b++) sum += g.n_deliv[b];
    s_part[threadIdx.x] = sum;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
        const uint32_t v = threadIdx.x >= (uint32_t)d ? s_part[threadIdx.x - d] : 0u;
        __syncthreads();
        s_part[threadIdx.x] += v;
        __syncthreads();
    }
    uint32_t run = s_part[threadIdx.x] - sum;
    for (uint32_t b = lo; b < hi; b++) { g.offsets[b] = run; run += g.n_deliv[b]; }
    if (threadIdx.x == 1023) {
        g.offsets[n_buffers] = s_part[1023];
        g.flags[2] = s_part[1023];
        if (s_part[1023] > capacity) g.flags[1] = 1;                    // the emit pass would overrun the delivery buffer
    }
}

// Receiver pool: one warp per list entry i replays data buffer 2i+1 from its receiver's cache.
// kEmit = false counts the deliveries and leaves the cache alone; kEmit = true writes the deliveries
// at offsets[i], the statistics, and the cache back.
template <bool kEmit>
__global__ void __launch_bounds__(32 * kWarpsPerCta)
pool_resolve_kernel(PoolResolve p, const modes_candidate *__restrict__ records, const modes_tile *__restrict__ tiles,
                    uint32_t n_tiles, uint32_t n, int check_crc) {
    __shared__ __align__(16) uint32_t s_cache[kWarpsPerCta][1024];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t i = blockIdx.x * kWarpsPerCta + warp;
    if (i >= n) return;                                                // the whole warp
    const uint32_t id = p.ids[i] & ~kPoolFresh;
    const bool fresh = p.ids[i] & kPoolFresh;
    uint32_t *cache = s_cache[warp];
    uint4 *resident = reinterpret_cast<uint4 *>(p.caches + (size_t)id * 1024);
#pragma unroll
    for (int k = 0; k < 8; k++)
        reinterpret_cast<uint4 *>(cache)[32 * k + lane] = fresh ? make_uint4(0, 0, 0, 0) : resident[32 * k + lane];
    __syncwarp();
    SharedCache sc{cache, lane};
    rcore::BufferState st;
    st.next_j = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) st.stats[k] = 0;
    const uint32_t b = 2 * i + 1;
    const uint32_t n_out = replay_buffer<kEmit>(sc, st, records, tiles, n_tiles, b, check_crc, lane, p.out,
                                                kEmit ? p.offsets[i] : 0u, p.capacity, (uint64_t)b * kBufSamples);
    if (!kEmit) {
        if (lane == 0) p.n_deliv[i] = n_out;
        return;
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 8; k++) resident[32 * k + lane] = reinterpret_cast<const uint4 *>(cache)[32 * k + lane];
    if (lane == 0) {                                                   // p.stats is only 4-byte aligned
#pragma unroll
        for (int k = 0; k < 8; k++) p.stats[(size_t)i * 8 + k] = st.stats[k];
    }
}

}  // namespace

void launch_gpu_resolve(const GpuResolve &g, const modes_candidate *records, const modes_tile *tiles, uint32_t n_tiles,
                        uint32_t n_buffers, int check_crc, int sm_count, cudaStream_t stream) {
    const uint32_t init_threads = n_buffers * 1024u;
    resolve_init_kernel<<<(init_threads + 255) / 256, 256, 0, stream>>>(g, n_buffers);
    uint32_t grid = (n_buffers + kWarpsPerCta - 1) / kWarpsPerCta;
    if (grid > (uint32_t)sm_count * 4) grid = (uint32_t)sm_count * 4;
    for (int round = 0; round < kGpuResolveRounds; round++) {
        resolve_replay_kernel<false><<<grid, 32 * kWarpsPerCta, 0, stream>>>(g, records, tiles, n_tiles, n_buffers, check_crc);
        if (round == kGpuResolveRounds - 1) cudaMemsetAsync(g.flags, 0, sizeof(uint32_t), stream);   // flags[0] = pending after the LAST hand-over
        resolve_handover_kernel<<<8, 128, 0, stream>>>(g, n_buffers);
    }
    resolve_offsets_kernel<<<1, 1024, 0, stream>>>(g, n_buffers, g.capacity);
    resolve_replay_kernel<true><<<grid, 32 * kWarpsPerCta, 0, stream>>>(g, records, tiles, n_tiles, n_buffers, check_crc);
}

void launch_pool_resolve(const PoolResolve &p, const modes_candidate *records, const modes_tile *tiles, uint32_t n_tiles,
                         uint32_t n, int check_crc, cudaStream_t stream) {
    const uint32_t grid = (n + kWarpsPerCta - 1) / kWarpsPerCta;
    pool_resolve_kernel<false><<<grid, 32 * kWarpsPerCta, 0, stream>>>(p, records, tiles, n_tiles, n, check_crc);
    GpuResolve g{};                                                    // the fields resolve_offsets_kernel uses
    g.n_deliv = p.n_deliv; g.offsets = p.offsets; g.flags = p.flags;
    resolve_offsets_kernel<<<1, 1024, 0, stream>>>(g, n, p.capacity);
    pool_resolve_kernel<true><<<grid, 32 * kWarpsPerCta, 0, stream>>>(p, records, tiles, n_tiles, n, check_crc);
}

}  // namespace modes
