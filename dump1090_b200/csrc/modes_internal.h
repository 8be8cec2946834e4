// modes_internal.h — declarations shared by the CUDA kernels (modes_kernels.cu),
// the host resolve (modes_resolve.cpp), the C-ABI glue (modes_api.cpp) and the
// receiver pool (modes_pool.cpp).
// Product code; never includes anything from oracle/.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>
#include "modes_b200.h"

namespace modes {

// ---- geometry of the "virtual" sample array a batch is scanned over --------
// A batch is n_buffers whole reference buffers (131072 new samples each,
// dump1090.c:54) resident in HBM, preceded by the 238 samples the reference
// carries over from the previous buffer (dump1090.c:481).  The carry lives in
// a separate 480-byte device block (2 unused samples + 238 carry) so that the
// body keeps its 16-byte alignment:
//     virtual index v in [0, 240)      -> halo[v]
//     virtual index v in [240, 240+N)  -> body[v-240]
// The reference's buffer-relative position of v is t = v - 2 = 131072*k + j,
// and the scan visits j in [0, 131070) (dump1090.c:1593).
constexpr int      kHaloSamples  = 240;
constexpr int      kHaloBytes    = 480;
constexpr int      kHaloAlloc    = 512;                         // + 16 bytes of "no signal" (127) after the carry: kernels read it for out-of-range chunks
constexpr int      kTileSamples  = MODES_TILE_SAMPLES;          // one scan tile: 8 rows of 31 lanes x 32 positions (modes_scan2.cu)
constexpr uint32_t kBufSamples   = MODES_BUFFER_SAMPLES;
constexpr uint32_t kScanLimit    = kBufSamples - 2;             // j < 131070
constexpr int      kNLutEntries  = 32769;                       // magnitude by i*i+q*q
constexpr int      kFixHashSlots = 256;
constexpr int      kPairHashBits = 14;                          // == serial::kPairHashBits
constexpr int      kPairHashSlots = 1 << kPairHashBits;          // two-bit patterns: 5671 entries
constexpr int      kPairHashMaxProbe = 16;                      // checked at table construction
constexpr int      kLutIqStride  = 136;                         // == serial::kIqLutStride (modes_eval_serial.cuh)
constexpr int      kLutIqEntries = 129 * kLutIqStride;

struct DeviceTables {
    const uint16_t *lutn;        // [32769] round(sqrt(n)*360), dump1090.c:362 keyed by n=i*i+q*q
    const uint16_t *lut_iq;      // [129 x kLutIqStride] the same keyed by (|I-127|, |Q-127|); 16-byte aligned
    const uint32_t *bit_syn;     // [112] syndrome of a single flipped bit (dump1090.c:683-698 + parity bits)
    const uint32_t *fix_hash;    // [256] open-addressed inverse of bit_syn: (syndrome<<8 | pos), 0xFFFFFFFF empty
    const uint32_t *pair_hash;   // [16384] two flipped bits p < q: (syndrome<<7 | p), 0xFFFFFFFF empty
};

struct BatchView {
    const uint8_t *body;         // n_samples*2 bytes, 16-byte aligned
    const uint8_t *halo;         // kHaloBytes, 16-byte aligned
    uint64_t       n_samples;    // N = n_buffers * 131072
};

struct ScanOutputs {
    uint32_t   *cand_v;          // virtual positions of candidates, tile by tile
    uint32_t    cand_capacity;
    modes_tile *tiles;           // [n_tiles]
    uint32_t   *counters;        // [0] candidates found (may exceed capacity), [1] overflow flag, [2]/[3] scan tile / eval chunk hand-out
};

inline uint32_t tiles_for(uint64_t n_samples) {
    return (uint32_t)((n_samples + kHaloSamples + kTileSamples - 1) / kTileSamples);
}

// Kernel launchers (launch_scan: modes_scan2.cu; the rest: modes_kernels.cu).  All asynchronous on `stream`.
void launch_scan(const BatchView &in, const DeviceTables &tab, const ScanOutputs &out, int sm_count,
                 cudaStream_t stream);
void launch_eval(const BatchView &in, const DeviceTables &tab, const ScanOutputs &scan,
                 modes_candidate *records, int fix_errors, int aggressive, int sm_count,
                 cudaStream_t stream);
// The single-walk frame evaluation (modes_eval_fused.cu); parts = 1: whole windows staged, 2: half windows.
void launch_eval_fused(const BatchView &in, const DeviceTables &tab, const ScanOutputs &scan, modes_candidate *records,
                       int fix_errors, int aggressive, int sm_count, int parts, cudaStream_t stream);
void launch_magnitude(const uint8_t *d_iq, uint16_t *d_mag, uint64_t n_samples, const uint16_t *lutn,
                      cudaStream_t stream);
// CRC / fix on raw frame bytes (hex door): n frames of 14 bytes -> n modes_frame_eval.
void launch_eval_frames(const uint8_t *d_frames, modes_frame_eval *d_out, uint32_t n, const DeviceTables &tab,
                        int fix_errors, int aggressive, cudaStream_t stream);

// Host-side table construction (modes_tables.cpp).
void build_lutn(uint16_t *out /*[32769]*/);
void build_lut_iq(uint16_t *out /*[kLutIqEntries]*/);
void build_bit_syndromes(uint32_t *out /*[112]*/);
bool build_fix_hash(const uint32_t *bit_syn, uint32_t *out /*[256]*/);
bool build_pair_hash(const uint32_t *bit_syn, uint32_t *out /*[kPairHashSlots]*/);

// ---- device resolve (modes_resolve_gpu.cu) ----------------------------------
// One delivered message as the device resolve hands it over: position, the evaluated frame, and
// what the sequential half decided.  bits = crcok | phase_corrected << 8 | extra_is_ap << 16;
// extra = DF11 interrogator id, or the address recovered from an address/parity field.
struct modes_delivery { int64_t t; modes_frame_eval eval; uint32_t extra; uint32_t bits; };
static_assert(sizeof(modes_delivery) == 40, "delivery record layout");
constexpr int kGpuResolveRounds = 4;                 // replay + hand-over rounds before the emit pass (two suffice on real traffic)

struct GpuResolve {
    uint32_t *start, *end;       // [n_buffers][1024] address cache at the start / end of each buffer
    uint32_t *written, *readfirst;   // [n_buffers][32]  slots a buffer wrote / read before writing
    uint32_t *rerun, *n_deliv, *offsets;   // [n_buffers] (+1 for offsets)
    uint32_t *flags;             // [0] a buffer still needed another replay, [1] delivery capacity exceeded, [2] deliveries
    const uint32_t *cache_in;    // [1024] cache at the start of the batch
    uint32_t *cache_out;         // [1024] cache at its end
    uint64_t *stats_out;         // [8]
    modes_delivery *out;         // deliveries in stream order
    uint32_t capacity;           // entries of `out`
};
void launch_gpu_resolve(const GpuResolve &g, const modes_candidate *records, const modes_tile *tiles, uint32_t n_tiles,
                        uint32_t n_buffers, int check_crc, int sm_count, cudaStream_t stream);

// The device resolve of a receiver pool (modes_pool.cpp): a batch of n receivers laid out pad, data, pad,
// data, ...; list entry i owns data buffer 2i+1.  Every receiver's buffer is independent of the others
// (the skip state restarts at each buffer, and a receiver is listed once per batch), so one warp per
// entry replays from that receiver's resident cache and writes the cache back: no guessing, no hand-over.
struct PoolResolve {
    uint32_t *caches;            // [n_receivers][1024] resident address caches
    const uint32_t *ids;         // [n] receiver of entry i | kPoolFresh: start from an empty cache
    uint32_t *n_deliv;           // [n] deliveries of entry i, followed by
    uint32_t *stats;             //   [n][8] its statistics of this batch
    uint32_t *offsets;           // [n + 1]
    uint32_t *flags;             // [4] scratch of resolve_offsets_kernel
    modes_delivery *out;         // deliveries, entry by entry in list order, each in stream order; t = position
    uint32_t capacity;           //   inside the receiver's own buffer.  2 x the batch's candidates: cannot overflow
};
constexpr uint32_t kPoolFresh = 1u << 31;
void launch_pool_resolve(const PoolResolve &p, const modes_candidate *records, const modes_tile *tiles, uint32_t n_tiles,
                         uint32_t n, int check_crc, cudaStream_t stream);

// ---- sequential resolve (modes_resolve.cpp) --------------------------------
struct ResolveState {
    uint32_t icao[1024];         // dump1090.c:335: address per slot (TTL: never expires within a run)
    int64_t  stats[8];
    int64_t  cur_buffer;         // buffer whose skip state is live, -1 = none
    uint32_t next_j;             // first position not skipped in cur_buffer
    void reset();
};

struct ResolveConfig { int fix_errors, aggressive, check_crc; };

// Where delivered messages go: a callback, and/or a caller-owned array that is
// filled in place (count keeps running past capacity).
struct MessageOut {
    modes_sink_fn sink = nullptr; void *user = nullptr;
    modes_message *array = nullptr; size_t capacity = 0; size_t count = 0;
};

// Working memory of the resolve (verdict lists, per-shard runs), owned by a context / resolver and
// kept between calls: grown once, never handed back (re-faulting ~14 MB of verdicts per GiB in every
// call costs more than the verdicts themselves).
struct ResolveScratch;
ResolveScratch *scratch_create();
void scratch_destroy(ResolveScratch *s);

void resolve_candidates(ResolveState &st, const ResolveConfig &cfg, const modes_candidate *cands,
                        const modes_tile *tiles, size_t n_tiles, int64_t buffer_base, MessageOut &out,
                        ResolveScratch *scratch);
void resolve_shards(ResolveState &st, const ResolveConfig &cfg, size_t n_shards, const modes_candidate *const *cands,
                    const modes_tile *const *tiles, const size_t *n_tiles, const int64_t *buffer_base,
                    MessageOut &out, ResolveScratch *scratch);
// A shard resolved from a GUESSED address cache (one rank / one GPU thread of a sharded decode):
// verdicts only, deliveries held back in the scratch until the guess is verified.
void resolve_tentative(ResolveState &st, const ResolveConfig &cfg, const modes_candidate *cands, const modes_tile *tiles,
                       size_t n_tiles, int64_t buffer_base, ResolveScratch *scratch);
void resolve_commit(MessageOut &out, ResolveScratch *scratch);
// Messages from the device resolve's delivery records (structs built in parallel, sink called in order).
void deliver_gpu(const modes_delivery *d, size_t n, int64_t buffer_base, MessageOut &out);
// The order-dependent tail of decodeModesMessage + field decode for one evaluated frame.
int finish_message(ResolveState &st, const modes_frame_eval &p, modes_message *out);

// ---- C-ABI glue (modes_api.cpp) ----------------------------------------------
// Where the context's last modes_detect_device / _host left its results on the device (its own
// workspace; valid after modes_detect_wait until the next detect call), and its tile count.
void detect_results(const modes_ctx *ctx, const modes_candidate **records, const modes_tile **tiles, uint32_t *n_tiles);
// cudaStreamSynchronize, or its sleeping equivalent under modes_set_host_wait(1).
cudaError_t wait_stream(cudaStream_t st);

}  // namespace modes
