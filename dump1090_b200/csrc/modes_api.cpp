// modes_api.cpp — the C ABI declared in include/modes_b200.h: context, device
// workspaces, the two-slot host->device pipeline, and glue to the kernels
// (modes_kernels.cu) and the sequential resolve (modes_resolve.cpp).
//
// No CPU fallback: every entry point that computes runs the CUDA kernels, and
// modes_create() fails when no device is usable.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <new>
#include <string>
#include <vector>
#include "modes_internal.h"

using namespace modes;

namespace {

thread_local std::string g_create_error;

struct Slot {
    cudaStream_t stream = nullptr;
    uint8_t *d_iq = nullptr;         size_t iq_bytes = 0;
    uint8_t *d_halo = nullptr;
    uint32_t *d_cand_v = nullptr;    uint32_t cand_cap = 0;
    modes_candidate *d_records = nullptr;
    modes_tile *d_tiles = nullptr;   uint32_t tiles_cap = 0;
    uint32_t *d_counters = nullptr;
    // pinned carry blocks: a ring, because modes_detect_device/_host return without waiting and the
    // next call must not rewrite a block whose host-to-device copy is still queued
    static constexpr int kHaloRing = 8;
    uint8_t *h_halo = nullptr;       // kHaloRing x kHaloAlloc
    cudaEvent_t halo_ev[kHaloRing] = {};
    unsigned halo_next = 0;
    uint32_t *h_counters = nullptr;  // pinned
    modes_candidate *h_records = nullptr; size_t h_records_cap = 0;   // pinned
    modes_tile *h_tiles = nullptr;   size_t h_tiles_cap = 0;          // pinned
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    // cfg.gpu_resolve: workspace of the device resolve, sized for gr_buffers buffers / gr.capacity deliveries
    GpuResolve gr{};
    size_t gr_buffers = 0;
    uint32_t *h_gr_flags = nullptr;       // pinned: flags[3] + pad, then stats[8] as u64, then the end cache [1024]
    modes_delivery *h_deliveries = nullptr; size_t h_deliveries_cap = 0;   // pinned
    // in-flight batch
    bool busy = false;
    size_t n_buffers = 0;
    int64_t buffer_base = 0;
    const void *batch_iq = nullptr;   // device address the batch was scanned from
    bool own_outputs = true;          // results in this slot's own buffers (growable)
    uint32_t want_cap = 0;            // grow the candidate buffers to at least this on the next ensure
    // where this batch's results live (own workspace unless the caller supplied memory)
    modes_candidate *out_records = nullptr;
    modes_tile *out_tiles = nullptr;
    uint32_t out_cap = 0;
};

}  // namespace

struct modes_ctx {
    modes_config cfg;
    int sm_count = 148;
    uint16_t *d_lutn = nullptr;
    uint16_t *d_lut_iq = nullptr;
    uint32_t *d_bit_syn = nullptr;
    uint32_t *d_fix_hash = nullptr;
    uint32_t *d_pair_hash = nullptr;
    DeviceTables tab{};
    Slot slot[2];
    Slot detect;                      // stage-level API workspace
    // cfg.n_gpus > 1: this context is the front of a multi-GPU decode and owns one single-GPU
    // context per device; it keeps the stream state, the resolve state and the outputs itself
    // cfg.gpu_resolve: the address cache lives on the device, handed from batch to batch
    uint32_t *d_cache[2] = {nullptr, nullptr};
    int cache_cur = 0;
    cudaEvent_t ev_resolved = nullptr;    // the last batch's device resolve has finished (its cache_out is valid)
    bool resolved_pending = false;
    // hex door staging (modes_decode_frames)
    uint8_t *d_frames = nullptr; modes_frame_eval *d_frame_evals = nullptr, *h_frame_evals = nullptr; size_t frames_cap = 0;
    std::vector<modes_ctx *> gpus;
    size_t group_n[2] = {0, 0};       // batches in flight per slot parity
    uint64_t last_detect_count = 0;
    // stream state
    uint8_t *pending = nullptr;       // pinned, one reference buffer
    size_t pending_len = 0;
    uint8_t carry[MODES_CARRY_BYTES];
    int64_t buffers_done = 0;
    bool finished = false;
    ResolveState rs;
    ResolveScratch *scratch = nullptr;
    MessageOut out;                       // modes_set_sink / modes_set_output
    cudaStream_t own_detect_stream = nullptr;
    std::string err;
    uint64_t launches = 0;
    // cfg.profile: ring of CUDA-event triplets, one per batch, recorded on the launching stream
    static constexpr int kProfRing = 512;
    cudaEvent_t prof_ev[kProfRing][3];
    bool prof_ready = false;
    uint64_t prof_head = 0, prof_tail = 0;   // batches recorded / batches already reported
};

namespace {

int fail(modes_ctx *ctx, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf; else g_create_error = buf;
    return -1;
}

#define CK(ctx, call)                                                                   \
    do {                                                                                \
        cudaError_t e_ = (call);                                                        \
        if (e_ != cudaSuccess)                                                          \
            return fail(ctx, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// How host threads wait for the GPU.  0 (default): the CUDA runtime's own choice, which spins on a
// many-core host — lowest latency, one core busy per waiting thread.  1: sleep until the GPU signals
// (events with cudaEventBlockingSync) — for hosts that run more ranks than they have cores to burn,
// e.g. eight one-GPU processes under a small cgroup CPU quota.  Process-wide; contexts pick it up
// when they are created.  MODES_HOST_WAIT=block sets the initial value.
std::atomic<int> g_host_wait{-1};

int host_wait_mode() {
    int m = g_host_wait.load(std::memory_order_relaxed);
    if (m < 0) {
        const char *e = std::getenv("MODES_HOST_WAIT");
        m = (e && (*e == 'b' || *e == 'B' || *e == '1')) ? 1 : 0;
        g_host_wait.store(m, std::memory_order_relaxed);
    }
    return m;
}

unsigned event_flags(bool timing) {
    return (timing ? 0u : (unsigned)cudaEventDisableTiming) | (host_wait_mode() ? (unsigned)cudaEventBlockingSync : 0u);
}

}  // namespace

// cudaStreamSynchronize, or its sleeping equivalent (the stream must belong to the current device).
cudaError_t modes::wait_stream(cudaStream_t st) {
    if (!host_wait_mode()) return cudaStreamSynchronize(st);
    static thread_local cudaEvent_t ev[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return cudaStreamSynchronize(st);
    if (!ev[dev] && cudaEventCreateWithFlags(&ev[dev], cudaEventDisableTiming | cudaEventBlockingSync) != cudaSuccess) {
        ev[dev] = nullptr;
        (void)cudaGetLastError();
        return cudaStreamSynchronize(st);
    }
    if (cudaEventRecord(ev[dev], st) != cudaSuccess) { (void)cudaGetLastError(); return cudaStreamSynchronize(st); }
    return cudaEventSynchronize(ev[dev]);
}

namespace {

uint32_t default_cand_capacity(uint64_t n_samples) {
    uint64_t c = n_samples / 64 + 4096;
    return c > 0xFFFFFFF0ull ? 0xFFFFFFF0u : (uint32_t)c;
}

int slot_init(modes_ctx *ctx, Slot &s) {
    CK(ctx, cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
    CK(ctx, cudaMalloc(&s.d_halo, kHaloAlloc));
    CK(ctx, cudaMalloc(&s.d_counters, 4 * sizeof(uint32_t)));
    CK(ctx, cudaMallocHost(&s.h_halo, (size_t)kHaloAlloc * Slot::kHaloRing));
    for (auto &e : s.halo_ev) CK(ctx, cudaEventCreateWithFlags(&e, event_flags(false)));
    CK(ctx, cudaMallocHost(&s.h_counters, 4 * sizeof(uint32_t)));
    for (auto &e : s.ev) CK(ctx, cudaEventCreateWithFlags(&e, event_flags(true)));
    return 0;
}

void slot_free(Slot &s) {
    if (s.stream) wait_stream(s.stream);
    cudaFree(s.d_iq); cudaFree(s.d_halo); cudaFree(s.d_cand_v); cudaFree(s.d_records);
    cudaFree(s.d_tiles); cudaFree(s.d_counters);
    cudaFreeHost(s.h_halo); cudaFreeHost(s.h_counters); cudaFreeHost(s.h_records); cudaFreeHost(s.h_tiles);
    cudaFree(s.gr.start); cudaFree(s.gr.end); cudaFree(s.gr.written); cudaFree(s.gr.readfirst); cudaFree(s.gr.rerun);
    cudaFree(s.gr.n_deliv); cudaFree(s.gr.offsets); cudaFree(s.gr.flags); cudaFree(s.gr.stats_out); cudaFree(s.gr.out);
    cudaFreeHost(s.h_gr_flags); cudaFreeHost(s.h_deliveries);
    for (auto &e : s.ev) if (e) cudaEventDestroy(e);
    for (auto &e : s.halo_ev) if (e) cudaEventDestroy(e);
    if (s.stream) cudaStreamDestroy(s.stream);
    s = Slot();
}

// Make sure the slot can hold a batch of n_samples (device staging only if need_iq).
int slot_ensure(modes_ctx *ctx, Slot &s, uint64_t n_samples, bool need_iq, bool need_records) {
    if (need_iq && s.iq_bytes < n_samples * 2) {
        cudaFree(s.d_iq); s.d_iq = nullptr; s.iq_bytes = 0;
        CK(ctx, cudaMalloc(&s.d_iq, n_samples * 2));
        s.iq_bytes = n_samples * 2;
    }
    uint32_t cap = default_cand_capacity(n_samples);
    if (cap < s.want_cap) cap = s.want_cap;
    if (s.cand_cap < cap) {
        cudaFree(s.d_cand_v); s.d_cand_v = nullptr;
        cudaFree(s.d_records); s.d_records = nullptr;
        s.cand_cap = 0;
        CK(ctx, cudaMalloc(&s.d_cand_v, (size_t)cap * sizeof(uint32_t)));
        s.cand_cap = cap;
    }
    if (need_records && !s.d_records) CK(ctx, cudaMalloc(&s.d_records, (size_t)s.cand_cap * sizeof(modes_candidate)));
    uint32_t nt = tiles_for(n_samples);
    if (s.tiles_cap < nt) {
        cudaFree(s.d_tiles); s.d_tiles = nullptr;
        CK(ctx, cudaMalloc(&s.d_tiles, (size_t)nt * sizeof(modes_tile)));
        s.tiles_cap = nt;
    }
    return 0;
}

int host_ensure(modes_ctx *ctx, Slot &s, size_t n_records, size_t n_tiles) {
    if (s.h_records_cap < n_records) {
        cudaFreeHost(s.h_records); s.h_records = nullptr; s.h_records_cap = 0;
        size_t cap = n_records + n_records / 2 + 1024;
        CK(ctx, cudaMallocHost(&s.h_records, cap * sizeof(modes_candidate)));
        s.h_records_cap = cap;
    }
    if (s.h_tiles_cap < n_tiles) {
        cudaFreeHost(s.h_tiles); s.h_tiles = nullptr; s.h_tiles_cap = 0;
        CK(ctx, cudaMallocHost(&s.h_tiles, n_tiles * sizeof(modes_tile)));
        s.h_tiles_cap = n_tiles;
    }
    return 0;
}

int launch_batch(modes_ctx *ctx, Slot &s);

// Workspace of the device resolve for the slot's current batch.
int gpu_resolve_ensure(modes_ctx *ctx, Slot &s) {
    const size_t nb = s.n_buffers;
    if (s.gr_buffers < nb) {
        cudaFree(s.gr.start); cudaFree(s.gr.end); cudaFree(s.gr.written); cudaFree(s.gr.readfirst); cudaFree(s.gr.rerun);
        cudaFree(s.gr.n_deliv); cudaFree(s.gr.offsets);
        s.gr.start = s.gr.end = s.gr.written = s.gr.readfirst = s.gr.rerun = s.gr.n_deliv = s.gr.offsets = nullptr;
        s.gr_buffers = 0;
        CK(ctx, cudaMalloc(&s.gr.start, nb * 4096)); CK(ctx, cudaMalloc(&s.gr.end, nb * 4096));
        CK(ctx, cudaMalloc(&s.gr.written, nb * 128)); CK(ctx, cudaMalloc(&s.gr.readfirst, nb * 128));
        CK(ctx, cudaMalloc(&s.gr.rerun, nb * 4)); CK(ctx, cudaMalloc(&s.gr.n_deliv, nb * 4)); CK(ctx, cudaMalloc(&s.gr.offsets, (nb + 1) * 4));
        s.gr_buffers = nb;
    }
    if (!s.gr.flags) {
        CK(ctx, cudaMalloc(&s.gr.flags, 4 * sizeof(uint32_t)));
        CK(ctx, cudaMalloc(&s.gr.stats_out, 8 * sizeof(uint64_t)));
        CK(ctx, cudaMallocHost(&s.h_gr_flags, (20 + 1024) * sizeof(uint32_t)));
    }
    if (s.gr.capacity < s.cand_cap) {                     // at most two deliveries per candidate; one per candidate is 2x the dense capture
        cudaFree(s.gr.out); s.gr.out = nullptr; s.gr.capacity = 0;
        CK(ctx, cudaMalloc(&s.gr.out, (size_t)s.cand_cap * sizeof(modes_delivery)));
        s.gr.capacity = s.cand_cap;
    }
    return 0;
}

// Queue one batch on the slot's stream: (optional H2D) + halo + scan + frame evaluation.
int submit(modes_ctx *ctx, Slot &s, const uint8_t *host_iq, const void *d_iq, size_t n_buffers,
           const uint8_t *carry476, modes_candidate *d_records_ext, uint32_t cap_ext, modes_tile *d_tiles_ext) {
    const uint64_t n_samples = (uint64_t)n_buffers * kBufSamples;
    if (n_samples + kHaloSamples >= (1ull << 32)) return fail(ctx, "batch too large: %zu buffers", n_buffers);
    // caller-supplied record buffers: the slot's own position list must hold as many candidates
    if (d_records_ext && cap_ext > s.want_cap) s.want_cap = cap_ext;
    if (slot_ensure(ctx, s, n_samples, host_iq != nullptr, d_records_ext == nullptr)) return -1;
    if (host_iq) {
        CK(ctx, cudaMemcpyAsync(s.d_iq, host_iq, n_samples * 2, cudaMemcpyHostToDevice, s.stream));
        d_iq = s.d_iq;
    }
    if ((reinterpret_cast<uintptr_t>(d_iq) & 15) != 0) return fail(ctx, "device I/Q pointer must be 16-byte aligned");
    const unsigned hi = s.halo_next++ % Slot::kHaloRing;
    uint8_t *h_halo = s.h_halo + (size_t)hi * kHaloAlloc;
    CK(ctx, cudaEventSynchronize(s.halo_ev[hi]));                         // its previous copy (8 submits ago) has left the host
    memset(h_halo, 127, kHaloAlloc);                                      // dump1090.c:344 no-signal
    if (carry476) memcpy(h_halo + (kHaloBytes - MODES_CARRY_BYTES), carry476, MODES_CARRY_BYTES);
    CK(ctx, cudaMemcpyAsync(s.d_halo, h_halo, kHaloAlloc, cudaMemcpyHostToDevice, s.stream));
    CK(ctx, cudaEventRecord(s.halo_ev[hi], s.stream));
    s.batch_iq = d_iq;
    s.n_buffers = n_buffers;
    s.own_outputs = d_records_ext == nullptr;
    s.out_records = d_records_ext ? d_records_ext : s.d_records;
    s.out_tiles = d_tiles_ext ? d_tiles_ext : s.d_tiles;
    s.out_cap = d_records_ext ? (cap_ext < s.cand_cap ? cap_ext : s.cand_cap) : s.cand_cap;
    return launch_batch(ctx, s);
}

// The two kernels over the slot's staged batch (also used to repeat a batch that overflowed).
int launch_batch(modes_ctx *ctx, Slot &s) {
    const uint64_t n_samples = (uint64_t)s.n_buffers * kBufSamples;
    CK(ctx, cudaMemsetAsync(s.d_counters, 0, 4 * sizeof(uint32_t), s.stream));
    BatchView in{static_cast<const uint8_t *>(s.batch_iq), s.d_halo, n_samples};
    ScanOutputs so{s.d_cand_v, s.out_cap, s.out_tiles, s.d_counters};

    cudaEvent_t *pe = nullptr;
    if (ctx->cfg.profile) {
        if (!ctx->prof_ready) {
            for (auto &trip : ctx->prof_ev) for (auto &e : trip) CK(ctx, cudaEventCreateWithFlags(&e, event_flags(true)));
            ctx->prof_ready = true;
        }
        if (ctx->prof_head - ctx->prof_tail >= (uint64_t)modes_ctx::kProfRing) ctx->prof_tail = ctx->prof_head - modes_ctx::kProfRing + 1;
        pe = ctx->prof_ev[ctx->prof_head % modes_ctx::kProfRing];
        ctx->prof_head++;
    }
    if (pe) CK(ctx, cudaEventRecord(pe[0], s.stream));
    launch_scan(in, ctx->tab, so, ctx->sm_count, s.stream);
    if (pe) CK(ctx, cudaEventRecord(pe[1], s.stream));
    launch_eval(in, ctx->tab, so, s.out_records, ctx->cfg.fix_errors, ctx->cfg.aggressive, ctx->sm_count, s.stream);
    if (pe) CK(ctx, cudaEventRecord(pe[2], s.stream));
    CK(ctx, cudaGetLastError());
    ctx->launches += 2;
    if (ctx->cfg.gpu_resolve && s.own_outputs && &s != &ctx->detect) {
        if (gpu_resolve_ensure(ctx, s)) return -1;
        // the address cache comes from the previous batch's resolve (other slot, other stream)
        if (ctx->resolved_pending) CK(ctx, cudaStreamWaitEvent(s.stream, ctx->ev_resolved, 0));
        s.gr.cache_in = ctx->d_cache[ctx->cache_cur];
        s.gr.cache_out = ctx->d_cache[ctx->cache_cur ^ 1];
        ctx->cache_cur ^= 1;
        launch_gpu_resolve(s.gr, s.out_records, s.out_tiles, tiles_for(n_samples), (uint32_t)s.n_buffers, ctx->cfg.check_crc,
                           ctx->sm_count, s.stream);
        CK(ctx, cudaGetLastError());
        ctx->launches += 3 + 2 * kGpuResolveRounds;
        CK(ctx, cudaEventRecord(ctx->ev_resolved, s.stream));
        ctx->resolved_pending = true;
        CK(ctx, cudaMemcpyAsync(s.h_gr_flags, s.gr.flags, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s.stream));
        CK(ctx, cudaMemcpyAsync(s.h_gr_flags + 4, s.gr.stats_out, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost, s.stream));
        CK(ctx, cudaMemcpyAsync(s.h_gr_flags + 20, s.gr.cache_out, 1024 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s.stream));
    }
    CK(ctx, cudaMemcpyAsync(s.h_counters, s.d_counters, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s.stream));
    CK(ctx, cudaEventRecord(s.ev[3], s.stream));
    s.busy = true;
    return 0;
}

// Wait for the slot's batch; returns the number of candidates stored.  A batch denser than the
// candidate buffers (default: one candidate per 64 samples) is repeated with larger buffers when
// they are the slot's own; caller-supplied buffers cannot grow and report the overflow.
int wait_batch(modes_ctx *ctx, Slot &s, uint64_t *n_out) {
    for (;;) {
        CK(ctx, cudaEventSynchronize(s.ev[3]));
        if (!s.h_counters[1] && s.h_counters[0] <= s.out_cap) break;
        if (ctx->cfg.gpu_resolve && &s != &ctx->detect) break;           // reported by collect(): the device resolve ran on a truncated list
        const uint32_t found = s.h_counters[0];
        if (!s.own_outputs)
            return fail(ctx, "candidate capacity exceeded: %u found, room for %u", found, s.out_cap);
        s.want_cap = found + found / 8 + 1024;
        if (slot_ensure(ctx, s, (uint64_t)s.n_buffers * kBufSamples, false, true)) return -1;
        s.out_records = s.d_records;
        s.out_cap = s.cand_cap;
        if (launch_batch(ctx, s)) return -1;
    }
    *n_out = s.h_counters[0];
    return 0;
}

// Fetch the slot's results to pinned host memory and run the sequential resolve.
double now_ms() {
    timespec t; clock_gettime(CLOCK_MONOTONIC, &t);
    return t.tv_sec * 1e3 + t.tv_nsec * 1e-6;
}

int collect(modes_ctx *ctx, Slot &s) {
    if (!s.busy) return 0;
    s.busy = false;
    uint64_t n = 0;
    const bool dbg = getenv("MODES_DEBUG_TIMING") != nullptr;
    const double t0 = dbg ? now_ms() : 0;
    if (wait_batch(ctx, s, &n)) return -1;
    s.busy = false;                                     // a repeated (overflowed) batch re-arms the flag
    const double t1 = dbg ? now_ms() : 0;
    if (ctx->cfg.gpu_resolve) {
        // the verdicts were taken on the device: fetch the deliveries, build the structs
        if (s.h_counters[1] || s.h_counters[0] > s.out_cap) return fail(ctx, "gpu_resolve: candidate capacity exceeded (%u found)", s.h_counters[0]);
        if (s.h_gr_flags[0]) return fail(ctx, "gpu_resolve: address caches did not settle in %d rounds", kGpuResolveRounds);
        if (s.h_gr_flags[1]) return fail(ctx, "gpu_resolve: delivery capacity exceeded (%u messages)", s.h_gr_flags[2]);
        const size_t nd = s.h_gr_flags[2];
        if (s.h_deliveries_cap < nd) {
            cudaFreeHost(s.h_deliveries); s.h_deliveries = nullptr; s.h_deliveries_cap = 0;
            const size_t cap = nd + nd / 2 + 1024;
            CK(ctx, cudaMallocHost(&s.h_deliveries, cap * sizeof(modes_delivery)));
            s.h_deliveries_cap = cap;
        }
        if (nd) CK(ctx, cudaMemcpyAsync(s.h_deliveries, s.gr.out, nd * sizeof(modes_delivery), cudaMemcpyDeviceToHost, s.stream));
        CK(ctx, wait_stream(s.stream));
        uint64_t st8[8];
        memcpy(st8, s.h_gr_flags + 4, sizeof(st8));
        for (int i = 0; i < 8; i++) ctx->rs.stats[i] += (int64_t)st8[i];
        memcpy(ctx->rs.icao, s.h_gr_flags + 20, sizeof(ctx->rs.icao));    // host copy for the hex door / a later host resolve
        deliver_gpu(s.h_deliveries, nd, s.buffer_base, ctx->out);
        return 0;
    }
    const size_t nt = tiles_for((uint64_t)s.n_buffers * kBufSamples);
    if (host_ensure(ctx, s, n, nt)) return -1;
    if (n) CK(ctx, cudaMemcpyAsync(s.h_records, s.out_records, n * sizeof(modes_candidate), cudaMemcpyDeviceToHost, s.stream));
    CK(ctx, cudaMemcpyAsync(s.h_tiles, s.out_tiles, nt * sizeof(modes_tile), cudaMemcpyDeviceToHost, s.stream));
    CK(ctx, wait_stream(s.stream));
    const double t2 = dbg ? now_ms() : 0;
    ResolveConfig rc{ctx->cfg.fix_errors, ctx->cfg.aggressive, ctx->cfg.check_crc};
    resolve_candidates(ctx->rs, rc, s.h_records, s.h_tiles, nt, s.buffer_base, ctx->out, ctx->scratch);
    if (dbg) fprintf(stderr, "[collect] %zu buffers, %llu cands: wait %.3f ms, d2h %.3f ms, resolve %.3f ms (t=%.3f)\n",
                     s.n_buffers, (unsigned long long)n, t1 - t0, t2 - t1, now_ms() - t2, now_ms());
    return 0;
}

// Multi-GPU: wait for the group of batches in slot `parity` (one per GPU), bring their records to
// the host over every GPU's own link at once, and resolve the group exactly, shards in parallel.
int collect_group(modes_ctx *ctx, int parity) {
    const size_t n = ctx->group_n[parity];
    if (!n) return 0;
    ctx->group_n[parity] = 0;
    std::vector<const modes_candidate *> cands(n);
    std::vector<const modes_tile *> tiles(n);
    std::vector<size_t> n_tiles(n);
    std::vector<int64_t> base(n);
    for (size_t k = 0; k < n; k++) {
        modes_ctx *g = ctx->gpus[k];
        Slot &s = g->slot[parity];
        CK(ctx, cudaSetDevice(g->cfg.device));
        uint64_t nc = 0;
        s.busy = false;
        if (wait_batch(g, s, &nc)) return fail(ctx, "GPU %d: %s", g->cfg.device, g->err.c_str());
        s.busy = false;
        n_tiles[k] = tiles_for((uint64_t)s.n_buffers * kBufSamples);
        if (host_ensure(g, s, nc, n_tiles[k])) return fail(ctx, "GPU %d: %s", g->cfg.device, g->err.c_str());
        if (nc) CK(ctx, cudaMemcpyAsync(s.h_records, s.out_records, nc * sizeof(modes_candidate), cudaMemcpyDeviceToHost, s.stream));
        CK(ctx, cudaMemcpyAsync(s.h_tiles, s.out_tiles, n_tiles[k] * sizeof(modes_tile), cudaMemcpyDeviceToHost, s.stream));
        cands[k] = s.h_records; tiles[k] = s.h_tiles; base[k] = s.buffer_base;
    }
    for (size_t k = 0; k < n; k++) {
        CK(ctx, cudaSetDevice(ctx->gpus[k]->cfg.device));
        CK(ctx, wait_stream(ctx->gpus[k]->slot[parity].stream));
    }
    ResolveConfig rc{ctx->cfg.fix_errors, ctx->cfg.aggressive, ctx->cfg.check_crc};
    resolve_shards(ctx->rs, rc, n, cands.data(), tiles.data(), n_tiles.data(), base.data(), ctx->out, ctx->scratch);
    return 0;
}

// Multi-GPU streaming decode: batches of whole buffers dealt round-robin to the GPUs, one group of
// gpus.size() batches in flight per slot parity; group g-1 is resolved while group g uploads and runs.
int run_buffers_multi(modes_ctx *ctx, const uint8_t *host_iq, size_t n_buffers) {
    size_t max_b = (size_t)(ctx->cfg.max_batch_bytes / MODES_BUFFER_BYTES);
    if (max_b < 1) max_b = 1;
    int cur = 0;
    bool have_prev = false;
    while (n_buffers) {
        size_t k = 0;
        for (; k < ctx->gpus.size() && n_buffers; k++) {
            // an even share of what is left, so that a short call still uses every GPU
            size_t nb = (n_buffers + (ctx->gpus.size() - k) - 1) / (ctx->gpus.size() - k);
            if (nb > max_b) nb = max_b;
            modes_ctx *g = ctx->gpus[k];
            Slot &s = g->slot[cur];
            CK(ctx, cudaSetDevice(g->cfg.device));
            s.buffer_base = ctx->buffers_done;
            if (submit(g, s, host_iq, nullptr, nb, ctx->carry, nullptr, 0, nullptr)) return fail(ctx, "GPU %d: %s", g->cfg.device, g->err.c_str());
            memcpy(ctx->carry, host_iq + nb * MODES_BUFFER_BYTES - MODES_CARRY_BYTES, MODES_CARRY_BYTES);
            ctx->buffers_done += (int64_t)nb;
            host_iq += nb * MODES_BUFFER_BYTES;
            n_buffers -= nb;
            ctx->launches += 2;
        }
        ctx->group_n[cur] = k;
        if (have_prev && collect_group(ctx, cur ^ 1)) return -1;
        have_prev = true;
        cur ^= 1;
    }
    if (collect_group(ctx, cur ^ 1)) return -1;
    return cudaSetDevice(ctx->cfg.device) == cudaSuccess ? 0 : fail(ctx, "cudaSetDevice failed");
}

// Decode n_buffers whole reference buffers that sit in host memory.
int run_buffers(modes_ctx *ctx, const uint8_t *host_iq, size_t n_buffers) {
    if (!ctx->gpus.empty()) return run_buffers_multi(ctx, host_iq, n_buffers);
    size_t max_b = (size_t)(ctx->cfg.max_batch_bytes / MODES_BUFFER_BYTES);
    if (max_b < 1) max_b = 1;
    int cur = 0;
    constexpr size_t kTaperFloor = 16;                   // buffers (4 MiB)
    while (n_buffers) {
        size_t nb = n_buffers < max_b ? n_buffers : max_b;
        // The last batches of a call halve in size: what remains to be done after the final upload
        // (its kernels, record download and resolve) then belongs to a small batch, not a full one.
        if (n_buffers <= max_b && n_buffers > kTaperFloor) nb = (n_buffers + 1) / 2;
        Slot &s = ctx->slot[cur];
        if (collect(ctx, s)) return -1;                                  // slot may still hold batch b-2
        s.buffer_base = ctx->buffers_done;
        if (submit(ctx, s, host_iq, nullptr, nb, ctx->carry, nullptr, 0, nullptr)) return -1;
        memcpy(ctx->carry, host_iq + nb * MODES_BUFFER_BYTES - MODES_CARRY_BYTES, MODES_CARRY_BYTES);
        ctx->buffers_done += (int64_t)nb;
        host_iq += nb * MODES_BUFFER_BYTES;
        n_buffers -= nb;
        cur ^= 1;
        if (collect(ctx, ctx->slot[cur])) return -1;                     // resolve batch b-1 while b runs
    }
    if (collect(ctx, ctx->slot[cur])) return -1;
    if (collect(ctx, ctx->slot[cur ^ 1])) return -1;
    return 0;
}

}  // namespace

void modes::detect_results(const modes_ctx *ctx, const modes_candidate **records, const modes_tile **tiles, uint32_t *n_tiles) {
    const Slot &s = ctx->detect;
    *records = s.out_records;
    *tiles = s.out_tiles;
    *n_tiles = tiles_for((uint64_t)s.n_buffers * kBufSamples);
}

// ------------------------------------------------------------------- C ABI

extern "C" {

int modes_abi_version(void) { return MODES_B200_ABI_VERSION; }

void modes_default_config(modes_config *cfg) {
    memset(cfg, 0, sizeof(*cfg));
    cfg->fix_errors = 1;
    cfg->aggressive = 0;
    cfg->check_crc = 1;
    cfg->drop_eof_buffer = 0;
    cfg->device = 0;
    cfg->profile = 0;
    cfg->max_batch_bytes = 64ull << 20;
    cfg->n_gpus = 1;
}

const char *modes_last_error(const modes_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

void modes_destroy(modes_ctx *ctx) {
    if (!ctx) return;
    for (modes_ctx *g : ctx->gpus) modes_destroy(g);
    ctx->gpus.clear();
    cudaSetDevice(ctx->cfg.device);
    if (ctx->own_detect_stream) { wait_stream(ctx->detect.stream); ctx->detect.stream = ctx->own_detect_stream; }
    slot_free(ctx->slot[0]); slot_free(ctx->slot[1]); slot_free(ctx->detect);
    cudaFree(ctx->d_lutn); cudaFree(ctx->d_lut_iq); cudaFree(ctx->d_bit_syn); cudaFree(ctx->d_fix_hash); cudaFree(ctx->d_pair_hash);
    cudaFree(ctx->d_frames); cudaFree(ctx->d_frame_evals); cudaFreeHost(ctx->h_frame_evals);
    cudaFree(ctx->d_cache[0]); cudaFree(ctx->d_cache[1]);
    if (ctx->ev_resolved) cudaEventDestroy(ctx->ev_resolved);
    if (ctx->prof_ready) for (auto &trip : ctx->prof_ev) for (auto &e : trip) cudaEventDestroy(e);
    cudaFreeHost(ctx->pending);
    scratch_destroy(ctx->scratch);
    delete ctx;
}

static int create_impl(modes_ctx *ctx) {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, "no CUDA device available (%s); this library has no CPU path",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (ctx->cfg.device < 0 || ctx->cfg.device >= ndev) return fail(nullptr, "device %d out of range", ctx->cfg.device);
    CK(nullptr, cudaSetDevice(ctx->cfg.device));
    cudaDeviceProp prop;
    CK(nullptr, cudaGetDeviceProperties(&prop, ctx->cfg.device));
    if (prop.major < 10) return fail(nullptr, "device %d is sm_%d%d; kernels are built for sm_100a only", ctx->cfg.device, prop.major, prop.minor);
    ctx->sm_count = prop.multiProcessorCount;
    ctx->scratch = scratch_create();
    if (!ctx->scratch) return fail(nullptr, "out of memory");

    std::vector<uint16_t> lutn(kNLutEntries);
    uint32_t syn[112], hash[kFixHashSlots];
    build_lutn(lutn.data());
    std::vector<uint16_t> lut_iq(kLutIqEntries);
    build_lut_iq(lut_iq.data());
    build_bit_syndromes(syn);
    if (!build_fix_hash(syn, hash)) return fail(nullptr, "internal: syndrome hash construction failed");
    CK(nullptr, cudaMalloc(&ctx->d_lutn, kNLutEntries * sizeof(uint16_t)));
    CK(nullptr, cudaMalloc(&ctx->d_lut_iq, kLutIqEntries * sizeof(uint16_t)));
    CK(nullptr, cudaMemcpy(ctx->d_lut_iq, lut_iq.data(), kLutIqEntries * sizeof(uint16_t), cudaMemcpyHostToDevice));
    CK(nullptr, cudaMalloc(&ctx->d_bit_syn, sizeof(syn)));
    CK(nullptr, cudaMalloc(&ctx->d_fix_hash, sizeof(hash)));
    CK(nullptr, cudaMemcpy(ctx->d_lutn, lutn.data(), kNLutEntries * sizeof(uint16_t), cudaMemcpyHostToDevice));
    CK(nullptr, cudaMemcpy(ctx->d_bit_syn, syn, sizeof(syn), cudaMemcpyHostToDevice));
    CK(nullptr, cudaMemcpy(ctx->d_fix_hash, hash, sizeof(hash), cudaMemcpyHostToDevice));
    std::vector<uint32_t> pair(kPairHashSlots);
    if (!build_pair_hash(syn, pair.data())) return fail(nullptr, "internal: two-bit syndrome table construction failed");
    CK(nullptr, cudaMalloc(&ctx->d_pair_hash, pair.size() * sizeof(uint32_t)));
    CK(nullptr, cudaMemcpy(ctx->d_pair_hash, pair.data(), pair.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    ctx->tab = DeviceTables{ctx->d_lutn, ctx->d_lut_iq, ctx->d_bit_syn, ctx->d_fix_hash, ctx->d_pair_hash};
    CK(nullptr, cudaMallocHost(&ctx->pending, MODES_BUFFER_BYTES));
    if (ctx->cfg.gpu_resolve) {
        if (ctx->cfg.n_gpus > 1) return fail(nullptr, "gpu_resolve and n_gpus > 1 cannot be combined");
        for (auto &c : ctx->d_cache) { CK(nullptr, cudaMalloc(&c, 4096)); CK(nullptr, cudaMemset(c, 0, 4096)); }
        CK(nullptr, cudaEventCreateWithFlags(&ctx->ev_resolved, cudaEventDisableTiming));
    }
    for (Slot *s : {&ctx->slot[0], &ctx->slot[1], &ctx->detect})
        if (slot_init(ctx, *s)) { g_create_error = ctx->err; return -1; }
    return 0;
}

modes_ctx *modes_create(const modes_config *cfg) {
    modes_ctx *ctx = new (std::nothrow) modes_ctx();
    if (!ctx) { g_create_error = "out of memory"; return nullptr; }
    if (cfg) ctx->cfg = *cfg; else modes_default_config(&ctx->cfg);
    if (ctx->cfg.max_batch_bytes == 0) ctx->cfg.max_batch_bytes = 64ull << 20;
    ctx->rs.reset();
    memset(ctx->carry, 127, sizeof(ctx->carry));
    if (create_impl(ctx)) { modes_destroy(ctx); return nullptr; }
    if (ctx->cfg.n_gpus > 1) {
        int ndev = 0;
        cudaGetDeviceCount(&ndev);
        for (int k = 0; k < ctx->cfg.n_gpus; k++) {
            modes_config c = ctx->cfg;
            c.n_gpus = 1;
            c.profile = 0;
            c.device = (ctx->cfg.device + k) % (ndev > 0 ? ndev : 1);   // fewer devices than shards: reuse them round-robin
            modes_ctx *g = modes_create(&c);
            if (!g) { modes_destroy(ctx); return nullptr; }               // g_create_error holds the reason
            ctx->gpus.push_back(g);
        }
        cudaSetDevice(ctx->cfg.device);
    }
    return ctx;
}

int modes_set_sink(modes_ctx *ctx, modes_sink_fn fn, void *user) {
    if (!ctx) return -1;
    ctx->out.sink = fn; ctx->out.user = user;
    return 0;
}

int modes_set_output(modes_ctx *ctx, modes_message *out, size_t capacity) {
    if (!ctx) return -1;
    ctx->out.array = capacity ? out : nullptr;
    ctx->out.capacity = out ? capacity : 0;
    ctx->out.count = 0;
    return 0;
}

size_t modes_output_count(const modes_ctx *ctx) { return ctx ? ctx->out.count : 0; }

int modes_set_stream(modes_ctx *ctx, void *cuda_stream) {
    if (!ctx) return -1;
    if (ctx->detect.busy) wait_stream(ctx->detect.stream);
    if (!ctx->own_detect_stream) ctx->own_detect_stream = ctx->detect.stream;
    ctx->detect.stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->own_detect_stream;
    return 0;
}

int modes_reset(modes_ctx *ctx) {
    if (!ctx) return -1;
    ctx->rs.reset();
    if (ctx->cfg.gpu_resolve) {
        cudaSetDevice(ctx->cfg.device);
        cudaDeviceSynchronize();
        for (auto &c : ctx->d_cache) cudaMemset(c, 0, 4096);
        ctx->resolved_pending = false;
    }
    ctx->pending_len = 0;
    ctx->buffers_done = 0;
    ctx->finished = false;
    memset(ctx->carry, 127, sizeof(ctx->carry));
    return 0;
}

int modes_process(modes_ctx *ctx, const uint8_t *iq, size_t nbytes) {
    if (!ctx) return -1;
    if (ctx->finished) return fail(ctx, "modes_process after modes_finish; call modes_reset first");
    CK(ctx, cudaSetDevice(ctx->cfg.device));
    if (ctx->pending_len) {
        size_t take = MODES_BUFFER_BYTES - ctx->pending_len;
        if (take > nbytes) take = nbytes;
        memcpy(ctx->pending + ctx->pending_len, iq, take);
        ctx->pending_len += take; iq += take; nbytes -= take;
        if (ctx->pending_len < MODES_BUFFER_BYTES) return 0;
        if (run_buffers(ctx, ctx->pending, 1)) return -1;
        ctx->pending_len = 0;
    }
    size_t whole = nbytes / MODES_BUFFER_BYTES;
    if (whole && run_buffers(ctx, iq, whole)) return -1;
    iq += whole * MODES_BUFFER_BYTES; nbytes -= whole * MODES_BUFFER_BYTES;
    if (nbytes) { memcpy(ctx->pending, iq, nbytes); ctx->pending_len = nbytes; }
    return 0;
}

int modes_finish(modes_ctx *ctx) {
    if (!ctx) return -1;
    if (ctx->finished) return 0;
    CK(ctx, cudaSetDevice(ctx->cfg.device));
    ctx->finished = true;
    // The read that hits EOF still hands a 127-padded buffer to the decoder (dump1090.c:496-510);
    // whether it is decoded is the reference's race, made a switch here.
    memset(ctx->pending + ctx->pending_len, 127, MODES_BUFFER_BYTES - ctx->pending_len);
    ctx->pending_len = 0;
    if (ctx->cfg.drop_eof_buffer) return 0;
    return run_buffers(ctx, ctx->pending, 1);
}

int modes_get_stats(const modes_ctx *ctx, modes_stats *out) {
    if (!ctx || !out) return -1;
    memcpy(out->v, ctx->rs.stats, sizeof(out->v));
    return 0;
}

int modes_compute_magnitude(modes_ctx *ctx, const uint8_t *iq, size_t nsamples, uint16_t *mag) {
    if (!ctx) return -1;
    if (!nsamples) return 0;
    CK(ctx, cudaSetDevice(ctx->cfg.device));
    uint8_t *d_iq = nullptr; uint16_t *d_mag = nullptr;
    cudaStream_t st = ctx->detect.stream;
    cudaError_t e = cudaMalloc(&d_iq, nsamples * 2);
    if (e == cudaSuccess) e = cudaMalloc(&d_mag, nsamples * 2);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_iq, iq, nsamples * 2, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
        launch_magnitude(d_iq, d_mag, nsamples, ctx->d_lutn, st);
        ctx->launches++;
        e = cudaMemcpyAsync(mag, d_mag, nsamples * 2, cudaMemcpyDeviceToHost, st);
    }
    if (e == cudaSuccess) e = wait_stream(st);
    cudaFree(d_iq); cudaFree(d_mag);
    if (e != cudaSuccess) return fail(ctx, "magnitude kernel failed: %s", cudaGetErrorString(e));
    return 0;
}

int modes_detect_device(modes_ctx *ctx, const void *d_iq, size_t n_buffers, const uint8_t *carry476,
                        void *d_candidates, size_t cand_capacity, void *d_tiles) {
    if (!ctx) return -1;
    if (!d_iq || !n_buffers) return fail(ctx, "modes_detect_device: empty input");
    CK(ctx, cudaSetDevice(ctx->cfg.device));
    uint32_t cap = cand_capacity > 0xFFFFFFF0ull ? 0xFFFFFFF0u : (uint32_t)cand_capacity;
    return submit(ctx, ctx->detect, nullptr, d_iq, n_buffers, carry476,
                  static_cast<modes_candidate *>(d_candidates), cap, static_cast<modes_tile *>(d_tiles));
}

int modes_detect_host(modes_ctx *ctx, const uint8_t *iq, size_t n_buffers, const uint8_t *carry476,
                      void *d_candidates, size_t cand_capacity, void *d_tiles) {
    if (!ctx) return -1;
    if (!iq || !n_buffers) return fail(ctx, "modes_detect_host: empty input");
    CK(ctx, cudaSetDevice(ctx->cfg.device));
    uint32_t cap = cand_capacity > 0xFFFFFFF0ull ? 0xFFFFFFF0u : (uint32_t)cand_capacity;
    return submit(ctx, ctx->detect, iq, nullptr, n_buffers, carry476,
                  static_cast<modes_candidate *>(d_candidates), cap, static_cast<modes_tile *>(d_tiles));
}

int modes_detect_wait(modes_ctx *ctx, uint64_t *n_candidates) {
    if (!ctx) return -1;
    if (!ctx->detect.busy) return fail(ctx, "modes_detect_wait without modes_detect_device");
    uint64_t n = 0;
    if (wait_batch(ctx, ctx->detect, &n)) return -1;
    ctx->last_detect_count = n;
    if (n_candidates) *n_candidates = n;
    return 0;
}

int modes_detect_fetch(modes_ctx *ctx, modes_candidate *candidates, modes_tile *tiles) {
    if (!ctx) return -1;
    Slot &s = ctx->detect;
    if (!s.busy) return fail(ctx, "modes_detect_fetch without modes_detect_device");
    uint64_t n = 0;
    if (wait_batch(ctx, s, &n)) return -1;
    const size_t nt = tiles_for((uint64_t)s.n_buffers * kBufSamples);
    if (n && candidates)
        CK(ctx, cudaMemcpyAsync(candidates, s.out_records, n * sizeof(modes_candidate), cudaMemcpyDeviceToHost, s.stream));
    if (tiles) CK(ctx, cudaMemcpyAsync(tiles, s.out_tiles, nt * sizeof(modes_tile), cudaMemcpyDeviceToHost, s.stream));
    CK(ctx, wait_stream(s.stream));
    return 0;
}

int modes_resolve(modes_ctx *ctx, const modes_candidate *candidates, const modes_tile *tiles, size_t n_tiles,
                  int64_t buffer_base) {
    if (!ctx || !tiles) return -1;
    ResolveConfig rc{ctx->cfg.fix_errors, ctx->cfg.aggressive, ctx->cfg.check_crc};
    resolve_candidates(ctx->rs, rc, candidates, tiles, n_tiles, buffer_base, ctx->out, ctx->scratch);
    return 0;
}

struct modes_resolver {
    ResolveState rs; ResolveConfig rc; MessageOut out; ResolveScratch *scratch = nullptr;
    ResolveState tentative;             // end state of the last modes_resolver_run_tentative
    bool has_tentative = false;
};

modes_resolver *modes_resolver_create(const modes_config *cfg) {
    modes_resolver *r = new (std::nothrow) modes_resolver();
    if (!r) return nullptr;
    modes_config c;
    if (cfg) c = *cfg; else modes_default_config(&c);
    r->rc = ResolveConfig{c.fix_errors, c.aggressive, c.check_crc};
    r->rs.reset();
    r->scratch = scratch_create();
    if (!r->scratch) { delete r; return nullptr; }
    return r;
}

void modes_resolver_destroy(modes_resolver *r) { if (r) { scratch_destroy(r->scratch); delete r; } }

int modes_resolver_run(modes_resolver *r, const modes_candidate *candidates, const modes_tile *tiles,
                       size_t n_tiles, int64_t buffer_base, modes_sink_fn sink, void *user) {
    if (!r || !tiles) return -1;
    r->out.sink = sink; r->out.user = user;
    resolve_candidates(r->rs, r->rc, candidates, tiles, n_tiles, buffer_base, r->out, r->scratch);
    return 0;
}

int modes_resolver_run_shards(modes_resolver *r, size_t n_shards, const modes_candidate *const *candidates,
                              const modes_tile *const *tiles, const size_t *n_tiles, const int64_t *buffer_base,
                              modes_sink_fn sink, void *user) {
    if (!r || (n_shards && (!candidates || !tiles || !n_tiles || !buffer_base))) return -1;
    r->out.sink = sink; r->out.user = user;
    resolve_shards(r->rs, r->rc, n_shards, candidates, tiles, n_tiles, buffer_base, r->out, r->scratch);
    return 0;
}

int modes_resolver_get_cache(const modes_resolver *r, uint32_t cache[MODES_ICAO_CACHE_SLOTS]) {
    if (!r || !cache) return -1;
    memcpy(cache, r->has_tentative ? r->tentative.icao : r->rs.icao, sizeof(r->rs.icao));
    return 0;
}

int modes_resolver_set_cache(modes_resolver *r, const uint32_t cache[MODES_ICAO_CACHE_SLOTS]) {
    if (!r) return -1;
    if (cache) memcpy(r->rs.icao, cache, sizeof(r->rs.icao)); else memset(r->rs.icao, 0, sizeof(r->rs.icao));
    r->rs.cur_buffer = -1; r->rs.next_j = 0;
    r->has_tentative = false;
    return 0;
}

int modes_resolver_tail_cache(const modes_resolver *r, const modes_candidate *candidates, const modes_tile *tiles,
                              size_t n_tiles, int64_t buffer_base, size_t n_tail_tiles, uint32_t cache[MODES_ICAO_CACHE_SLOTS]) {
    if (!r || !tiles || !cache) return -1;
    ResolveState st;
    st.reset();
    ResolveScratch *tmp = scratch_create();
    if (!tmp) return -1;
    if (n_tail_tiles > n_tiles) n_tail_tiles = n_tiles;
    resolve_tentative(st, r->rc, candidates, tiles + (n_tiles - n_tail_tiles), n_tail_tiles, buffer_base, tmp);
    scratch_destroy(tmp);
    memcpy(cache, st.icao, sizeof(st.icao));
    return 0;
}

int modes_resolver_run_tentative(modes_resolver *r, const modes_candidate *candidates, const modes_tile *tiles,
                                 size_t n_tiles, int64_t buffer_base) {
    if (!r || !tiles) return -1;
    r->tentative = r->rs;
    memset(r->tentative.stats, 0, sizeof(r->tentative.stats));
    r->tentative.cur_buffer = -1; r->tentative.next_j = 0;
    resolve_tentative(r->tentative, r->rc, candidates, tiles, n_tiles, buffer_base, r->scratch);
    r->has_tentative = true;
    return 0;
}

int modes_resolver_commit(modes_resolver *r, modes_sink_fn sink, void *user) {
    if (!r || !r->has_tentative) return -1;
    r->out.sink = sink; r->out.user = user;
    for (int i = 0; i < 8; i++) r->rs.stats[i] += r->tentative.stats[i];
    memcpy(r->rs.icao, r->tentative.icao, sizeof(r->rs.icao));
    r->rs.cur_buffer = r->tentative.cur_buffer; r->rs.next_j = r->tentative.next_j;
    resolve_commit(r->out, r->scratch);
    r->has_tentative = false;
    return 0;
}

int modes_resolver_set_output(modes_resolver *r, modes_message *out, size_t capacity) {
    if (!r) return -1;
    r->out.array = capacity ? out : nullptr;
    r->out.capacity = out ? capacity : 0;
    r->out.count = 0;
    return 0;
}

size_t modes_resolver_output_count(const modes_resolver *r) { return r ? r->out.count : 0; }

int modes_resolver_reset(modes_resolver *r) {
    if (!r) return -1;
    r->rs.reset();
    return 0;
}

int modes_resolver_stats(const modes_resolver *r, modes_stats *out) {
    if (!r || !out) return -1;
    memcpy(out->v, r->rs.stats, sizeof(out->v));
    return 0;
}

int modes_decode_frames(modes_ctx *ctx, const uint8_t *frames, size_t n, modes_message *out) {
    if (!ctx || (n && (!frames || !out))) return -1;
    if (!n) return 0;
    if (n > 0x7fffffffu) return fail(ctx, "too many frames");
    CK(ctx, cudaSetDevice(ctx->cfg.device));
    // persistent device / pinned staging, grown on demand (the hex door is called per line by a
    // network feeder: no allocation per call)
    if (ctx->frames_cap < n) {
        cudaFree(ctx->d_frames); cudaFree(ctx->d_frame_evals); cudaFreeHost(ctx->h_frame_evals);
    cudaFree(ctx->d_cache[0]); cudaFree(ctx->d_cache[1]);
    if (ctx->ev_resolved) cudaEventDestroy(ctx->ev_resolved);
        ctx->d_frames = nullptr; ctx->d_frame_evals = nullptr; ctx->h_frame_evals = nullptr; ctx->frames_cap = 0;
        const size_t cap = n < 64 ? 64 : n + n / 2;
        CK(ctx, cudaMalloc(&ctx->d_frames, cap * 14));
        CK(ctx, cudaMalloc(&ctx->d_frame_evals, cap * sizeof(modes_frame_eval)));
        CK(ctx, cudaMallocHost(&ctx->h_frame_evals, cap * sizeof(modes_frame_eval)));
        ctx->frames_cap = cap;
    }
    cudaStream_t st = ctx->detect.stream;
    CK(ctx, cudaMemcpyAsync(ctx->d_frames, frames, n * 14, cudaMemcpyHostToDevice, st));
    launch_eval_frames(ctx->d_frames, ctx->d_frame_evals, (uint32_t)n, ctx->tab, ctx->cfg.fix_errors, ctx->cfg.aggressive, st);
    ctx->launches++;
    CK(ctx, cudaMemcpyAsync(ctx->h_frame_evals, ctx->d_frame_evals, n * sizeof(modes_frame_eval), cudaMemcpyDeviceToHost, st));
    CK(ctx, wait_stream(st));
    for (size_t i = 0; i < n; i++) {                       // in order: the address cache is sequential
        finish_message(ctx->rs, ctx->h_frame_evals[i], &out[i]);
        out[i].sample_pos = -1;
    }
    return 0;
}

int modes_decode_frame(modes_ctx *ctx, const uint8_t msg[14], modes_message *out) {
    return modes_decode_frames(ctx, msg, 1, out);
}

void *modes_stream(modes_ctx *ctx) { return ctx ? (void *)ctx->detect.stream : nullptr; }

void *modes_device_alloc(size_t nbytes) {
    void *p = nullptr;
    if (cudaMalloc(&p, nbytes ? nbytes : 1) != cudaSuccess) return nullptr;
    return p;
}

void modes_device_free(void *p) { if (p) cudaFree(p); }

int modes_ipc_export(const void *dptr, uint8_t handle[64]) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
    cudaIpcMemHandle_t h;
    if (!dptr || cudaIpcGetMemHandle(&h, const_cast<void *>(dptr)) != cudaSuccess) return -1;
    memcpy(handle, &h, 64);
    return 0;
}

void *modes_ipc_open(const uint8_t handle[64]) {
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    void *p = nullptr;
    if (cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

int modes_ipc_close(void *mapped) { return mapped && cudaIpcCloseMemHandle(mapped) == cudaSuccess ? 0 : -1; }

int modes_copy_to_host(void *dst_host, const void *src_device, size_t nbytes) {
    // own non-blocking stream per calling thread: never serialises with the caller's other streams
    static thread_local cudaStream_t st = nullptr;
    static thread_local int st_dev = -1;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, src_device) != cudaSuccess) return -1;
    if (cudaSetDevice(at.device) != cudaSuccess) return -1;
    if (!st || st_dev != at.device) {
        if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) return -1;
        st_dev = at.device;
    }
    if (cudaMemcpyAsync(dst_host, src_device, nbytes, cudaMemcpyDeviceToHost, st) != cudaSuccess) return -1;
    return wait_stream(st) == cudaSuccess ? 0 : -1;
}

int modes_set_host_wait(int mode) {
    if (mode != 0 && mode != 1) return -1;
    g_host_wait.store(mode, std::memory_order_relaxed);
    return 0;
}

int modes_device_memset(void *dst_device, int value, size_t nbytes) {
    if (cudaMemset(dst_device, value, nbytes) != cudaSuccess) return -1;
    return cudaDeviceSynchronize() == cudaSuccess ? 0 : -1;
}

int modes_detect_publish_count(modes_ctx *ctx, void *dst) {
    if (!ctx || !dst) return -1;
    CK(ctx, cudaMemcpyAsync(dst, ctx->detect.d_counters, 4 * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->detect.stream));
    return 0;
}

void *modes_host_alloc(size_t nbytes) {
    void *p = nullptr;
    if (cudaMallocHost(&p, nbytes ? nbytes : 1) != cudaSuccess) return nullptr;
    return p;
}

void modes_host_free(void *p) { if (p) cudaFreeHost(p); }

int modes_get_kernel_times(modes_ctx *ctx, float ms[4]) {
    if (!ctx || !ms) return -1;
    ms[0] = ms[1] = ms[2] = ms[3] = 0.f;
    if (!ctx->prof_ready) return 0;
    double a = 0, b = 0, c = 0; int n = 0;
    for (; ctx->prof_tail < ctx->prof_head; ctx->prof_tail++) {
        cudaEvent_t *pe = ctx->prof_ev[ctx->prof_tail % modes_ctx::kProfRing];
        if (cudaEventSynchronize(pe[2]) != cudaSuccess) continue;
        float x = 0, y = 0, z = 0;
        cudaEventElapsedTime(&x, pe[0], pe[1]); cudaEventElapsedTime(&y, pe[1], pe[2]); cudaEventElapsedTime(&z, pe[0], pe[2]);
        a += x; b += y; c += z; n++;
    }
    if (n) { ms[0] = (float)(a / n); ms[1] = (float)(b / n); ms[2] = (float)(c / n); ms[3] = (float)n; }
    return 0;
}

uint64_t modes_launch_count(const modes_ctx *ctx) { return ctx ? ctx->launches : 0; }

size_t modes_tile_count(size_t n_buffers) { return tiles_for((uint64_t)n_buffers * kBufSamples); }

}  // extern "C"
