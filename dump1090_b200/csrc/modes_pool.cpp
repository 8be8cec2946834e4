// modes_pool.cpp — many receivers on one GPU: "batch across receivers instead of across time"
// (SURVEY.md §8(f) item 4).
//
// One dump1090 process serves one RTL-SDR: rtlsdrCallback (dump1090.c:442-456) hands it 131072
// samples at a time, each buffer is prefixed with the last 238 samples of the previous one (:481),
// and detectModeS keeps its ICAO address cache, skip state and statistics for that one stream.  A
// B200 decodes ~12 000 such 2 MHz streams in real time (the limit is the PCIe link), but a single
// stream only fills it with seconds of data at a time.  The pool takes ONE buffer from each of many
// receivers and decodes them in one batch, with everything per stream kept per receiver.
//
// The kernels are untouched: they see a batch as consecutive buffers of ONE stream, each buffer's
// carry being the tail of the buffer before it.  The batch is therefore laid out as pairs
//     [pad buffer of receiver i: no signal, its last 238 samples = receiver i's carry][receiver i's buffer]
// resident in HBM (twice: two batches may be in flight, one being uploaded and scanned while the one
// before it is resolved); per call only the data buffers and the 476-byte carries cross PCIe.  A position
// of a data buffer never looks beyond that buffer and its 238 carried samples (dump1090.c:1593:
// j < 131070, window j..j+239 of a 131310-sample array), so its candidates are exactly those of the
// receiver's own stream; whatever the scan finds inside the pad buffers is dropped.  The price is a
// second scan over constant buffers (the scan runs at 2 T samples/s; the link delivers 25 G samples/s).
//
// The order-dependent half (cfg.gpu_resolve = 0) is the existing host resolver, one per receiver: the
// records of a data buffer are re-based to that receiver's own stream position and replayed with its
// own address cache.  With cfg.gpu_resolve = 1 the same replay runs on the device at collect, one warp
// per receiver, each receiver's address cache resident in HBM between batches (launch_pool_resolve,
// modes_resolve_gpu.cu); only the 40-byte records of the delivered messages and 36 bytes of counts and
// statistics per receiver cross PCIe, and the host builds the structs.  Within a batch no receiver's
// buffer depends on another's, so unlike the single-stream device resolve there is nothing to guess.
// The detection runs through the public C ABI (modes_detect_device / _wait / _fetch); the host resolve
// through modes_resolver_*; the device resolve reads the records where modes_detect_device left them
// (modes::detect_results) and builds structs with modes::deliver_gpu.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <condition_variable>
#include <cstdlib>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>
#include <cuda_runtime.h>
#include "modes_b200.h"
#include "modes_internal.h"

namespace {

constexpr size_t kBuf = MODES_BUFFER_BYTES;
constexpr int64_t kBufSamples = MODES_BUFFER_SAMPLES;

struct Receiver {
    modes_resolver *res = nullptr;
    int64_t buffers = 0;                       // buffers of this receiver decoded so far
    uint8_t carry[MODES_CARRY_BYTES];
    // cfg.gpu_resolve: the statistics so far, and whether its resident cache is to be ignored (reset)
    int64_t stats[8] = {};
    bool fresh = true;
};

// A few persistent helper threads: run(n, f) executes f(0..n-1), f(0) on the calling thread.
class Crew {
public:
    explicit Crew(size_t helpers) {
        for (size_t w = 0; w < helpers; w++) threads_.emplace_back([this, w] { loop(w + 1); });
    }
    ~Crew() {
        { std::lock_guard<std::mutex> g(m_); stop_ = true; gen_++; }
        cv_.notify_all();
        for (std::thread &t : threads_) t.join();
    }
    size_t size() const { return threads_.size() + 1; }
    void run(size_t n, const std::function<void(size_t)> &f) {
        if (n > size()) n = size();
        { std::lock_guard<std::mutex> g(m_); f_ = &f; n_ = n; pending_ = n ? n - 1 : 0; gen_++; }
        cv_.notify_all();
        if (n) f(0);
        std::unique_lock<std::mutex> g(m_);
        done_.wait(g, [this] { return pending_ == 0; });
        f_ = nullptr;
    }
private:
    void loop(size_t me) {
        uint64_t seen = 0;
        for (;;) {
            const std::function<void(size_t)> *f;
            {
                std::unique_lock<std::mutex> g(m_);
                cv_.wait(g, [&] { return gen_ != seen; });
                seen = gen_;
                if (stop_) return;
                if (me >= n_) continue;
                f = f_;
            }
            (*f)(me);
            { std::lock_guard<std::mutex> g(m_); pending_--; }
            done_.notify_one();
        }
    }
    std::vector<std::thread> threads_;
    std::mutex m_;
    std::condition_variable cv_, done_;
    const std::function<void(size_t)> *f_ = nullptr;
    size_t n_ = 0, pending_ = 0;
    uint64_t gen_ = 0;
    bool stop_ = false;
};

}  // namespace

struct modes_pool {
    modes_config cfg;
    std::vector<Receiver> rx;
    size_t max_batch = 0;
    std::string err;
    // device half (created on the first modes_pool_submit / _ingest): two batches may be in flight, so
    // that one is uploaded and scanned while the one before it is resolved on the host
    struct Slot {
        modes_ctx *ctx = nullptr;
        uint8_t *d_batch = nullptr;            // [2 * max_batch] buffers: pad, data, pad, data, ...
        uint8_t *h_carry = nullptr;            // pinned [max_batch][MODES_CARRY_BYTES]
        std::vector<uint32_t> ids;             // the receivers of the batch in flight
        bool busy = false;
    } slot[2];
    unsigned submitted = 0, collected = 0;     // batches so far: slot = number & 1
    std::vector<modes_candidate> cands;
    std::vector<modes_tile> tiles;
    // the per-receiver resolve: one block of the receiver list per host thread
    struct Block {
        std::vector<modes_candidate> local;    // one receiver's records, re-based to its buffer
        std::vector<modes_tile> local_tiles;
        std::vector<modes_message> msgs;       // the block's messages, receiver by receiver
        std::vector<size_t> counts;            // messages of each receiver of the block
        size_t used = 0, at = 0;               // messages of the block; where they start in the call's sequence
        int64_t failed = -1;
    };
    std::vector<Block> blocks;
    std::unique_ptr<Crew> crew;
    // cfg.gpu_resolve: the device resolve's memory, used by one collect at a time
    struct Device {
        uint32_t *caches = nullptr;            // [n_receivers][1024]
        uint32_t *work = nullptr;              // ids [max_batch], offsets [max_batch + 1], flags [4], then n_deliv [n] + stats [n][8]
        uint32_t *h_work = nullptr;            // pinned: ids [max_batch], then n_deliv [n] + stats [n][8]
        modes::modes_delivery *out = nullptr;  // [out_cap]
        modes::modes_delivery *h_out = nullptr;   // pinned [out_cap]
        size_t out_cap = 0;
        std::vector<modes_message> spill;      // structs that do not fit the output array, for the sink
        std::vector<size_t> first;             // [n + 1] where entry i's deliveries start
    } dev;
    // optional caller-owned output array (modes_pool_set_output)
    modes_message *out = nullptr; uint32_t *out_rx = nullptr; size_t out_cap = 0, out_count = 0;
};

namespace {

int fail(modes_pool *p, const char *fmt, ...) {
    char buf[256];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    p->err = buf;
    return -1;
}

int check_ids(modes_pool *p, const uint32_t *receivers, size_t n) {
    if (!receivers && n) return fail(p, "no receiver list");
    if (n > p->max_batch) return fail(p, "%zu receivers in one call, the pool was created for %zu", n, p->max_batch);
    for (size_t i = 0; i < n; i++) {
        if (receivers[i] >= p->rx.size()) return fail(p, "receiver %u out of range (%zu receivers)", receivers[i], p->rx.size());
        for (size_t k = 0; k < i; k++)
            if (receivers[k] == receivers[i]) return fail(p, "receiver %u listed twice: one buffer per receiver and call", receivers[i]);
    }
    return 0;
}

// Host threads of the per-receiver resolve: MODES_POOL_THREADS, else 4 (receivers are independent; one
// block of 16 or more receivers per thread).
size_t pool_threads() {
    static const size_t n = [] {
        const char *e = std::getenv("MODES_POOL_THREADS");
        long v = e ? std::strtol(e, nullptr, 10) : 4;
        return (size_t)(v < 1 ? 1 : v > 64 ? 64 : v);
    }();
    return n;
}

int ensure_device(modes_pool *p) {
    if (p->slot[0].ctx) return 0;
    modes_config c = p->cfg;
    c.n_gpus = 1; c.gpu_resolve = 0;
    const size_t bytes = 2 * p->max_batch * kBuf;
    for (modes_pool::Slot &sl : p->slot) {
        sl.ctx = modes_create(&c);
        if (!sl.ctx) return fail(p, "%s", modes_last_error(nullptr));
        sl.d_batch = static_cast<uint8_t *>(modes_device_alloc(bytes));
        sl.h_carry = static_cast<uint8_t *>(modes_host_alloc(p->max_batch * MODES_CARRY_BYTES));
        if (!sl.d_batch || !sl.h_carry) return fail(p, "out of memory for %zu receivers per batch", p->max_batch);
        if (modes_device_memset(sl.d_batch, 127, bytes)) return fail(p, "device memset failed");      // dump1090.c:344 no signal
    }
    if (p->cfg.gpu_resolve) {
        // no clearing: every receiver starts fresh, and its first batch writes its whole cache
        modes_pool::Device &d = p->dev;
        const size_t mb = p->max_batch;
        if (cudaMalloc(&d.caches, p->rx.size() * 1024 * sizeof(uint32_t)) != cudaSuccess ||
            cudaMalloc(&d.work, (2 * mb + 5 + 9 * mb) * sizeof(uint32_t)) != cudaSuccess ||
            cudaMallocHost(&d.h_work, 10 * mb * sizeof(uint32_t)) != cudaSuccess)
            return fail(p, "out of memory for the device resolve of %zu receivers", p->rx.size());
    }
    return 0;
}

// Blocks of the receiver list for the host threads: one block of 16 or more receivers per thread.
size_t blocks_for(size_t n) {
    size_t n_blocks = pool_threads();
    if (n_blocks > (n + 15) / 16) n_blocks = (n + 15) / 16;
    return n_blocks < 1 ? 1 : n_blocks;
}

// cfg.gpu_resolve: the verdicts of the collected batch in slot `sl` (its records are where
// modes_detect_device left them) on the device, then the structs on the host, handed over in list order.
int resolve_on_device(modes_pool *p, const modes_pool::Slot &sl, uint64_t n_cand, modes_pool_sink_fn sink, void *user) {
    modes_pool::Device &d = p->dev;
    const uint32_t *ids = sl.ids.data();
    const size_t n = sl.ids.size(), mb = p->max_batch;
    cudaStream_t st = static_cast<cudaStream_t>(modes_stream(sl.ctx));
    const size_t cap = 2 * (n_cand ? n_cand : 1);                  // a candidate delivers at most two messages
    if (d.out_cap < cap) {
        cudaFree(d.out); cudaFreeHost(d.h_out); d.out = nullptr; d.h_out = nullptr; d.out_cap = 0;
        const size_t c = cap + cap / 2;
        if (cudaMalloc(&d.out, c * sizeof(modes::modes_delivery)) != cudaSuccess ||
            cudaMallocHost(&d.h_out, c * sizeof(modes::modes_delivery)) != cudaSuccess)
            return fail(p, "out of memory for %zu deliveries", c);
        d.out_cap = c;
    }
    for (size_t i = 0; i < n; i++) {
        Receiver &r = p->rx[ids[i]];
        d.h_work[i] = ids[i] | (r.fresh ? modes::kPoolFresh : 0u);
        r.fresh = false;
    }
    modes::PoolResolve pr;
    pr.caches = d.caches;
    pr.ids = d.work;
    pr.offsets = d.work + mb;
    pr.flags = d.work + 2 * mb + 1;
    pr.n_deliv = d.work + 2 * mb + 5;
    pr.stats = pr.n_deliv + n;
    pr.out = d.out;
    pr.capacity = (uint32_t)cap;
    const modes_candidate *records; const modes_tile *tiles; uint32_t n_tiles;
    modes::detect_results(sl.ctx, &records, &tiles, &n_tiles);
    uint32_t *h_counts = d.h_work + mb, *h_stats = h_counts + n;
    cudaError_t e = cudaSetDevice(p->cfg.device);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d.work, d.h_work, n * sizeof(uint32_t), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
        modes::launch_pool_resolve(pr, records, tiles, n_tiles, (uint32_t)n, p->cfg.check_crc, st);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_counts, pr.n_deliv, 9 * n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = modes::wait_stream(st);
    if (e != cudaSuccess) return fail(p, "device resolve failed: %s", cudaGetErrorString(e));
    d.first.resize(n + 1);
    d.first[0] = 0;
    for (size_t i = 0; i < n; i++) d.first[i + 1] = d.first[i] + h_counts[i];
    const size_t total = d.first[n];
    if (total) {
        e = cudaMemcpyAsync(d.h_out, d.out, total * sizeof(modes::modes_delivery), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = modes::wait_stream(st);
        if (e != cudaSuccess) return fail(p, "delivery download failed: %s", cudaGetErrorString(e));
    }
    for (size_t i = 0; i < n; i++) {
        Receiver &r = p->rx[ids[i]];
        for (int k = 0; k < 8; k++) r.stats[k] += h_stats[8 * i + k];
    }
    // The structs, receiver by receiver (each from its own stream position), one block of receivers per
    // host thread: into the caller's array where they fit, into `spill` where the sink needs the rest.
    const size_t base = p->out_count, out_cap = p->out ? p->out_cap : 0;
    const size_t fit = base >= out_cap ? 0 : (total < out_cap - base ? total : out_cap - base);
    if (sink && d.spill.size() < total - fit) d.spill.resize(total - fit);
    const size_t n_blocks = blocks_for(n);
    auto build = [&](size_t b) {
        for (size_t i = n * b / n_blocks; i < n * (b + 1) / n_blocks; i++) {
            const int64_t buffers = p->rx[ids[i]].buffers;
            const size_t f0 = d.first[i], f1 = d.first[i + 1], in_array = f1 < fit ? f1 : (f0 < fit ? fit : f0);
            if (in_array > f0) {
                modes::MessageOut mo;
                mo.array = p->out + base; mo.capacity = fit; mo.count = f0;
                modes::deliver_gpu(d.h_out + f0, in_array - f0, buffers, mo);
                for (size_t k = f0; k < in_array; k++) p->out_rx[base + k] = ids[i];
            }
            if (sink && f1 > in_array) {
                modes::MessageOut mo;
                mo.array = d.spill.data(); mo.capacity = total - fit; mo.count = in_array - fit;
                modes::deliver_gpu(d.h_out + in_array, f1 - in_array, buffers, mo);
            }
        }
    };
    if (p->out || sink) {
        if (!p->crew) p->crew.reset(new Crew(pool_threads() - 1));
        p->crew->run(n_blocks, build);
    }
    if (p->out) p->out_count += total;
    if (sink)
        for (size_t i = 0; i < n; i++)
            for (size_t k = d.first[i]; k < d.first[i + 1]; k++)
                sink(user, ids[i], k < fit ? &p->out[base + k] : &d.spill[k - fit]);
    for (size_t i = 0; i < n; i++) p->rx[ids[i]].buffers++;
    return 0;
}

}  // namespace

extern "C" {

modes_pool *modes_pool_create(const modes_config *cfg, size_t n_receivers, size_t max_batch_receivers) {
    if (!cfg || !n_receivers) return nullptr;
    modes_pool *p = new modes_pool();
    p->cfg = *cfg;
    p->max_batch = max_batch_receivers && max_batch_receivers < n_receivers ? max_batch_receivers : n_receivers;
    p->rx.resize(n_receivers);
    for (Receiver &r : p->rx) {
        r.res = modes_resolver_create(cfg);
        memset(r.carry, 127, sizeof r.carry);
        if (!r.res) { modes_pool_destroy(p); return nullptr; }
    }
    return p;
}

void modes_pool_destroy(modes_pool *p) {
    if (!p) return;
    for (Receiver &r : p->rx) if (r.res) modes_resolver_destroy(r.res);
    for (modes_pool::Slot &sl : p->slot) {
        if (sl.d_batch) modes_device_free(sl.d_batch);
        if (sl.h_carry) modes_host_free(sl.h_carry);
        if (sl.ctx) modes_destroy(sl.ctx);
    }
    if (p->dev.caches) cudaFree(p->dev.caches);
    if (p->dev.work) cudaFree(p->dev.work);
    if (p->dev.h_work) cudaFreeHost(p->dev.h_work);
    if (p->dev.out) { cudaFree(p->dev.out); cudaFreeHost(p->dev.h_out); }
    delete p;
}

const char *modes_pool_last_error(const modes_pool *p) { return p ? p->err.c_str() : "no pool"; }

int modes_pool_resolve(modes_pool *p, const uint32_t *receivers, size_t n, const modes_candidate *candidates,
                       const modes_tile *tiles, modes_pool_sink_fn sink, void *user) {
    if (!p) return -1;
    if (p->cfg.gpu_resolve)
        return fail(p, "this pool resolves on the device (gpu_resolve = 1): its address caches live there, "
                       "so modes_pool_resolve (the host half of a gpu_resolve = 0 pool) is not available");
    if (check_ids(p, receivers, n)) return -1;
    if (!n) return 0;
    if (!tiles) return fail(p, "no tile table");
    const size_t n_tiles = modes_tile_count(2 * n);
    const size_t n_local = modes_tile_count(1);
    // Receivers are independent: the list is cut into blocks, one host thread each; a block's messages
    // land in its own array and are moved to the caller's array / handed to the sink in list order.
    const size_t n_blocks = blocks_for(n);
    if (p->blocks.size() < n_blocks) p->blocks.resize(n_blocks);
    auto tile_range = [&](size_t i, size_t &g0, size_t &g1) {
        // the data buffer of pair i is buffer 2i+1 of the batch; a position t belongs to the tile
        // that holds virtual position t + 2
        const int64_t t0 = kBufSamples * (int64_t)(2 * i + 1), t1 = t0 + kBufSamples;
        g0 = (size_t)((t0 + 2) / MODES_TILE_SAMPLES); g1 = (size_t)((t1 + 1) / MODES_TILE_SAMPLES);
        if (g1 >= n_tiles) g1 = n_tiles - 1;
    };
    auto work = [&](size_t b) {
        modes_pool::Block &bl = p->blocks[b];
        const size_t i0 = n * b / n_blocks, i1 = n * (b + 1) / n_blocks;
        bl.failed = -1;
        bl.counts.assign(i1 - i0, 0);
        size_t room = 0, ga, gb, gc, gd;
        tile_range(i0, ga, gb); tile_range(i1 - 1, gc, gd);
        for (size_t g = ga; g <= gd; g++) room += 2 * (size_t)tiles[g].count;  // a candidate delivers at most two messages (both attempts without --check-crc... dump1090.c:1803)
        if (bl.msgs.size() < room) bl.msgs.resize(room);
        bl.local_tiles.resize(n_local);
        size_t used = 0;
        for (size_t i = i0; i < i1; i++) {
            Receiver &r = p->rx[receivers[i]];
            const int64_t t0 = kBufSamples * (int64_t)(2 * i + 1), t1 = t0 + kBufSamples;
            size_t g0, g1;
            tile_range(i, g0, g1);
            bl.local.clear();
            for (modes_tile &lt : bl.local_tiles) { lt.offset = 0; lt.count = 0; }
            for (size_t g = g0; g <= g1; g++) {
                const modes_candidate *c = candidates + tiles[g].offset;
                for (uint32_t k = 0; k < tiles[g].count; k++) {
                    if (c[k].t < t0 || c[k].t >= t1) continue;
                    modes_candidate lc = c[k];
                    lc.t -= t0;                           // position inside the receiver's own buffer
                    const size_t lg = (size_t)((lc.t + 2) / MODES_TILE_SAMPLES);
                    if (lg >= n_local) { bl.failed = (int64_t)i; return; }
                    bl.local_tiles[lg].count++;
                    bl.local.push_back(lc);
                }
            }
            uint32_t off = 0;
            for (modes_tile &lt : bl.local_tiles) { lt.offset = off; off += lt.count; }
            modes_resolver_set_output(r.res, bl.msgs.data() + used, room - used);
            if (modes_resolver_run(r.res, bl.local.data(), bl.local_tiles.data(), n_local, r.buffers, nullptr, nullptr)) {
                bl.failed = (int64_t)i; return;
            }
            const size_t k = modes_resolver_output_count(r.res);
            modes_resolver_set_output(r.res, nullptr, 0);
            bl.counts[i - i0] = k;
            used += k;
            r.buffers++;
        }
        bl.used = used;
    };
    if (!p->crew) p->crew.reset(new Crew(pool_threads() - 1));
    p->crew->run(n_blocks, work);
    for (size_t b = 0; b < n_blocks; b++)
        if (p->blocks[b].failed >= 0) return fail(p, "resolve of receiver %u failed", receivers[p->blocks[b].failed]);
    // in list order into the caller's array (the count keeps running past its capacity): every block
    // moves its own messages
    size_t total = 0;
    for (size_t b = 0; b < n_blocks; b++) { p->blocks[b].at = total; total += p->blocks[b].used; }
    if (p->out) {
        const size_t base = p->out_count, cap = p->out_cap;
        auto move = [&](size_t b) {
            const modes_pool::Block &bl = p->blocks[b];
            const size_t i0 = n * b / n_blocks, first = base + bl.at;
            const size_t fit = first >= cap ? 0 : (bl.used < cap - first ? bl.used : cap - first);
            if (fit) memcpy(p->out + first, bl.msgs.data(), fit * sizeof(modes_message));
            size_t at = 0;
            for (size_t j = 0; j < bl.counts.size(); j++)
                for (size_t m = 0; m < bl.counts[j]; m++, at++)
                    if (at < fit) p->out_rx[first + at] = receivers[i0 + j];
        };
        p->crew->run(n_blocks, move);
        p->out_count += total;
    }
    if (sink)
        for (size_t b = 0; b < n_blocks; b++) {
            const modes_pool::Block &bl = p->blocks[b];
            const size_t i0 = n * b / n_blocks;
            size_t at = 0;
            for (size_t j = 0; j < bl.counts.size(); j++)
                for (size_t m = 0; m < bl.counts[j]; m++, at++) sink(user, receivers[i0 + j], &bl.msgs[at]);
        }
    return 0;
}

int modes_pool_submit(modes_pool *p, const uint32_t *receivers, const uint8_t *const *iq, size_t n) {
    if (!p) return -1;
    if (check_ids(p, receivers, n)) return -1;
    if (!n) return fail(p, "an empty batch");
    if (!iq) return fail(p, "no buffers");
    if (ensure_device(p)) return -1;
    modes_pool::Slot &sl = p->slot[p->submitted & 1];
    if (sl.busy) return fail(p, "two batches are in flight: modes_pool_collect first");
    cudaStream_t st = static_cast<cudaStream_t>(modes_stream(sl.ctx));
    // the carries into the tails of the pad buffers, the new buffers behind them
    for (size_t i = 0; i < n; i++) {
        if (!iq[i]) return fail(p, "receiver %u: no buffer", receivers[i]);
        memcpy(sl.h_carry + i * MODES_CARRY_BYTES, p->rx[receivers[i]].carry, MODES_CARRY_BYTES);
    }
    if (cudaMemcpy2DAsync(sl.d_batch + kBuf - MODES_CARRY_BYTES, 2 * kBuf, sl.h_carry, MODES_CARRY_BYTES, MODES_CARRY_BYTES, n,
                          cudaMemcpyHostToDevice, st) != cudaSuccess)
        return fail(p, "carry upload failed: %s", cudaGetErrorString(cudaGetLastError()));
    // receivers' buffers at a constant distance in host memory (one staging block): one strided copy
    // instead of n calls (2-3 us of host time each: at 256 receivers more than the copy itself takes)
    bool strided = n > 1 && iq[1] > iq[0];
    const size_t stride = strided ? (size_t)(iq[1] - iq[0]) : 0;
    for (size_t i = 1; strided && i + 1 < n; i++) strided = iq[i + 1] > iq[i] && (size_t)(iq[i + 1] - iq[i]) == stride;
    if (strided && stride >= kBuf && stride < ((size_t)1 << 30)) {
        if (cudaMemcpy2DAsync(sl.d_batch + kBuf, 2 * kBuf, iq[0], stride, kBuf, n, cudaMemcpyHostToDevice, st) != cudaSuccess)
            return fail(p, "buffer upload failed: %s", cudaGetErrorString(cudaGetLastError()));
    } else {
        for (size_t i = 0; i < n; i++)
            if (cudaMemcpyAsync(sl.d_batch + (2 * i + 1) * kBuf, iq[i], kBuf, cudaMemcpyHostToDevice, st) != cudaSuccess)
                return fail(p, "buffer upload failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    if (modes_detect_device(sl.ctx, sl.d_batch, 2 * n, nullptr, nullptr, 0, nullptr)) return fail(p, "%s", modes_last_error(sl.ctx));
    // what each receiver carries into its next buffer (dump1090.c:481)
    for (size_t i = 0; i < n; i++)
        memcpy(p->rx[receivers[i]].carry, iq[i] + kBuf - MODES_CARRY_BYTES, MODES_CARRY_BYTES);
    sl.ids.assign(receivers, receivers + n);
    sl.busy = true;
    p->submitted++;
    return 0;
}

int modes_pool_collect(modes_pool *p, modes_pool_sink_fn sink, void *user) {
    if (!p) return -1;
    if (p->collected == p->submitted) return fail(p, "no batch in flight");
    modes_pool::Slot &sl = p->slot[p->collected & 1];
    uint64_t n_cand = 0;
    if (modes_detect_wait(sl.ctx, &n_cand)) return fail(p, "%s", modes_last_error(sl.ctx));
    if (p->cfg.gpu_resolve) {
        sl.busy = false;
        p->collected++;
        return resolve_on_device(p, sl, n_cand, sink, user);
    }
    const size_t n = sl.ids.size();
    p->cands.resize(n_cand ? n_cand : 1);
    p->tiles.resize(modes_tile_count(2 * n));
    if (modes_detect_fetch(sl.ctx, p->cands.data(), p->tiles.data())) return fail(p, "%s", modes_last_error(sl.ctx));
    sl.busy = false;
    p->collected++;
    return modes_pool_resolve(p, sl.ids.data(), n, p->cands.data(), p->tiles.data(), sink, user);
}

int modes_pool_ingest(modes_pool *p, const uint32_t *receivers, const uint8_t *const *iq, size_t n,
                      modes_pool_sink_fn sink, void *user) {
    if (!p) return -1;
    if (p->collected != p->submitted) return fail(p, "a submitted batch is in flight: modes_pool_collect first");
    if (!n) return check_ids(p, receivers, n);
    if (modes_pool_submit(p, receivers, iq, n)) return -1;
    return modes_pool_collect(p, sink, user);
}

int modes_pool_stats(const modes_pool *p, uint32_t receiver, modes_stats *out) {
    if (!p || receiver >= p->rx.size() || !out) return -1;
    if (p->cfg.gpu_resolve) {
        memcpy(out->v, p->rx[receiver].stats, sizeof(out->v));
        return 0;
    }
    return modes_resolver_stats(p->rx[receiver].res, out);
}

int modes_pool_reset(modes_pool *p, uint32_t receiver) {
    if (!p || receiver >= p->rx.size()) return -1;
    Receiver &r = p->rx[receiver];
    r.buffers = 0;
    memset(r.carry, 127, sizeof r.carry);
    memset(r.stats, 0, sizeof r.stats);
    r.fresh = true;                            // its next collected batch starts from an empty cache
    return modes_resolver_reset(r.res);
}

int modes_pool_set_output(modes_pool *p, modes_message *out, uint32_t *receiver_of, size_t capacity) {
    if (!p || ((out == nullptr) != (receiver_of == nullptr))) return -1;
    p->out = out; p->out_rx = receiver_of; p->out_cap = out ? capacity : 0; p->out_count = 0;
    return 0;
}

size_t modes_pool_output_count(const modes_pool *p) { return p ? p->out_count : 0; }

int64_t modes_pool_buffers(const modes_pool *p, uint32_t receiver) {
    if (!p || receiver >= p->rx.size()) return -1;
    return p->rx[receiver].buffers;
}

}  // extern "C"
