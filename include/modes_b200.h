/* modes_b200.h — C ABI of the B200-native Mode S / ADS-B demodulator.
 *
 * Drop-in boundary for dump1090's --ifile decode path.  The reference has no
 * plugin/FFI surface; the seam is its main loop (dump1090.c:2968-2990):
 *
 *     computeMagnitudeVector();                       dump1090.c:1454 / :2974
 *     detectModeS(Modes.magnitude, Modes.data_len/2); dump1090.c:1563 / :2986
 *         -> decodeModesMessage(&mm, msg)             dump1090.c:1091 / :1735
 *         -> useModesMessage(&mm)                     dump1090.c:1802 / :1777
 *
 * Each entry point below names the reference interface it replaces.  Plain C
 * types only; the library owns all device memory, streams and chunking, so
 * a caller passes raw file bytes in file order in pieces of any size and gets
 * back, in stream order, exactly the messages (and struct modesMessage fields)
 * the reference hands to useModesMessage() for the same bytes.
 *
 * There is no CPU fallback: modes_create() fails (NULL + modes_last_error)
 * when no CUDA device is usable.
 *
 * Threading: a context is not re-entrant (one thread at a time per modes_ctx, like the
 * reference's single decode thread); distinct contexts are independent.  Callbacks run on the
 * calling thread.  Status codes: 0 = ok, <0 = error with text in modes_last_error(ctx); the
 * library never calls exit().
 */
#ifndef MODES_B200_H
#define MODES_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MODES_B200_ABI_VERSION 3

/* Sizes fixed by the reference's buffering (dump1090.c:54, :61, :331). */
#define MODES_BUFFER_BYTES    262144      /* MODES_DATA_LEN: new bytes per reference buffer */
#define MODES_BUFFER_SAMPLES  131072
#define MODES_CARRY_BYTES     476         /* (MODES_FULL_LEN-1)*4 carried into the next buffer */
#define MODES_CARRY_SAMPLES   238

/* Replaces the four globals that change hot-path results: Modes.fix_errors
 * (dump1090.c:167, --no-fix :2873), Modes.aggressive (:179, :2896),
 * Modes.check_crc (:168, :2875), plus the EOF-buffer race made explicit
 * (dump1090.c:497 vs :2989; SURVEY.md fact 3). */
typedef struct modes_config {
    int32_t fix_errors;         /* 1 (default): 1-bit (2-bit if aggressive) CRC repair on DF11/17/18 */
    int32_t aggressive;         /* 0 (default) */
    int32_t check_crc;          /* 1 (default): deliver only messages with crcok */
    int32_t drop_eof_buffer;    /* 0 (default): decode the buffer that hit EOF; 1: drop it, as the
                                   stock binary does in most runs */
    int32_t device;             /* CUDA device ordinal, default 0 */
    int32_t profile;            /* 1: record per-kernel CUDA-event times (modes_get_kernel_times) */
    uint64_t max_batch_bytes;   /* device staging per in-flight batch; 0 = 64 MiB */
    int32_t n_gpus;             /* 0 or 1: one GPU (`device`).  N > 1: the streaming decode (modes_process /
                                   modes_finish) deals its batches of whole reference buffers round-robin to N
                                   devices starting at `device` — one stream, one pinned-to-device copy and
                                   two staging slots per GPU, every GPU behind its own PCIe link — and the
                                   calling thread resolves each group of N batches exactly (the speculative
                                   shard resolve of modes_resolver_run_shards).  With fewer than N devices
                                   present, devices are reused round-robin.  The stage-level entry points
                                   stay on `device`. */
    int32_t gpu_resolve;        /* 0 (default): the order-dependent half (retry/skip state machine, ICAO cache,
                                   statistics: dump1090.c:1769-1791, :898-983) is replayed on the host over the
                                   candidate records.  1: it runs on the GPU too — one warp per reference buffer,
                                   address caches handed from buffer to buffer and verified (SURVEY.md §8(f) item
                                   4) — and only 40-byte records of the delivered messages cross PCIe; the host
                                   builds the struct fields.  Same messages, same statistics.  Streaming decode
                                   on one GPU only; a batch denser than one candidate per 64 samples is an error
                                   in this mode.  A receiver pool (modes_pool_*) with gpu_resolve = 1 resolves on
                                   the device too: one warp per receiver, every receiver's address cache kept in
                                   device memory between batches; there a dense batch is repeated as usual. */
} modes_config;

/* Replaces struct modesMessage (dump1090.c:211-260): same field names and
 * meaning, 32-bit fields in a fixed order.  Fields the reference leaves
 * unassigned for a given DF are 0 here.  nfixed and sample_pos are additions. */
typedef struct modes_message {
    uint8_t  msg[14];
    uint8_t  pad0[2];
    int32_t  msgbits, msgtype, crcok;
    uint32_t crc;
    int32_t  errorbit, aa1, aa2, aa3, phase_corrected;
    int32_t  ca, iid;
    int32_t  metype, mesub, heading_is_valid, heading, aircraft_type;
    int32_t  fflag, tflag, raw_latitude, raw_longitude;
    char     flight[9];
    char     pad1[3];
    int32_t  ew_dir, ew_velocity, ns_dir, ns_velocity;
    int32_t  vert_rate_source, vert_rate_sign, vert_rate, velocity;
    int32_t  movement, movement_valid, ground_track, ground_track_valid;
    int32_t  fs, dr, um, identity;
    int32_t  altitude, unit;
    int32_t  nfixed;            /* bits repaired by the CRC fix (0/1/2) */
    int32_t  pad2;
    int64_t  sample_pos;        /* stream sample index of the preamble start */
} modes_message;

/* One evaluated frame attempt at one preamble position: everything
 * detectModeS()+decodeModesMessage() compute that is a pure function of the
 * samples and the flags (dump1090.c:1668-1735, :1099-1128). */
typedef struct modes_frame_eval {
    uint8_t  msg[14];           /* frame bytes, after the CRC fix if one was applied */
    uint8_t  msgtype;           /* DF of the demodulated frame (before any fix) */
    uint8_t  flags;             /* MODES_EVAL_* */
    uint8_t  errorbit;          /* first repaired bit, 0xFF = none */
    uint8_t  nfixed;
    uint32_t crc;               /* 24-bit syndrome after the fix; 0 when not decoded */
} modes_frame_eval;

#define MODES_EVAL_GATE_OK   1  /* mean |low-high| >= 2550             dump1090.c:1723 */
#define MODES_EVAL_ERRORS    2  /* demodulation error in first 56 bits dump1090.c:1682 */
#define MODES_EVAL_DECODED   4  /* decodeModesMessage reached          dump1090.c:1731 */
#define MODES_EVAL_P2_VALID  8  /* pass[1] (phase-corrected retry) was evaluated */

/* One preamble candidate: a position that passes the tests of
 * dump1090.c:1602-1650, with the first attempt and the phase-corrected retry
 * (dump1090.c:1653-1664) both evaluated on the device. */
typedef struct modes_candidate {
    int64_t t;                  /* 131072*buffer_index + j  (j = index inside the reference buffer) */
    modes_frame_eval pass[2];
} modes_candidate;

/* Per scan tile: where its candidates sit in the candidate array.  Tiles are
 * in stream order; candidates inside a tile are in stream order.  How many positions a tile
 * covers is the scan kernel's business: size tile tables with modes_tile_count(). */
typedef struct modes_tile { uint32_t offset, count; } modes_tile;
#define MODES_TILE_SAMPLES 7936             /* 8 rows of 31 x 32 positions, see csrc/modes_scan2.cu */

/* Replaces Modes.stat_* (dump1090.c:186-195) in the order the reference prints
 * them (:2994-3003): valid_preamble, out_of_phase, demodulated, goodcrc,
 * badcrc, fixed, single_bit_fix, two_bits_fix. */
typedef struct modes_stats { int64_t v[8]; } modes_stats;

typedef struct modes_ctx modes_ctx;

/* Replaces useModesMessage(struct modesMessage*) (dump1090.c:1802): called on
 * the calling thread from modes_process/modes_finish/modes_resolve, in stream
 * order, once per message that passes the reference's gate (:1803).  The
 * pointer is valid only during the call. */
typedef void (*modes_sink_fn)(void *user, const modes_message *mm);

/* ---- lifecycle ---------------------------------------------------------- */
int         modes_abi_version(void);
void        modes_default_config(modes_config *cfg);                 /* modesInitConfig, dump1090.c:299 */
modes_ctx  *modes_create(const modes_config *cfg);                   /* modesInit, dump1090.c:321 */
void        modes_destroy(modes_ctx *ctx);
const char *modes_last_error(const modes_ctx *ctx);                  /* ctx may be NULL: create() error */
int         modes_set_sink(modes_ctx *ctx, modes_sink_fn fn, void *user);

/* Alternative to a callback: append every delivered message to a caller-owned
 * array (NULL/0 to stop).  modes_output_count() keeps counting past capacity. */
int    modes_set_output(modes_ctx *ctx, modes_message *out, size_t capacity);
size_t modes_output_count(const modes_ctx *ctx);

/* ---- streaming decode: the main loop, dump1090.c:2968-2990 -------------- */
/* Feed the next `nbytes` of the u8 I/Q stream (host memory, pinned or not).
 * Whole reference buffers are decoded as they complete.  0 = ok, <0 = error. */
int  modes_process(modes_ctx *ctx, const uint8_t *iq, size_t nbytes);
/* End of stream: 127-pad and decode (or drop) the EOF buffer (dump1090.c:496-507). */
int  modes_finish(modes_ctx *ctx);
/* Forget stream position, carry, ICAO cache and statistics (a new --ifile run). */
int  modes_reset(modes_ctx *ctx);
int  modes_get_stats(const modes_ctx *ctx, modes_stats *out);

/* ---- stage-level entry points (tests, bench, multi-GPU sharding) -------- */
/* computeMagnitudeVector() alone (dump1090.c:1454-1469): nsamples I/Q pairs in
 * host memory -> nsamples u16 magnitudes in host memory, computed on the device. */
int  modes_compute_magnitude(modes_ctx *ctx, const uint8_t *iq, size_t nsamples, uint16_t *mag);

/* The device half of detectModeS() on data already in HBM.  d_iq: n_buffers *
 * MODES_BUFFER_BYTES bytes of device memory (16-byte aligned) holding whole
 * reference buffers of the stream; carry476: the MODES_CARRY_BYTES stream
 * bytes preceding d_iq (host memory), or NULL at stream start (no-signal).
 * Launches the scan and frame-evaluation kernels on the context's stream and
 * returns without waiting.  d_candidates (capacity cand_capacity records) and
 * d_tiles (modes_tile_count(n_buffers) entries) are device memory supplied by the caller, or
 * NULL to use the context's own workspace. */
int  modes_detect_device(modes_ctx *ctx, const void *d_iq, size_t n_buffers, const uint8_t *carry476,
                         void *d_candidates, size_t cand_capacity, void *d_tiles);
/* Same, from HOST memory (pinned for full speed): the library stages the buffers into its own device
 * memory with one asynchronous copy on the same stream, then launches the kernels. */
int  modes_detect_host(modes_ctx *ctx, const uint8_t *iq, size_t n_buffers, const uint8_t *carry476,
                       void *d_candidates, size_t cand_capacity, void *d_tiles);
/* Wait for the last modes_detect_device; returns the candidate count. */
int  modes_detect_wait(modes_ctx *ctx, uint64_t *n_candidates);
/* Copy the last result to host memory (arrays sized by the caller from
 * modes_detect_wait's count and modes_tile_count(n_buffers) tiles). */
int  modes_detect_fetch(modes_ctx *ctx, modes_candidate *candidates, modes_tile *tiles);

/* The sequential half of detectModeS(): retry/skip state machine
 * (dump1090.c:1769-1791), ICAO cache (:898-983, :1183-1210), statistics and the
 * sink gate (:1803), replayed over candidates in stream order.  buffer_base is
 * the stream index of the first reference buffer the arrays describe. */
int  modes_resolve(modes_ctx *ctx, const modes_candidate *candidates, const modes_tile *tiles,
                   size_t n_tiles, int64_t buffer_base);

/* The same sequential half as a standalone host object (no device needed): what
 * rank 0 runs over gathered candidate records in a multi-GPU job. */
typedef struct modes_resolver modes_resolver;
modes_resolver *modes_resolver_create(const modes_config *cfg);
void modes_resolver_destroy(modes_resolver *r);
int  modes_resolver_run(modes_resolver *r, const modes_candidate *candidates, const modes_tile *tiles,
                        size_t n_tiles, int64_t buffer_base, modes_sink_fn sink, void *user);
/* Several consecutive shards of one stream at once (one per GPU): resolved concurrently on host
 * threads by speculating the ICAO cache at each shard boundary and verifying it; the result is
 * identical to calling modes_resolver_run shard by shard. */
int  modes_resolver_run_shards(modes_resolver *r, size_t n_shards, const modes_candidate *const *candidates,
                               const modes_tile *const *tiles, const size_t *n_tiles, const int64_t *buffer_base,
                               modes_sink_fn sink, void *user);
/* One shard of a sharded decode, resolved where its records are (one rank or GPU thread per shard).
 * The only state crossing a shard boundary is the 1024-slot address cache (dump1090.c:335, :898-983):
 * a shard is resolved TENTATIVELY from a guess of the cache at its start — the job's starting cache
 * overwritten by what the tail of the previous shard leaves (modes_resolver_tail_cache, exchanged
 * between the shards' owners, 4 KiB) — the guess is compared with what the previous shard really
 * ended with (modes_resolver_get_cache after its tentative run), and a shard whose guess was wrong
 * is run again from the right cache.  modes_resolver_commit then delivers the messages and adds the
 * statistics.  dump1090_b200/sharded.py:resolve_distributed is the protocol over torch.distributed;
 * modes_resolver_run_shards is the same thing inside one process. */
#define MODES_ICAO_CACHE_SLOTS 1024
int  modes_resolver_get_cache(const modes_resolver *r, uint32_t cache[MODES_ICAO_CACHE_SLOTS]);  /* of the tentative run if one is pending */
int  modes_resolver_set_cache(modes_resolver *r, const uint32_t cache[MODES_ICAO_CACHE_SLOTS]);  /* NULL = empty; drops a pending run */
int  modes_resolver_tail_cache(const modes_resolver *r, const modes_candidate *candidates, const modes_tile *tiles,
                               size_t n_tiles, int64_t buffer_base, size_t n_tail_tiles, uint32_t cache[MODES_ICAO_CACHE_SLOTS]);
int  modes_resolver_run_tentative(modes_resolver *r, const modes_candidate *candidates, const modes_tile *tiles,
                                  size_t n_tiles, int64_t buffer_base);            /* records must stay valid until commit */
int  modes_resolver_commit(modes_resolver *r, modes_sink_fn sink, void *user);
int  modes_resolver_reset(modes_resolver *r);           /* forget ICAO cache, skip state, statistics */
int  modes_resolver_stats(const modes_resolver *r, modes_stats *out);
int    modes_resolver_set_output(modes_resolver *r, modes_message *out, size_t capacity);   /* like modes_set_output */
size_t modes_resolver_output_count(const modes_resolver *r);

/* decodeModesMessage() on frame bytes (the reference's hex door,
 * decodeHexMessage dump1090.c:2472-2502): CRC, fix and field decode run on the
 * device + resolve path with the context's ICAO cache. */
int  modes_decode_frame(modes_ctx *ctx, const uint8_t msg[14], modes_message *out);
/* n frames of 14 bytes each in one launch (device staging is kept by the context); decoded in
 * order, as n calls of modes_decode_frame would. */
int  modes_decode_frames(modes_ctx *ctx, const uint8_t *frames, size_t n, modes_message *out);

/* ---- presentation (SURVEY.md §8(f) item 1) -------------------------------- */
/* The reference's default (non --raw) text for one message: displayModesMessage()
 * (dump1090.c:1314-1450) plus the blank line of useModesMessage() (:1813), byte for byte.
 * check_crc = the --no-crc-check state (it changes one line, :1445).  Returns the length the text
 * needs; at most capacity-1 bytes + NUL are written.  Pure host code. */
size_t modes_format_message(const modes_message *mm, int check_crc, char *buf, size_t capacity);

/* SURVEY.md §8(f) item 2 — the raw TCP wire formats.  Output line of port 30002
 * (modesSendRawOutput, dump1090.c:2381-2393): "*" + UPPERCASE hex + ";\n". */
size_t modes_format_raw_net(const modes_message *mm, char *buf, size_t capacity);
/* Input line of port 30001, the parsing half of decodeHexMessage (dump1090.c:2472-2497).  Returns
 * the number of frame bytes written to msg (0..14; the rest zeroed) or -1 where the reference
 * discards the line.  Feed the bytes to modes_decode_frame() for the decoding half. */
int    modes_parse_hex_line(const char *line, uint8_t msg[14]);

/* ---- SURVEY.md §8(f) item 3 — aircraft tracker, CPR positions, SBS / JSON records -------------
 * The per-aircraft reduce over the delivered message stream that the reference's interactive
 * mode, HTTP map and SBS port share (dump1090.c:1822-2164).  Pure host code, no GPU involved.
 * Time is supplied by the caller in milliseconds: wall clock for a live feed (what the reference
 * uses, time()/mstime()), or stream time for a file: MODES_STREAM_EPOCH_MS + sample_pos / 2000.
 * The epoch matters: a new aircraft's odd/even CPR times start at 0, and the reference pairs two
 * frames when their times differ by <= 10 s (dump1090.c:2122) — with a clock that starts near 0
 * the first position frame of a file would be "paired" with the empty slot and decoded against
 * zeros.  mstime() is ~1.7e12, so the reference never does that; neither does a stream clock
 * that starts at the epoch below. */
#define MODES_STREAM_EPOCH_MS 1000000000000LL
typedef struct modes_tracker modes_tracker;

/* struct aircraft (dump1090.c:112-130) */
typedef struct modes_aircraft {
    uint32_t addr;                  /* ICAO address */
    char     hexaddr[7];            /* "%06x" */
    char     flight[9];
    int32_t  altitude, speed, track;
    int64_t  seen;                  /* seconds: now_ms / 1000 at the last message (time(NULL) in the reference) */
    int64_t  messages;
    int32_t  odd_cprlat, odd_cprlon, even_cprlat, even_cprlon;
    double   lat, lon;
    int64_t  odd_cprtime, even_cprtime;   /* ms (mstime() in the reference) */
} modes_aircraft;

/* check_crc: messages with crcok == 0 are ignored when set (dump1090.c:2073). */
modes_tracker *modes_tracker_create(int check_crc);
void   modes_tracker_destroy(modes_tracker *t);
/* interactiveReceiveData() (dump1090.c:2069-2164) incl. decodeCPR (:1952-1988), decodeCPRSurface
 * (:2004-2052), decodeMovementField (:2056-2066) and the receiver reference position.  Returns
 * the aircraft (valid until the next expire/destroy) or NULL when the message is ignored. */
const modes_aircraft *modes_tracker_update(modes_tracker *t, const modes_message *mm, int64_t now_ms);
size_t modes_tracker_count(const modes_tracker *t);
/* The aircraft in the reference's list order: most recently created first (dump1090.c:2080-2083). */
size_t modes_tracker_list(const modes_tracker *t, modes_aircraft *out, size_t capacity);
/* interactiveRemoveStaleAircrafts() (dump1090.c:2205-2229): drops aircraft not heard for more than
 * ttl_seconds; returns how many were removed. */
size_t modes_tracker_expire(modes_tracker *t, int64_t now_ms, int ttl_seconds);
/* Receiver reference position (running mean of decoded airborne positions, dump1090.c:2127-2141). */
void   modes_tracker_reference(const modes_tracker *t, double *lat, double *lon, int *count);
/* aircraftsToJson() (dump1090.c:2505-2551).  Returns the length needed; writes at most capacity-1 bytes + NUL. */
size_t modes_tracker_format_json(const modes_tracker *t, int metric, char *buf, size_t capacity);
/* The interactive-mode screen, interactiveShowData() (dump1090.c:2167-2199): clear-screen sequence,
 * header with the activity dot, one row per aircraft up to max_rows.  Same length convention. */
size_t modes_tracker_format_table(const modes_tracker *t, int metric, int max_rows, int64_t now_ms, char *buf, size_t capacity);
/* One SBS (BaseStation, port 30003) line for a message and its aircraft, modesSendSBSOutput()
 * (dump1090.c:2396-2446), newline included.  Returns the length needed, 0 for message types that
 * produce no line. */
size_t modes_format_sbs(const modes_message *mm, const modes_aircraft *a, char *buf, size_t capacity);
/* cprNLFunction (dump1090.c:1869-1931), exposed for tests. */
int    modes_cpr_nl(double lat);

/* ---- plumbing ----------------------------------------------------------- */
void *modes_stream(modes_ctx *ctx);                    /* the cudaStream_t modes_detect_device launches on */
int   modes_set_stream(modes_ctx *ctx, void *cuda_stream);   /* use the caller's stream for it (NULL: own) */
/* Device memory that other ranks on the same node can write into (CUDA IPC): rank 0 of a
 * multi-GPU job allocates the gather buffer with modes_device_alloc, exports it, and every other
 * rank maps it and passes its segment as d_candidates / d_tiles of modes_detect_device, so the
 * frame-evaluation kernel stores its records straight into rank 0's HBM over NVLink — the record
 * gather is fused into the kernel instead of following it as a collective. */
void *modes_device_alloc(size_t nbytes);
void  modes_device_free(void *p);
int   modes_ipc_export(const void *dptr, uint8_t handle[64]);
void *modes_ipc_open(const uint8_t handle[64]);          /* on the importing rank's current device */
int   modes_ipc_close(void *mapped);
int   modes_copy_to_host(void *dst_host, const void *src_device, size_t nbytes);   /* synchronous */
int   modes_device_memset(void *dst_device, int value, size_t nbytes);            /* synchronous */
/* Queue a device-to-device copy of the last modes_detect_device's counters {found, overflow,0,0}
 * (16 bytes) to `dst` (may be peer memory) on the detect stream. */
int   modes_detect_publish_count(modes_ctx *ctx, void *dst);
void *modes_host_alloc(size_t nbytes);                 /* pinned host memory for modes_process input */
void  modes_host_free(void *p);
/* cfg.profile: mean device time (CUDA events on the launching stream) per batch
 * since the previous call: [0] scan kernel (magnitude+preamble), [1] frame
 * evaluation kernel, [2] both, [3] number of batches averaged. */
int  modes_get_kernel_times(modes_ctx *ctx, float ms[4]);
/* Cumulative count of kernel launches issued by this context. */
uint64_t modes_launch_count(const modes_ctx *ctx);
/* How host threads wait for the GPU, process-wide (contexts read it when they are created).
 * 0 (default): the CUDA runtime's choice — on a many-core host it spins: lowest latency, one core
 * busy per waiting thread.  1: sleep until the GPU signals (cudaEventBlockingSync): for hosts that
 * run more GPU processes than they have cores to spare (e.g. one process per GPU under a small
 * container CPU quota).  The environment variable MODES_HOST_WAIT=block sets the initial value.
 * The helper threads that build message structs are sized from the CPUs this process may really
 * use (affinity mask cut down to the cgroup CPU quota); MODES_BUILD_THREADS=<n> overrides, e.g.
 * quota / ranks for several processes on one host. */
int  modes_set_host_wait(int mode);
/* Entries of the tile table of a batch of n_buffers reference buffers. */
size_t modes_tile_count(size_t n_buffers);

/* ---- many receivers on one GPU (SURVEY.md 8(f) item 4: batch across receivers, not across time) ----
 * One dump1090 process serves one RTL-SDR: rtlsdrCallback (dump1090.c:442-456) fills one buffer of
 * 131072 samples at a time, readDataFromFile/rtlsdrCallback prefix it with the last 238 samples of the
 * previous one (:481-485), and detectModeS keeps ONE address cache, skip state and set of statistics.
 * A pool keeps all of that per receiver for many independent 2 MHz streams and decodes one buffer of each
 * of them in ONE batch on the device (csrc/modes_pool.cpp: each buffer rides behind a resident pad buffer
 * whose tail is that receiver's carry, so the kernels are the single-stream ones).  Messages of a
 * receiver are delivered in its stream order with sample_pos counted in its own stream; receivers are
 * served in the order they are listed.  Every receiver's output equals a modes_ctx fed that receiver's
 * buffers alone.
 * cfg->gpu_resolve = 0 (default): each receiver's buffer is resolved on the host, by that receiver's own
 * modes_resolver, on MODES_POOL_THREADS threads (default 4).  cfg->gpu_resolve = 1: modes_pool_collect
 * resolves on the device, one warp per receiver, each receiver's address cache resident in device memory
 * (4 KiB per receiver); only the delivered messages' 40-byte records cross PCIe, and the host builds the
 * structs.  The output (messages, order, fields, sample_pos, receiver_of, statistics, buffers) is the same
 * byte for byte.  cfg->n_gpus is ignored: a pool uses `device` alone. */
typedef struct modes_pool modes_pool;
typedef void (*modes_pool_sink_fn)(void *user, uint32_t receiver, const modes_message *mm);
/* max_batch_receivers: most receivers one modes_pool_ingest call names (0: n_receivers); sizes the
 * resident batch (2 x 256 KiB per receiver).  No device is touched before the first modes_pool_ingest. */
modes_pool *modes_pool_create(const modes_config *cfg, size_t n_receivers, size_t max_batch_receivers);
void        modes_pool_destroy(modes_pool *p);
const char *modes_pool_last_error(const modes_pool *p);
/* iq[i]: the next MODES_BUFFER_BYTES of receiver receivers[i] (host memory, pinned for full speed); a
 * receiver may be named once per call and need not be named in every call. */
int  modes_pool_ingest(modes_pool *p, const uint32_t *receivers, const uint8_t *const *iq, size_t n,
                       modes_pool_sink_fn sink, void *user);
/* The two halves of modes_pool_ingest, for overlap: submit uploads the buffers and launches the kernels
 * and returns without waiting (the buffers must stay valid until the batch is collected); collect waits
 * for the OLDEST submitted batch, resolves it and delivers its messages.  Two batches may be in flight:
 *     submit(k+1); collect(k);      -- batch k+1 crosses PCIe and is scanned while batch k is resolved
 * A receiver may be named in both. */
int  modes_pool_submit(modes_pool *p, const uint32_t *receivers, const uint8_t *const *iq, size_t n);
int  modes_pool_collect(modes_pool *p, modes_pool_sink_fn sink, void *user);
/* The host half alone, for candidate records produced elsewhere over a batch laid out as the pool lays
 * it out: buffer 2i = pad buffer of receivers[i] (no signal, last MODES_CARRY_BYTES = its carry), buffer
 * 2i+1 = its new buffer; candidates/tiles as modes_detect_fetch returns them for those 2n buffers.
 * Fails on a pool created with gpu_resolve = 1, whose address caches live on the device. */
int  modes_pool_resolve(modes_pool *p, const uint32_t *receivers, size_t n, const modes_candidate *candidates,
                        const modes_tile *tiles, modes_pool_sink_fn sink, void *user);
/* Like modes_set_output: messages are ALSO written to a caller-owned array, all receivers' in delivery
 * order, receiver_of[k] naming the receiver of out[k]; the count keeps running past capacity, calling
 * it again restarts the array.  NULL, NULL, 0 turns it off.  The sink may then be NULL. */
int    modes_pool_set_output(modes_pool *p, modes_message *out, uint32_t *receiver_of, size_t capacity);
size_t modes_pool_output_count(const modes_pool *p);
int  modes_pool_stats(const modes_pool *p, uint32_t receiver, modes_stats *out);
int  modes_pool_reset(modes_pool *p, uint32_t receiver);        /* the receiver starts a new stream */
int64_t modes_pool_buffers(const modes_pool *p, uint32_t receiver);   /* buffers of it decoded so far */

#ifdef __cplusplus
}
#endif
#endif /* MODES_B200_H */
