"""ctypes binding of include/modes_b200.h — the Python host side of the C ABI.

Mirrors the reference's main-loop contract (dump1090.c:2968-2990): a `Decoder`
is fed raw u8 I/Q bytes and hands back, in stream order, the messages the
reference would pass to useModesMessage() (dump1090.c:1802).  Everything that
computes runs in libmodes_b200.so (CUDA, sm_100a).  There is no CPU fallback:
constructing a Decoder without a usable GPU raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libmodes_b200.so"

BUFFER_BYTES = 262144
BUFFER_SAMPLES = 131072
CARRY_BYTES = 476
TILE_SAMPLES = 7936                       # MODES_TILE_SAMPLES
ICAO_CACHE_SLOTS = 1024                   # MODES_ICAO_CACHE_SLOTS
STREAM_EPOCH_MS = 1_000_000_000_000      # MODES_STREAM_EPOCH_MS: start of a file's stream clock for the tracker

EVAL_GATE_OK, EVAL_ERRORS, EVAL_DECODED, EVAL_P2_VALID = 1, 2, 4, 8


class Config(C.Structure):
    _fields_ = [("fix_errors", C.c_int32), ("aggressive", C.c_int32), ("check_crc", C.c_int32),
                ("drop_eof_buffer", C.c_int32), ("device", C.c_int32), ("profile", C.c_int32),
                ("max_batch_bytes", C.c_uint64), ("n_gpus", C.c_int32), ("gpu_resolve", C.c_int32)]


_MSG_A = ("errorbit aa1 aa2 aa3 phase_corrected ca iid metype mesub heading_is_valid heading "
          "aircraft_type fflag tflag raw_latitude raw_longitude").split()
_MSG_B = ("ew_dir ew_velocity ns_dir ns_velocity vert_rate_source vert_rate_sign vert_rate velocity "
          "movement movement_valid ground_track ground_track_valid fs dr um identity altitude unit "
          "nfixed pad2").split()


class Message(C.Structure):
    """struct modes_message == fields of struct modesMessage (dump1090.c:211-260)."""
    _fields_ = ([("msg", C.c_uint8 * 14), ("pad0", C.c_uint8 * 2), ("msgbits", C.c_int32),
                 ("msgtype", C.c_int32), ("crcok", C.c_int32), ("crc", C.c_uint32)]
                + [(n, C.c_int32) for n in _MSG_A]
                + [("flight", C.c_char * 9), ("pad1", C.c_char * 3)]
                + [(n, C.c_int32) for n in _MSG_B]
                + [("sample_pos", C.c_int64)])

    def hex(self) -> str:
        return bytes(self.msg[: self.msgbits // 8]).hex()

    def raw_line(self) -> str:
        """The --raw output line, dump1090.c:1324-1326."""
        return "*" + self.hex() + ";"

    def text(self, check_crc: int = 1) -> str:
        """The reference's default (non --raw) output for this message, dump1090.c:1314-1450."""
        buf = C.create_string_buffer(2048)
        n = lib().modes_format_message(C.byref(self), int(check_crc), buf, 2048)
        return buf.raw[:n].decode("latin1")

    def raw_net_line(self) -> str:
        """The TCP raw-output line (uppercase hex), dump1090.c:2381-2393."""
        buf = C.create_string_buffer(64)
        n = lib().modes_format_raw_net(C.byref(self), buf, 64)
        return buf.raw[:n].decode("latin1")

    def copy(self) -> "Message":
        m = Message()
        C.memmove(C.byref(m), C.byref(self), C.sizeof(Message))
        return m


class FrameEval(C.Structure):
    _fields_ = [("msg", C.c_uint8 * 14), ("msgtype", C.c_uint8), ("flags", C.c_uint8),
                ("errorbit", C.c_uint8), ("nfixed", C.c_uint8), ("crc", C.c_uint32)]


class Candidate(C.Structure):
    _fields_ = [("t", C.c_int64), ("passes", FrameEval * 2)]


class Tile(C.Structure):
    _fields_ = [("offset", C.c_uint32), ("count", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [("v", C.c_int64 * 8)]


STAT_NAMES = ["valid_preamble", "out_of_phase", "demodulated", "goodcrc", "badcrc", "fixed",
              "single_bit_fix", "two_bits_fix"]

SINK_FN = C.CFUNCTYPE(None, C.c_void_p, C.POINTER(Message))
POOL_SINK_FN = C.CFUNCTYPE(None, C.c_void_p, C.c_uint32, C.POINTER(Message))

CANDIDATE_DTYPE = np.dtype([("t", "<i8"),
                            ("p", [("msg", "u1", 14), ("msgtype", "u1"), ("flags", "u1"), ("errorbit", "u1"),
                                   ("nfixed", "u1"), ("crc", "<u4")], 2)], align=True)
TILE_DTYPE = np.dtype([("offset", "<u4"), ("count", "<u4")])
assert CANDIDATE_DTYPE.itemsize == C.sizeof(Candidate) == 56

_lib = None

# every symbol include/modes_b200.h declares
EXPORTS = ["modes_abi_version", "modes_default_config", "modes_create", "modes_destroy", "modes_last_error",
           "modes_set_sink", "modes_process", "modes_finish", "modes_reset", "modes_get_stats",
           "modes_compute_magnitude", "modes_detect_device", "modes_detect_host", "modes_detect_wait", "modes_detect_fetch",
           "modes_resolve", "modes_resolver_create", "modes_resolver_destroy", "modes_resolver_run",
           "modes_resolver_run_shards", "modes_resolver_get_cache", "modes_resolver_set_cache", "modes_resolver_tail_cache", "modes_resolver_run_tentative", "modes_resolver_commit", "modes_resolver_reset", "modes_resolver_stats", "modes_resolver_set_output", "modes_resolver_output_count", "modes_decode_frame", "modes_decode_frames", "modes_format_message", "modes_format_raw_net", "modes_parse_hex_line", "modes_stream", "modes_set_stream",
           "modes_set_output", "modes_output_count", "modes_device_alloc", "modes_device_free",
           "modes_ipc_export", "modes_ipc_open", "modes_ipc_close", "modes_copy_to_host", "modes_device_memset",
           "modes_detect_publish_count", "modes_host_alloc",
           "modes_host_free", "modes_get_kernel_times", "modes_launch_count", "modes_tile_count", "modes_set_host_wait",
           "modes_tracker_create", "modes_tracker_destroy", "modes_tracker_update", "modes_tracker_count",
           "modes_tracker_list", "modes_tracker_expire", "modes_tracker_reference", "modes_tracker_format_json",
           "modes_tracker_format_table", "modes_format_sbs", "modes_cpr_nl",
           "modes_pool_create", "modes_pool_destroy", "modes_pool_last_error", "modes_pool_ingest", "modes_pool_resolve",
           "modes_pool_stats", "modes_pool_reset", "modes_pool_buffers", "modes_pool_set_output", "modes_pool_output_count",
           "modes_pool_submit", "modes_pool_collect"]


def lib():
    """Load libmodes_b200.so (built in-tree by `make` / __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise RuntimeError(f"{LIB_PATH} is missing: build it with `make` (no CPU fallback exists)")
        L = C.CDLL(str(LIB_PATH))
        L.modes_create.restype = C.c_void_p
        L.modes_create.argtypes = [C.POINTER(Config)]
        L.modes_destroy.argtypes = [C.c_void_p]
        L.modes_last_error.restype = C.c_char_p
        L.modes_last_error.argtypes = [C.c_void_p]
        L.modes_set_sink.argtypes = [C.c_void_p, SINK_FN, C.c_void_p]
        L.modes_process.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.modes_finish.argtypes = [C.c_void_p]
        L.modes_reset.argtypes = [C.c_void_p]
        L.modes_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
        L.modes_compute_magnitude.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.modes_detect_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                          C.c_size_t, C.c_void_p]
        L.modes_detect_host.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                        C.c_size_t, C.c_void_p]
        L.modes_detect_wait.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
        L.modes_detect_fetch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.modes_resolve.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int64]
        L.modes_resolver_create.restype = C.c_void_p
        L.modes_resolver_create.argtypes = [C.POINTER(Config)]
        L.modes_resolver_destroy.argtypes = [C.c_void_p]
        L.modes_resolver_run.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int64, SINK_FN,
                                         C.c_void_p]
        L.modes_resolver_run_shards.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.c_void_p, SINK_FN, C.c_void_p]
        L.modes_resolver_reset.argtypes = [C.c_void_p]
        L.modes_resolver_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
        L.modes_resolver_set_output.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.modes_resolver_output_count.restype = C.c_size_t
        L.modes_resolver_output_count.argtypes = [C.c_void_p]
        L.modes_decode_frame.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Message)]
        L.modes_format_message.restype = C.c_size_t
        L.modes_format_message.argtypes = [C.POINTER(Message), C.c_int, C.c_char_p, C.c_size_t]
        L.modes_format_raw_net.restype = C.c_size_t
        L.modes_format_raw_net.argtypes = [C.POINTER(Message), C.c_char_p, C.c_size_t]
        L.modes_parse_hex_line.argtypes = [C.c_char_p, C.c_void_p]
        L.modes_stream.restype = C.c_void_p
        L.modes_stream.argtypes = [C.c_void_p]
        L.modes_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        L.modes_set_output.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.modes_output_count.restype = C.c_size_t
        L.modes_output_count.argtypes = [C.c_void_p]
        L.modes_device_alloc.restype = C.c_void_p
        L.modes_device_alloc.argtypes = [C.c_size_t]
        L.modes_device_free.argtypes = [C.c_void_p]
        L.modes_ipc_export.argtypes = [C.c_void_p, C.c_void_p]
        L.modes_ipc_open.restype = C.c_void_p
        L.modes_ipc_open.argtypes = [C.c_void_p]
        L.modes_ipc_close.argtypes = [C.c_void_p]
        L.modes_detect_publish_count.argtypes = [C.c_void_p, C.c_void_p]
        L.modes_copy_to_host.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.modes_device_memset.argtypes = [C.c_void_p, C.c_int, C.c_size_t]
        L.modes_host_alloc.restype = C.c_void_p
        L.modes_host_alloc.argtypes = [C.c_size_t]
        L.modes_host_free.argtypes = [C.c_void_p]
        L.modes_get_kernel_times.argtypes = [C.c_void_p, C.POINTER(C.c_float * 4)]
        L.modes_launch_count.restype = C.c_uint64
        L.modes_launch_count.argtypes = [C.c_void_p]
        L.modes_resolver_get_cache.argtypes = [C.c_void_p, C.c_void_p]
        L.modes_resolver_set_cache.argtypes = [C.c_void_p, C.c_void_p]
        L.modes_resolver_tail_cache.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int64, C.c_size_t, C.c_void_p]
        L.modes_resolver_run_tentative.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int64]
        L.modes_resolver_commit.argtypes = [C.c_void_p, SINK_FN, C.c_void_p]
        L.modes_tile_count.restype = C.c_size_t
        L.modes_tile_count.argtypes = [C.c_size_t]
        L.modes_pool_create.restype = C.c_void_p
        L.modes_pool_create.argtypes = [C.POINTER(Config), C.c_size_t, C.c_size_t]
        L.modes_pool_destroy.argtypes = [C.c_void_p]
        L.modes_pool_last_error.restype = C.c_char_p
        L.modes_pool_last_error.argtypes = [C.c_void_p]
        L.modes_pool_ingest.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, POOL_SINK_FN, C.c_void_p]
        L.modes_pool_submit.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
        L.modes_pool_collect.argtypes = [C.c_void_p, POOL_SINK_FN, C.c_void_p]
        L.modes_pool_resolve.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, POOL_SINK_FN, C.c_void_p]
        L.modes_pool_stats.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(Stats)]
        L.modes_pool_reset.argtypes = [C.c_void_p, C.c_uint32]
        L.modes_pool_set_output.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
        L.modes_pool_output_count.restype = C.c_size_t
        L.modes_pool_output_count.argtypes = [C.c_void_p]
        L.modes_pool_buffers.restype = C.c_int64
        L.modes_pool_buffers.argtypes = [C.c_void_p, C.c_uint32]
        _lib = L
    return _lib


def parse_hex_line(line: str | bytes):
    """decodeHexMessage's parser (dump1090.c:2472-2497): frame bytes, or None if the line is discarded."""
    if isinstance(line, str):
        line = line.encode("latin1")
    msg = (C.c_uint8 * 14)()
    n = lib().modes_parse_hex_line(line, msg)
    return None if n < 0 else bytes(msg)


def make_config(fix_errors=1, aggressive=0, check_crc=1, drop_eof_buffer=0, device=0, profile=0,
                max_batch_bytes=0, n_gpus=0, gpu_resolve=0) -> Config:
    cfg = Config()
    lib().modes_default_config(C.byref(cfg))
    cfg.fix_errors, cfg.aggressive, cfg.check_crc = int(fix_errors), int(aggressive), int(check_crc)
    cfg.drop_eof_buffer, cfg.device, cfg.profile = int(drop_eof_buffer), int(device), int(profile)
    if max_batch_bytes:
        cfg.max_batch_bytes = int(max_batch_bytes)
    cfg.n_gpus = int(n_gpus)
    cfg.gpu_resolve = int(gpu_resolve)
    return cfg


def tiles_for(n_buffers: int) -> int:
    """Entries of the tile table of a batch of n_buffers reference buffers (modes_tile_count)."""
    return int(lib().modes_tile_count(int(n_buffers)))


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


class _Collector:
    """A sink that copies every delivered message."""

    def __init__(self):
        self.messages: list[Message] = []
        self.fn = SINK_FN(self._on)

    def _on(self, _user, mm):
        self.messages.append(mm.contents.copy())


class PinnedBuffer:
    """Page-locked host memory (modes_host_alloc) exposed as a numpy u8 array."""

    def __init__(self, nbytes: int):
        self.ptr = lib().modes_host_alloc(nbytes)
        if not self.ptr:
            raise MemoryError("modes_host_alloc failed")
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(self.ptr))

    def free(self):
        if self.ptr:
            lib().modes_host_free(self.ptr)
            self.ptr = None
            self.array = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Decoder:
    """One GPU decode context (modes_create ... modes_destroy)."""

    def __init__(self, **cfg):
        self.cfg = make_config(**cfg)
        self._h = lib().modes_create(C.byref(self.cfg))
        if not self._h:
            raise RuntimeError("modes_create failed: " + lib().modes_last_error(None).decode())
        self._collector = _Collector()
        lib().modes_set_sink(self._h, self._collector.fn, None)

    # -- lifecycle
    def close(self):
        if self._h:
            lib().modes_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError(lib().modes_last_error(self._h).decode())

    # -- streaming path (the --ifile main loop)
    def process(self, data) -> None:
        a = np.ascontiguousarray(data, dtype=np.uint8) if not isinstance(data, (bytes, bytearray)) \
            else np.frombuffer(data, dtype=np.uint8)
        self._check(lib().modes_process(self._h, _ptr(a), a.size))

    def process_ptr(self, ptr: int, nbytes: int) -> None:
        self._check(lib().modes_process(self._h, C.c_void_p(ptr), nbytes))

    def finish(self) -> None:
        self._check(lib().modes_finish(self._h))

    def reset(self) -> None:
        self._check(lib().modes_reset(self._h))
        self._collector.messages = []

    def take_messages(self) -> list:
        out, self._collector.messages = self._collector.messages, []
        return out

    def decode(self, data, chunk: int | None = None) -> list:
        """Decode a whole stream like `dump1090 --ifile`: returns the message list."""
        self.reset()
        a = np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else \
            np.ascontiguousarray(data, dtype=np.uint8)
        if chunk:
            for off in range(0, a.size, chunk):
                self.process(a[off: off + chunk])
        else:
            self.process(a)
        self.finish()
        return self.take_messages()

    def set_output_array(self, capacity: int):
        """Deliver messages into a preallocated array instead of the Python callback
        (no per-message interpreter work).  Returns the ctypes array; capacity 0 restores the callback."""
        if capacity <= 0:
            self._out = None
            lib().modes_set_output(self._h, None, 0)
            lib().modes_set_sink(self._h, self._collector.fn, None)
            return None
        self._out = (Message * capacity)()
        lib().modes_set_sink(self._h, C.cast(None, SINK_FN), None)
        lib().modes_set_output(self._h, self._out, capacity)
        return self._out

    def rearm_output(self) -> None:
        lib().modes_set_output(self._h, self._out, len(self._out))

    def output_count(self) -> int:
        return int(lib().modes_output_count(self._h))

    def set_stream(self, cuda_stream: int) -> None:
        self._check(lib().modes_set_stream(self._h, C.c_void_p(cuda_stream)))

    def stats(self) -> dict:
        st = Stats()
        self._check(lib().modes_get_stats(self._h, C.byref(st)))
        return dict(zip(STAT_NAMES, [int(x) for x in st.v]))

    # -- stage-level entry points
    def magnitude(self, iq: np.ndarray) -> np.ndarray:
        a = np.ascontiguousarray(iq, dtype=np.uint8)
        out = np.empty(a.size // 2, dtype=np.uint16)
        self._check(lib().modes_compute_magnitude(self._h, _ptr(a), a.size // 2, _ptr(out)))
        return out

    def detect_device(self, d_iq_ptr: int, n_buffers: int, carry: bytes | None = None,
                      d_candidates_ptr: int = 0, cand_capacity: int = 0, d_tiles_ptr: int = 0) -> None:
        carr = None
        if carry is not None:
            assert len(carry) == CARRY_BYTES
            carr = (C.c_uint8 * CARRY_BYTES).from_buffer_copy(carry)
        self._check(lib().modes_detect_device(self._h, C.c_void_p(d_iq_ptr), n_buffers, carr,
                                              C.c_void_p(d_candidates_ptr), cand_capacity,
                                              C.c_void_p(d_tiles_ptr)))

    def detect_host(self, host_ptr: int, n_buffers: int, carry: bytes | None = None,
                    d_candidates_ptr: int = 0, cand_capacity: int = 0, d_tiles_ptr: int = 0) -> None:
        carr = (C.c_uint8 * CARRY_BYTES).from_buffer_copy(carry) if carry is not None else None
        self._check(lib().modes_detect_host(self._h, C.c_void_p(host_ptr), n_buffers, carr,
                                            C.c_void_p(d_candidates_ptr), cand_capacity, C.c_void_p(d_tiles_ptr)))

    def detect_wait(self) -> int:
        n = C.c_uint64(0)
        self._check(lib().modes_detect_wait(self._h, C.byref(n)))
        return int(n.value)

    def detect_fetch(self, n_buffers: int):
        n = self.detect_wait()
        cands = np.zeros(max(n, 1), dtype=CANDIDATE_DTYPE)
        tiles = np.zeros(tiles_for(n_buffers), dtype=TILE_DTYPE)
        self._check(lib().modes_detect_fetch(self._h, _ptr(cands), _ptr(tiles)))
        return cands[:n], tiles

    def detect_fetch_into(self, cands: np.ndarray, tiles: np.ndarray):
        """Like detect_fetch, into caller-owned arrays (pinned memory for full PCIe speed); returns views."""
        n = self.detect_wait()
        if n > cands.size:
            raise RuntimeError(f"record buffer too small: {n} > {cands.size}")
        self._check(lib().modes_detect_fetch(self._h, _ptr(cands), _ptr(tiles)))
        return cands[:n], tiles

    def resolve(self, cands: np.ndarray, tiles: np.ndarray, buffer_base: int = 0) -> None:
        self._check(lib().modes_resolve(self._h, _ptr(np.ascontiguousarray(cands)), _ptr(np.ascontiguousarray(tiles)),
                                        tiles.size, buffer_base))

    def decode_frame(self, frame: bytes) -> Message:
        buf = (C.c_uint8 * 14)(*(list(frame) + [0] * (14 - len(frame))))
        m = Message()
        self._check(lib().modes_decode_frame(self._h, buf, C.byref(m)))
        return m

    def decode_frames(self, frames) -> list:
        """A batch of frames (each padded to 14 bytes) through the hex door in one launch."""
        n = len(frames)
        buf = (C.c_uint8 * (14 * n))(*[b for f in frames for b in (list(f) + [0] * (14 - len(f)))])
        out = (Message * n)()
        self._check(lib().modes_decode_frames(self._h, buf, n, out))
        return [out[i] for i in range(n)]

    def publish_count(self, dst_ptr: int) -> None:
        self._check(lib().modes_detect_publish_count(self._h, C.c_void_p(dst_ptr)))

    def kernel_times_ms(self):
        t = (C.c_float * 4)()
        lib().modes_get_kernel_times(self._h, C.byref(t))
        return [float(x) for x in t]

    def launch_count(self) -> int:
        return int(lib().modes_launch_count(self._h))

    @property
    def stream(self) -> int:
        return int(lib().modes_stream(self._h) or 0)


class Resolver:
    """The sequential half alone (no device): modes_resolver_*."""

    def __init__(self, **cfg):
        self.cfg = make_config(**cfg)
        self._h = lib().modes_resolver_create(C.byref(self.cfg))
        self._collector = _Collector()

    def run(self, cands: np.ndarray, tiles: np.ndarray, buffer_base: int = 0) -> None:
        cands = np.ascontiguousarray(cands)
        tiles = np.ascontiguousarray(tiles)
        fn = C.cast(None, SINK_FN) if getattr(self, "_native", False) else self._collector.fn
        rc = lib().modes_resolver_run(self._h, _ptr(cands), _ptr(tiles), tiles.size, buffer_base, fn, None)
        if rc:
            raise RuntimeError("modes_resolver_run failed")

    def reset_state(self) -> None:
        lib().modes_resolver_reset(self._h)

    def run_shards(self, shards) -> None:
        """shards: [(cands ndarray, tiles ndarray, buffer_base)] in stream order; resolved concurrently."""
        n = len(shards)
        keep = [(np.ascontiguousarray(c), np.ascontiguousarray(t)) for c, t, _ in shards]
        cp = (C.c_void_p * n)(*[c.ctypes.data for c, _ in keep])
        tp = (C.c_void_p * n)(*[t.ctypes.data for _, t in keep])
        nt = (C.c_size_t * n)(*[t.size for _, t in keep])
        bb = (C.c_int64 * n)(*[int(b) for _, _, b in shards])
        fn = C.cast(None, SINK_FN) if getattr(self, "_native", False) else self._collector.fn
        if lib().modes_resolver_run_shards(self._h, n, cp, tp, nt, bb, fn, None):
            raise RuntimeError("modes_resolver_run_shards failed")

    # ---- one shard of a sharded decode (see include/modes_b200.h and sharded.resolve_distributed)
    def get_cache(self) -> np.ndarray:
        out = np.zeros(ICAO_CACHE_SLOTS, dtype=np.uint32)
        lib().modes_resolver_get_cache(self._h, _ptr(out))
        return out

    def set_cache(self, cache=None) -> None:
        c = None if cache is None else np.ascontiguousarray(cache, dtype=np.uint32)
        lib().modes_resolver_set_cache(self._h, None if c is None else _ptr(c))

    def tail_cache(self, cands: np.ndarray, tiles: np.ndarray, buffer_base: int = 0, n_tail_tiles: int | None = None) -> np.ndarray:
        out = np.zeros(ICAO_CACHE_SLOTS, dtype=np.uint32)
        if n_tail_tiles is None:
            n_tail_tiles = max(tiles.size // 16, 128)
        if lib().modes_resolver_tail_cache(self._h, _ptr(cands), _ptr(tiles), tiles.size, buffer_base, n_tail_tiles, _ptr(out)):
            raise RuntimeError("modes_resolver_tail_cache failed")
        return out

    def run_tentative(self, cands: np.ndarray, tiles: np.ndarray, buffer_base: int = 0) -> None:
        self._held = (cands, tiles)                       # the records must outlive the commit
        if lib().modes_resolver_run_tentative(self._h, _ptr(cands), _ptr(tiles), tiles.size, buffer_base):
            raise RuntimeError("modes_resolver_run_tentative failed")

    def commit(self) -> None:
        fn = C.cast(None, SINK_FN) if getattr(self, "_native", False) else self._collector.fn
        if lib().modes_resolver_commit(self._h, fn, None):
            raise RuntimeError("modes_resolver_commit without a tentative run")
        self._held = None

    def take_messages(self):
        out, self._collector.messages = self._collector.messages, []
        return out

    def set_output_array(self, capacity: int):
        """Fill a preallocated array in place instead of calling back into Python per message."""
        self._out = (Message * capacity)() if capacity > 0 else None
        self._native = capacity > 0
        lib().modes_resolver_set_output(self._h, self._out, max(capacity, 0))
        return self._out

    def rearm_output(self) -> None:
        lib().modes_resolver_set_output(self._h, self._out, len(self._out))

    def output_count(self) -> int:
        return int(lib().modes_resolver_output_count(self._h))

    def stats(self) -> dict:
        st = Stats()
        lib().modes_resolver_stats(self._h, C.byref(st))
        return dict(zip(STAT_NAMES, [int(x) for x in st.v]))

    def close(self):
        if self._h:
            lib().modes_resolver_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- SURVEY.md 8(f) item 4: many receivers on one GPU ----------------------------------------

class ReceiverPool:
    """modes_pool_*: independent 2 MHz streams (one address cache, carry, skip state and set of
    statistics each, as one dump1090 process keeps per receiver), one buffer of each decoded per
    batch.  Messages are collected per receiver (`take(receiver)`).

    gpu_resolve=1 (a make_config field, like fix_errors): the order-dependent half (skip / retry,
    address caches, statistics) runs on the device at collect(), one warp per receiver with every
    receiver's cache resident in device memory, and only the delivered messages' 40-byte records come
    back.  The output is the same as with gpu_resolve=0, byte for byte; resolve() (the host half alone)
    is then refused."""

    def __init__(self, n_receivers: int, max_batch: int = 0, **cfg):
        self.cfg = make_config(**cfg)
        self.n = n_receivers
        self._h = lib().modes_pool_create(C.byref(self.cfg), n_receivers, max_batch)
        if not self._h:
            raise RuntimeError("modes_pool_create failed")
        self.messages = [[] for _ in range(n_receivers)]
        self._fn = POOL_SINK_FN(self._on)

    def _on(self, _user, receiver, mm):
        self.messages[receiver].append(mm.contents.copy())

    def _check(self, rc):
        if rc:
            raise RuntimeError(lib().modes_pool_last_error(self._h).decode())

    def ingest(self, receivers, buffers) -> None:
        """buffers[i]: BUFFER_BYTES of uint8 I/Q (numpy) = the next buffer of receivers[i]."""
        ids = np.ascontiguousarray(receivers, dtype=np.uint32)
        bufs = [np.ascontiguousarray(b, dtype=np.uint8) for b in buffers]
        assert ids.size == len(bufs) and all(b.size == BUFFER_BYTES for b in bufs)
        ptrs = (C.c_void_p * len(bufs))(*[b.ctypes.data for b in bufs])
        self._check(lib().modes_pool_ingest(self._h, _ptr(ids), ptrs, ids.size, self._fn, None))

    def ingest_ptrs(self, receivers: np.ndarray, ptrs, sink=None) -> None:
        """The same from raw host addresses (pinned memory); sink: a POOL_SINK_FN or None to drop the messages."""
        fn = sink if sink is not None else C.cast(None, POOL_SINK_FN)
        self._check(lib().modes_pool_ingest(self._h, _ptr(receivers), ptrs, receivers.size, fn, None))

    def submit(self, receivers, buffers) -> None:
        """Upload + kernels, no waiting; `buffers` are kept alive until the matching collect()."""
        ids = np.ascontiguousarray(receivers, dtype=np.uint32)
        bufs = [np.ascontiguousarray(b, dtype=np.uint8) for b in buffers]
        assert ids.size == len(bufs) and all(b.size == BUFFER_BYTES for b in bufs)
        ptrs = (C.c_void_p * len(bufs))(*[b.ctypes.data for b in bufs])
        self._check(lib().modes_pool_submit(self._h, _ptr(ids), ptrs, ids.size))
        self._inflight = getattr(self, "_inflight", []) + [(ids, bufs)]

    def submit_ptrs(self, receivers: np.ndarray, ptrs) -> None:
        self._check(lib().modes_pool_submit(self._h, _ptr(receivers), ptrs, receivers.size))

    def collect(self, sink="collect") -> None:
        """Wait for the oldest submitted batch, resolve it, deliver its messages (sink=None: only to the output array)."""
        fn = self._fn if sink == "collect" else (sink if sink is not None else C.cast(None, POOL_SINK_FN))
        self._check(lib().modes_pool_collect(self._h, fn, None))
        if getattr(self, "_inflight", None):
            self._inflight.pop(0)

    def resolve(self, receivers, cands: np.ndarray, tiles: np.ndarray) -> None:
        """The host half alone over records of a batch laid out pad, data, pad, data, ..."""
        ids = np.ascontiguousarray(receivers, dtype=np.uint32)
        cands = np.ascontiguousarray(cands); tiles = np.ascontiguousarray(tiles)
        assert tiles.size == tiles_for(2 * ids.size)
        self._check(lib().modes_pool_resolve(self._h, _ptr(ids), ids.size, _ptr(cands), _ptr(tiles), self._fn, None))

    def take(self, receiver: int) -> list:
        out, self.messages[receiver] = self.messages[receiver], []
        return out

    def set_output_array(self, capacity: int):
        """Messages of all receivers into one array (+ the receiver of each), restarted by rearm_output()."""
        self._out = (Message * capacity)()
        self._out_rx = np.zeros(capacity, dtype=np.uint32)
        self._check(lib().modes_pool_set_output(self._h, C.addressof(self._out), _ptr(self._out_rx), capacity))
        return self._out, self._out_rx

    def rearm_output(self) -> None:
        self._check(lib().modes_pool_set_output(self._h, C.addressof(self._out), _ptr(self._out_rx), len(self._out)))

    def output_count(self) -> int:
        return int(lib().modes_pool_output_count(self._h))

    def stats(self, receiver: int) -> dict:
        st = Stats()
        lib().modes_pool_stats(self._h, receiver, C.byref(st))
        return dict(zip(STAT_NAMES, [int(x) for x in st.v]))

    def buffers(self, receiver: int) -> int:
        return int(lib().modes_pool_buffers(self._h, receiver))

    def reset(self, receiver: int) -> None:
        lib().modes_pool_reset(self._h, receiver)
        self.messages[receiver] = []

    def close(self):
        if self._h:
            lib().modes_pool_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- SURVEY.md 8(f) item 3: aircraft tracker (host only) -------------------------------------

class Aircraft(C.Structure):
    """struct modes_aircraft == struct aircraft (dump1090.c:112-130)."""
    _fields_ = [("addr", C.c_uint32), ("hexaddr", C.c_char * 7), ("flight", C.c_char * 9),
                ("altitude", C.c_int32), ("speed", C.c_int32), ("track", C.c_int32),
                ("seen", C.c_int64), ("messages", C.c_int64),
                ("odd_cprlat", C.c_int32), ("odd_cprlon", C.c_int32), ("even_cprlat", C.c_int32), ("even_cprlon", C.c_int32),
                ("lat", C.c_double), ("lon", C.c_double), ("odd_cprtime", C.c_int64), ("even_cprtime", C.c_int64)]

    def as_tuple(self):
        return (self.addr, self.hexaddr, self.flight, self.altitude, self.speed, self.track, self.seen, self.messages,
                self.odd_cprlat, self.odd_cprlon, self.even_cprlat, self.even_cprlon, self.lat, self.lon,
                self.odd_cprtime, self.even_cprtime)


class Tracker:
    """Per-aircraft state over a delivered message stream: the reference's interactiveReceiveData
    with CPR position decoding, plus the SBS and JSON record formats.  Needs no GPU."""

    def __init__(self, check_crc: int = 1):
        L = lib()
        L.modes_tracker_create.restype = C.c_void_p
        L.modes_tracker_update.restype = C.POINTER(Aircraft)
        L.modes_tracker_update.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
        L.modes_tracker_count.restype = C.c_size_t
        L.modes_tracker_count.argtypes = [C.c_void_p]
        L.modes_tracker_list.restype = C.c_size_t
        L.modes_tracker_list.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.modes_tracker_expire.restype = C.c_size_t
        L.modes_tracker_expire.argtypes = [C.c_void_p, C.c_int64, C.c_int]
        L.modes_tracker_reference.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.modes_tracker_format_json.restype = C.c_size_t
        L.modes_tracker_format_json.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]
        L.modes_tracker_destroy.argtypes = [C.c_void_p]
        L.modes_format_sbs.restype = C.c_size_t
        L.modes_format_sbs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
        self._h = L.modes_tracker_create(int(check_crc))
        if not self._h:
            raise MemoryError("modes_tracker_create failed")

    def update(self, msg: "Message", now_ms: int):
        """Returns (Aircraft copy, SBS line) or None when the message is ignored."""
        p = lib().modes_tracker_update(self._h, C.byref(msg), int(now_ms))
        if not p:
            return None
        buf = C.create_string_buffer(512)
        n = lib().modes_format_sbs(C.byref(msg), p, buf, 512)
        a = Aircraft()
        C.memmove(C.byref(a), p, C.sizeof(Aircraft))
        return a, buf.raw[:n].decode("latin1")

    def aircraft(self):
        n = lib().modes_tracker_count(self._h)
        arr = (Aircraft * max(n, 1))()
        lib().modes_tracker_list(self._h, arr, n)
        return [arr[i] for i in range(n)]

    def expire(self, now_ms: int, ttl_seconds: int) -> int:
        return int(lib().modes_tracker_expire(self._h, int(now_ms), int(ttl_seconds)))

    def reference(self):
        lat, lon, cnt = C.c_double(), C.c_double(), C.c_int()
        lib().modes_tracker_reference(self._h, C.byref(lat), C.byref(lon), C.byref(cnt))
        return lat.value, lon.value, cnt.value

    def json(self, metric: int = 0) -> str:
        need = lib().modes_tracker_format_json(self._h, int(metric), None, 0)
        buf = C.create_string_buffer(need + 1)
        lib().modes_tracker_format_json(self._h, int(metric), buf, need + 1)
        return buf.raw[:need].decode("latin1")

    def table(self, now_ms: int, metric: int = 0, max_rows: int = 15) -> str:
        """The interactive-mode screen, dump1090.c:2167-2199."""
        f = lib().modes_tracker_format_table
        f.restype = C.c_size_t
        f.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_size_t]
        need = f(self._h, int(metric), int(max_rows), int(now_ms), None, 0)
        buf = C.create_string_buffer(need + 1)
        f(self._h, int(metric), int(max_rows), int(now_ms), buf, need + 1)
        return buf.raw[:need].decode("latin1")

    def close(self):
        if self._h:
            lib().modes_tracker_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def cpr_nl(lat: float) -> int:
    f = lib().modes_cpr_nl
    f.restype = C.c_int
    f.argtypes = [C.c_double]
    return int(f(float(lat)))
