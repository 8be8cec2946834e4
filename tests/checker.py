"""ctypes access to the checker libraries (oracle/ and oracle/_ref) for tests.

TEST INFRASTRUCTURE.  Only tests/, __graft_entry__.smoke() and bench.py import
this.  `libref` (the unmodified reference compiled into oracle/_ref/libref.so)
exists only where `make -C oracle ref` ran with the reference sources present.
The tests never need it: what they compare with was recorded from it into
tests/golden/ (tests/golden/make_reference_answers.py).
"""
from __future__ import annotations

import atexit
import ctypes
import gzip
import hashlib
import os
import subprocess
import tempfile
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
ORACLE_DIR = ROOT / "oracle"
REF_SO = ORACLE_DIR / "_ref" / "libref.so"
ORACLE_SO = ORACLE_DIR / "_build" / "libmodes_oracle.so"
REFERENCE_ROOT = Path("/root/reference")

_I32 = ("errorbit aa1 aa2 aa3 phase_corrected ca iid metype mesub heading_is_valid heading "
        "aircraft_type fflag tflag raw_latitude raw_longitude").split()
_I32B = ("ew_dir ew_velocity ns_dir ns_velocity vert_rate_source vert_rate_sign vert_rate velocity "
         "movement movement_valid ground_track ground_track_valid fs dr um identity altitude unit "
         "nfixed pad2").split()


class Msg(ctypes.Structure):
    """Layout of struct oracle_msg / modes_message_t (fields of dump1090.c:211-260)."""
    _fields_ = ([("msg", ctypes.c_uint8 * 14), ("pad0", ctypes.c_uint8 * 2),
                 ("msgbits", ctypes.c_int32), ("msgtype", ctypes.c_int32), ("crcok", ctypes.c_int32),
                 ("crc", ctypes.c_uint32)]
                + [(n, ctypes.c_int32) for n in _I32]
                + [("flight", ctypes.c_char * 9), ("pad1", ctypes.c_char * 3)]
                + [(n, ctypes.c_int32) for n in _I32B]
                + [("sample_pos", ctypes.c_int64)])

    def hexline(self) -> str:
        return "*" + bytes(self.msg[: self.msgbits // 8]).hex() + ";"


class Pass(ctypes.Structure):
    _fields_ = [("msg", ctypes.c_uint8 * 14), ("msgtype", ctypes.c_uint8), ("flags", ctypes.c_uint8),
                ("errorbit", ctypes.c_uint8), ("nfixed", ctypes.c_uint8), ("crc", ctypes.c_uint32)]


class Cand(ctypes.Structure):
    _fields_ = [("t", ctypes.c_int64), ("passes", Pass * 2)]


OP_GATE_OK, OP_ERRORS, OP_DECODED, OP_P2_VALID = 1, 2, 4, 8

# Which struct fields the reference actually assigns, per downlink format
# (SURVEY §8 a13: everything else is left uninitialised on the caller's stack).
COMMON_FIELDS = ["msgbits", "msgtype", "crcok", "crc", "errorbit", "aa1", "aa2", "aa3",
                 "phase_corrected", "ca", "iid", "metype", "mesub", "fs", "dr", "um", "identity"]


def defined_fields(m: Msg):
    f = list(COMMON_FIELDS)
    df = m.msgtype
    if df in (0, 4, 16, 20):
        f += ["altitude"]
        if not (bytes(m.msg)[3] & 0x40) or True:
            f += ["unit"]
    if df in (17, 18):
        t, s = m.metype, m.mesub
        if 1 <= t <= 4:
            f += ["aircraft_type", "flight"]
        elif 5 <= t <= 8:
            f += ["movement", "movement_valid", "ground_track_valid", "ground_track", "fflag", "tflag",
                  "raw_latitude", "raw_longitude"]
        elif 9 <= t <= 18:
            f += ["fflag", "tflag", "altitude", "raw_latitude", "raw_longitude"]
            if bytes(m.msg)[5] & 1:
                f += ["unit"]
        elif t == 19 and 1 <= s <= 4:
            if s in (1, 2):
                f += ["ew_dir", "ew_velocity", "ns_dir", "ns_velocity", "vert_rate_source",
                      "vert_rate_sign", "vert_rate", "velocity", "heading"]
            else:
                f += ["heading_is_valid", "heading"]
    return f


def msg_fields(m: Msg, with_pos: bool = False) -> dict:
    d = {"hex": bytes(m.msg[: m.msgbits // 8]).hex()}
    for name in defined_fields(m):
        v = getattr(m, name)
        d[name] = v.decode("latin1") if isinstance(v, bytes) else int(v)
    if with_pos:
        d["sample_pos"] = int(m.sample_pos)
    return d


def build_oracle() -> None:
    """Compile the CPU restatement (and, where the reference is mounted, oracle/_ref)."""
    subprocess.run(["make", "-C", str(ORACLE_DIR)], check=True, capture_output=True)
    if os.path.isdir(REFERENCE_ROOT):                 # False where it is absent or not readable
        subprocess.run(["make", "-C", str(ORACLE_DIR), "ref"], check=True, capture_output=True)


_libs = {}


def _load(path: Path):
    if path not in _libs:
        if not path.exists():
            build_oracle()
        _libs[path] = ctypes.CDLL(str(path))
    return _libs[path]


def oracle_lib():
    return _load(ORACLE_SO)


def ref_lib():
    return _load(REF_SO)


def _as_u8(data) -> np.ndarray:
    a = np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else data,
                             dtype=np.uint8)
    return a


def _decode(lib, fname, data, fix=1, aggressive=0, check_crc=1, drop_eof=0, cap=None):
    a = _as_u8(data)
    fn = getattr(lib, fname)
    fn.restype = ctypes.c_long
    cap = cap or max(4096, a.size // 200)
    out = (Msg * cap)()
    st = (ctypes.c_longlong * 8)()
    n = fn(a.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(a.size), int(fix), int(aggressive),
           int(check_crc), int(drop_eof), out, ctypes.c_size_t(cap), st)
    assert n <= cap, "message capacity too small"
    return [out[i] for i in range(n)], list(st)


def oracle_decode(data, **kw):
    return _decode(oracle_lib(), "oracle_decode", data, **kw)


def ref_decode(data, **kw):
    return _decode(ref_lib(), "ref_decode", data, **kw)


def oracle_scan_candidates(data, fix=1, aggressive=0, drop_eof=0, cap=None):
    a = _as_u8(data)
    lib = oracle_lib()
    lib.oracle_scan_candidates.restype = ctypes.c_long
    cap = cap or max(4096, a.size // 100)
    out = (Cand * cap)()
    n = lib.oracle_scan_candidates(a.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(a.size), int(fix),
                                   int(aggressive), int(drop_eof), out, ctypes.c_size_t(cap))
    assert n <= cap
    return [out[i] for i in range(n)]


def oracle_magnitude(iq) -> np.ndarray:
    a = _as_u8(iq)
    out = np.empty(a.size // 2, dtype=np.uint16)
    oracle_lib().oracle_magnitude(a.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(a.size // 2),
                                  out.ctypes.data_as(ctypes.c_void_p))
    return out


def _time(lib, fname, data, fix=1, aggressive=0, check_crc=1, loops=1):
    a = _as_u8(data)
    fn = getattr(lib, fname)
    fn.restype = ctypes.c_double
    st = (ctypes.c_longlong * 8)()
    return fn(a.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(a.size), int(fix), int(aggressive),
              int(check_crc), int(loops), st)


def oracle_time(data, **kw):
    return _time(oracle_lib(), "oracle_time_decode", data, **kw)


def ref_time(data, **kw):
    return _time(ref_lib(), "ref_time_decode", data, **kw)


def ref_time_phases(data, fix=1, aggressive=0, check_crc=1, loops=1):
    """(seconds in computeMagnitudeVector, seconds in detectModeS) of the unmodified reference."""
    a = _as_u8(data)
    fn = ref_lib().ref_time_phases
    fn.restype = None
    out = (ctypes.c_double * 2)()
    fn(a.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(a.size), int(fix), int(aggressive), int(check_crc),
       int(loops), out)
    return float(out[0]), float(out[1])


MODES1_SHA256 = "3a33e16025da8669149c780075950b4e908ca036ea21f9583c113f60d5fb3094"
_modes1_file = None


def modes1() -> np.ndarray:
    """The reference's sample capture testfiles/modes1.bin (713 736 bytes), kept gzipped with the tests."""
    data = np.frombuffer(gzip.decompress((ROOT / "tests" / "golden" / "modes1.bin.gz").read_bytes()), dtype=np.uint8).copy()
    assert hashlib.sha256(data.tobytes()).hexdigest() == MODES1_SHA256, "tests/golden/modes1.bin.gz is damaged"
    return data


def modes1_path() -> Path:
    """modes1() as a file, for programs that read a capture (--ifile): written once per process to a
    temporary file, removed at exit."""
    global _modes1_file
    if _modes1_file is None:
        fd, name = tempfile.mkstemp(suffix="_modes1.bin")
        with os.fdopen(fd, "wb") as f:
            f.write(modes1().tobytes())
        atexit.register(os.unlink, name)
        _modes1_file = Path(name)
    return _modes1_file


# ---- tracker door of the reference harness (SURVEY.md 8(f) item 3) -----------------------------

class Aircraft(ctypes.Structure):
    """struct oracle_aircraft (oracle/oracle_msg.h) == struct aircraft, dump1090.c:112-130."""
    _fields_ = [("addr", ctypes.c_uint32), ("hexaddr", ctypes.c_char * 7), ("flight", ctypes.c_char * 9),
                ("altitude", ctypes.c_int32), ("speed", ctypes.c_int32), ("track", ctypes.c_int32),
                ("seen", ctypes.c_int64), ("messages", ctypes.c_int64),
                ("odd_cprlat", ctypes.c_int32), ("odd_cprlon", ctypes.c_int32),
                ("even_cprlat", ctypes.c_int32), ("even_cprlon", ctypes.c_int32),
                ("lat", ctypes.c_double), ("lon", ctypes.c_double),
                ("odd_cprtime", ctypes.c_int64), ("even_cprtime", ctypes.c_int64)]

    def as_tuple(self):
        return (self.addr, self.hexaddr, self.flight, self.altitude, self.speed, self.track, self.seen, self.messages,
                self.odd_cprlat, self.odd_cprlon, self.even_cprlat, self.even_cprlon, self.lat, self.lon,
                self.odd_cprtime, self.even_cprtime)


class RefTracker:
    """The reference's own interactiveReceiveData / modesSendSBSOutput / aircraftsToJson, one
    message at a time with an explicit clock."""

    def __init__(self, check_crc=1):
        self.lib = ref_lib()
        self.lib.ref_track_reset(int(check_crc))
        self.lib.ref_track_list.restype = ctypes.c_long
        self.lib.ref_track_expire.restype = ctypes.c_long

    def update(self, msg, now_ms):
        """msg: any ctypes struct with the oracle_msg layout (Msg here, api.Message)."""
        m = Msg()
        ctypes.memmove(ctypes.byref(m), ctypes.byref(msg), ctypes.sizeof(Msg))
        a = Aircraft()
        sbs = ctypes.create_string_buffer(512)
        ok = self.lib.ref_track_update(ctypes.byref(m), ctypes.c_longlong(int(now_ms)), ctypes.byref(a), sbs)
        return (a, sbs.value.decode("latin1")) if ok else None

    def aircraft(self):
        arr = (Aircraft * 4096)()
        n = self.lib.ref_track_list(arr, 4096)
        return [arr[i] for i in range(n)]

    def expire(self, now_ms, ttl_seconds):
        return int(self.lib.ref_track_expire(ctypes.c_longlong(int(now_ms)), int(ttl_seconds)))

    def reference(self):
        lat, lon, cnt = ctypes.c_double(), ctypes.c_double(), ctypes.c_int()
        self.lib.ref_track_reference(ctypes.byref(lat), ctypes.byref(lon), ctypes.byref(cnt))
        return lat.value, lon.value, cnt.value

    def json(self, metric=0):
        buf = ctypes.create_string_buffer(1 << 20)
        n = self.lib.ref_track_json(int(metric), buf, 1 << 20)
        return buf.raw[:n].decode("latin1")

    def table(self, now_ms, metric=0, max_rows=15):
        return ref_track_table(now_ms, metric, max_rows)


def ref_track_table(now_ms, metric=0, max_rows=15):
    buf = ctypes.create_string_buffer(1 << 16)
    n = ref_lib().ref_track_table(int(metric), int(max_rows), ctypes.c_longlong(int(now_ms)), buf, 1 << 16)
    return buf.raw[:n].decode("latin1")


def ref_cpr_nl(lat):
    f = ref_lib().ref_cpr_nl
    f.restype = ctypes.c_int
    f.argtypes = [ctypes.c_double]
    return int(f(float(lat)))
