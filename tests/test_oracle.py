"""CPU (-m "not gpu"): pin the oracle restatement against the reference and the golden fixtures."""
import ctypes
import hashlib

import numpy as np
import pytest

import checker as C
import golden_util as G
from dump1090_b200 import synth

FLAG_SETS = [dict(), dict(aggressive=1), dict(fix=0), dict(check_crc=0), dict(check_crc=0, aggressive=1),
             dict(drop_eof=1), dict(fix=0, drop_eof=1), dict(check_crc=0, aggressive=1, drop_eof=1)]

# SURVEY.md §4 / BASELINE.md §2: line count and md5 of the --raw output of the reference on modes1.bin
MODES1_PINS = {
    (): (284, "4a81758c8bec"), (("drop_eof", 1),): (217, "7b1719f22374"),
    (("aggressive", 1),): (284, "4a81758c8bec"), (("fix", 0),): (283, "ac539444a66e"),
    (("drop_eof", 1), ("fix", 0)): (217, "a76c3fc95b9a"), (("check_crc", 0),): (765, "a6092d178fcf"),
    (("aggressive", 1), ("check_crc", 0)): (824, "bec25488d6b8"),
    (("aggressive", 1), ("check_crc", 0), ("drop_eof", 1)): (629, "16e26b0aa79f"),
}


def _md5_lines(msgs):
    return hashlib.md5("".join(m.hexline() + "\n" for m in msgs).encode()).hexdigest()[:12]


def _fields(msgs):
    return [C.msg_fields(m) for m in msgs]


@pytest.mark.parametrize("kw", FLAG_SETS, ids=str)
def test_oracle_modes1_pins(kw, checker_libs):
    msgs, _ = C.oracle_decode(C.modes1(), **kw)
    key = tuple(sorted(kw.items()))
    if key in MODES1_PINS:
        assert (len(msgs), _md5_lines(msgs)) == MODES1_PINS[key]


def test_oracle_modes1_stats_pins(checker_libs):
    # SURVEY.md §4 stat counters (single-bit fixes are double counted by the reference: 8 -> 16)
    _, st = C.oracle_decode(C.modes1())
    assert st == [546, 282, 535, 276, 259, 8, 16, 0]
    _, st = C.oracle_decode(C.modes1(), fix=0)
    assert st[:5] == [546, 287, 535, 283, 252]
    msgs, _ = C.oracle_decode(C.modes1())
    hist = {}
    for m in msgs:
        hist[m.msgtype] = hist.get(m.msgtype, 0) + 1
    assert hist == {0: 10, 4: 4, 5: 10, 11: 82, 17: 159, 20: 13, 21: 6}


# The reference's side of the *_equals_reference tests is recorded in tests/golden/reference_answers.json.
@pytest.mark.parametrize("kw", FLAG_SETS, ids=str)
def test_oracle_equals_reference_modes1(kw, checker_libs):
    o, os_ = C.oracle_decode(C.modes1(), **kw)
    G.assert_answer(f"oracle_equals_reference_modes1/{kw}", [_fields(o), os_])


SYNTHETIC_SEEDS = [11, 12, 13]
SYNTHETIC_FLAGS = [dict(), dict(aggressive=1), dict(check_crc=0, aggressive=1)]


def synthetic_traffic(seed):
    return synth.random_traffic(200000 + 7777 * seed, 300, seed, sigma=1.0 + seed % 3)


@pytest.mark.parametrize("seed", SYNTHETIC_SEEDS)
@pytest.mark.parametrize("kw", SYNTHETIC_FLAGS, ids=str)
def test_oracle_equals_reference_synthetic(seed, kw, checker_libs):
    o, os_ = C.oracle_decode(synthetic_traffic(seed), **kw)
    G.assert_answer(f"oracle_equals_reference_synthetic/{seed}/{kw}", [_fields(o), os_])


@pytest.mark.parametrize("name,cid", G.CASES)
def test_oracle_equals_golden(name, cid, checker_libs):
    doc = G.load(name)
    case = doc["cases"][cid]
    data = G.make_input(doc)
    msgs, st = C.oracle_decode(data, **case["flags"])
    assert _fields(msgs) == case["messages"]
    assert st == case["stats"]


def test_magnitude_pins(checker_libs):
    # SURVEY.md §4 kernel-level pins for modes1.bin
    m = C.oracle_magnitude(C.modes1())
    assert m.size == 356868 and int(m.astype(np.int64).sum()) == 1732288336 and int(m.max()) == 64913
    assert hashlib.sha256(m.astype("<u2").tobytes()).hexdigest().startswith("f116ccd64c38ad15")


def magnitude_buffer():
    """One reference buffer of modes1.bin behind the 476-byte carry, as the reference lays it out."""
    buf = np.full(262620, 127, dtype=np.uint8)
    buf[476: 476 + 262144] = C.modes1()[:262144]
    return buf


def test_magnitude_equals_reference(checker_libs):
    G.assert_answer("magnitude_equals_reference", C.oracle_magnitude(magnitude_buffer()).astype("<u2"))


def test_candidate_pins(checker_libs):
    # SURVEY.md §4: positions passing all preamble tests, every j, no skip
    cands = C.oracle_scan_candidates(C.modes1())
    t = np.array([c.t for c in cands], dtype=np.int64)
    per_buffer = [int(((t >> 17) == k).sum()) for k in range(3)]
    assert per_buffer == [215, 212, 135]
    pos = t - 238
    assert pos[:5].tolist() == [794, 1918, 2552, 4196, 4235]
    assert hashlib.sha256(pos.astype("<i8").tobytes()).hexdigest().startswith("20d38768f8bae2fe")


def test_known_answer_frames(checker_libs):
    # README.md:151 and dump1090.c:2460: both have syndrome 0
    lib = C.oracle_lib()
    lib.oracle_checksum.restype = ctypes.c_uint32
    for hx in ("8D451E8B99019699C00B0A81F36E", "8D4B969699155600E87406F5B69F"):
        b = bytes.fromhex(hx)
        assert lib.oracle_checksum(b, 112) == 0
        assert synth.modes_parity(b[:11]) == int.from_bytes(b[11:], "big")
        for bit in (5, 40, 111):
            assert lib.oracle_checksum(synth.flip_bits(b, [bit]), 112) != 0


def test_crc_table_matches_reference(checker_libs):
    # a single set data bit b has checksum == the reference's table entry b (its checksum of
    # the 112-bit message with only data bit b set)
    tab = (ctypes.c_uint32 * 112)()
    C.oracle_lib().oracle_crc_table(tab)
    assert G.answer("crc_table_matches_reference") == list(tab[:88])
    assert tab[87] == 0xFFF409 and all(tab[b] == 0 for b in range(88, 112))


def test_magnitude_is_strictly_monotone_in_squared_amplitude(checker_libs):
    """The scan kernel compares squared amplitudes instead of magnitudes; that is exact
    iff round(360*sqrt(n)) is strictly increasing over reachable n = i*i+q*q."""
    lut = (ctypes.c_uint16 * 16641)()
    C.oracle_lib().oracle_maglut(lut)
    by_n = {}
    for i in range(129):
        for q in range(129):
            by_n.setdefault(i * i + q * q, set()).add(lut[i * 129 + q])
    assert all(len(v) == 1 for v in by_n.values())
    ns = sorted(by_n)
    ms = [next(iter(by_n[n])) for n in ns]
    assert all(a < b for a, b in zip(ms, ms[1:]))
    assert max(ms) == 65167


def decode_bytes_frames():
    """300 frames of every DF, 0, 1 or 2 bits flipped, padded to 14 bytes."""
    rng = synth.Counter(99)
    for k in range(300):
        df = [17, 17, 18, 11, 4, 5, 20, 21, 0, 16][k % 10]
        body = bytes(rng.below(256) for _ in range(10 if df >= 16 else 3))
        frame = synth.make_frame(df, rng.below(8), body)
        flips = [rng.below(len(frame) * 8) for _ in range(k % 3)]
        yield synth.flip_bits(frame, flips).ljust(14, b"\0")


def decode_bytes_fields(lib, fname):
    """msg_fields of every frame of decode_bytes_frames() decoded by lib.fname, without and with --aggressive."""
    fn = getattr(lib, fname)
    out = []
    for frame in decode_bytes_frames():
        for aggressive in (0, 1):
            m = C.Msg()
            fn(frame, 1, aggressive, ctypes.byref(m))
            out.append(C.msg_fields(m))
    return out


def test_decode_bytes_matches_reference(checker_libs):
    got = decode_bytes_fields(C.oracle_lib(), "oracle_decode_bytes")
    assert len(got) == 600
    G.assert_answer("decode_bytes_matches_reference", got)
