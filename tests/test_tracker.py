"""SURVEY.md §8(f) item 3: the aircraft tracker (modes_tracker_*, pure host code) against the
reference's own interactiveReceiveData / decodeCPR / decodeCPRSurface / modesSendSBSOutput /
aircraftsToJson, driven message by message with the same explicit clock.  Positions are compared
bit for bit (doubles), text byte for byte.  The reference's side of every run is recorded in
tests/golden/reference_answers.json (tests/golden/make_reference_answers.py)."""
import ctypes
import math

import numpy as np
import pytest

import checker as C
import golden_util as G
from dump1090_b200 import api, synth


def _decode_frame(frame: bytes) -> C.Msg:
    """decodeModesMessage on raw bytes (fresh ICAO cache), through the oracle, which
    test_oracle.py::test_decode_bytes_matches_reference holds to the reference's."""
    out = C.Msg()
    buf = (ctypes.c_uint8 * 14)(*(list(frame) + [0] * (14 - len(frame))))
    C.oracle_lib().oracle_decode_bytes(buf, 1, 0, ctypes.byref(out))
    return out


def _as_product(m) -> api.Message:
    p = api.Message()
    ctypes.memmove(ctypes.byref(p), ctypes.byref(m), ctypes.sizeof(api.Message))
    return p


def _plain(v):
    """An aircraft tuple as JSON values (the char fields as text)."""
    return [x.decode("latin1") if isinstance(x, bytes) else x for x in v]


def trace(tracker, messages, times):
    """What a tracker answers over a run: (aircraft state, SBS line) or None after every message,
    then the aircraft list, the reference position, the JSON and the interactive tables."""
    out = []
    for m, t in zip(messages, times):
        r = tracker.update(m, t)
        out.append(None if r is None else [_plain(r[0].as_tuple()), r[1]])
    out.append([_plain(a.as_tuple()) for a in tracker.aircraft()])
    out.append(list(tracker.reference()))
    for metric in (0, 1):
        out.append(tracker.json(metric))
        for rows in (3, 15, 100):
            out.append(tracker.table(times[-1] + 4321 * (rows + metric), metric, rows))
    return out


def _run_product(key, messages, times, check_crc=1):
    """Feed the product's tracker; its whole trace must equal the reference's. Returns (tracker, messages tracked)."""
    got = api.Tracker(check_crc)
    tr = trace(got, [_as_product(m) for m in messages], times)
    G.assert_answer(key, tr)
    return got, sum(r is not None for r in tr[: len(messages)])


def nl_latitudes():
    """A fine grid, and every transition latitude of the zone-count table with its neighbours one ulp and 1e-9 away."""
    nz = 15.0
    a = 1.0 - math.cos(math.pi / (2.0 * nz))
    lats = [float(x) for x in np.linspace(-90.5, 90.5, 20001)]
    for nl in range(2, 60):
        t = round(math.degrees(math.acos(math.sqrt(a / (1.0 - math.cos(2.0 * math.pi / nl))))), 8)
        for d in (t, np.nextafter(t, 0), np.nextafter(t, 100), t - 1e-9, t + 1e-9):
            lats += [float(d), -float(d)]
    return lats


def test_nl_function_matches_reference(checker_libs):
    """The zone-count table is generated from its defining formula: identical to the reference's
    literal table everywhere, including one ulp either side of every transition latitude."""
    G.assert_answer("nl_function_matches_reference", [api.cpr_nl(lat) for lat in nl_latitudes()])


def decoded_traffic(check_crc):
    data = synth.random_traffic(131072 * 12, 2600, 41, n_aircraft=25)
    msgs, _ = C.oracle_decode(data, check_crc=check_crc)
    return msgs, [1_700_000_000_000 + 37 * k for k in range(len(msgs))]          # ~27 messages per second


def test_tracker_on_decoded_traffic(checker_libs):
    """Everything the decoder delivers from a mixed-traffic stream (identification, airborne and
    surface positions with random CPR fields, velocities, address/parity replies)."""
    for check_crc in (1, 0):
        msgs, times = decoded_traffic(check_crc)
        _, tracked = _run_product(f"tracker_on_decoded_traffic/{check_crc}", msgs, times, check_crc)
        assert tracked > 300


def _cpr_encode(lat, lon, odd):
    """Airborne CPR encoding of a position (17 bits each), the inverse of what the tracker decodes."""
    dlat = 360.0 / (60 - odd)
    yz = math.floor(131072 * ((lat % dlat) / dlat) + 0.5)
    rlat = dlat * (yz / 131072 + math.floor(lat / dlat))
    nl = api.cpr_nl(rlat)
    dlon = 360.0 / max(nl - odd, 1)
    xz = math.floor(131072 * ((lon % dlon) / dlon) + 0.5)
    return yz & 0x1FFFF, xz & 0x1FFFF


def _position_frame(icao, tc, odd, yz, xz, alt12=0x3A5):
    bits = (tc << 51) | (alt12 << 36) | (odd << 34) | (yz << 17) | xz
    return synth.make_frame(17, 5, icao.to_bytes(3, "big") + bits.to_bytes(7, "big"))


def real_position_run():
    """(fleet, messages, times): eleven aircraft on straight tracks, surface frames in between."""
    rng = np.random.default_rng(5)
    fleet = [(0x4B1600 + i, 47.0 + rng.uniform(-3, 3), 8.0 + rng.uniform(-4, 4), rng.uniform(-0.002, 0.002),
              rng.uniform(-0.003, 0.003)) for i in range(8)]
    fleet += [(0xA00001, -33.9, 151.2, 0.001, 0.001), (0x7C0001, 69.7, 18.9, 0.0, 0.004), (0xE40001, -0.3, -78.5, 0.002, 0.0)]
    msgs, times = [], []
    t = 1_700_000_000_000
    for step in range(60):
        for icao, lat0, lon0, vlat, vlon in fleet:
            lat, lon = lat0 + vlat * step, lon0 + vlon * step
            odd = (step + icao) & 1
            yz, xz = _cpr_encode(lat, lon, odd)
            msgs.append(_decode_frame(_position_frame(icao, 11, odd, yz, xz)))
            times.append(t)
            t += int(rng.integers(20, 400))
            if step % 7 == 3:                                            # a surface frame from the same airframe
                sbits = (6 << 51) | (int(rng.integers(0, 128)) << 44) | (1 << 43) | (int(rng.integers(0, 128)) << 36) \
                        | (odd << 34) | ((yz * 4) & 0x1FFFF) << 17 | ((xz * 4) & 0x1FFFF)
                msgs.append(_decode_frame(synth.make_frame(17, 5, icao.to_bytes(3, "big") + sbits.to_bytes(7, "big"))))
                times.append(t)
                t += 50
        if step == 30:
            t += 11_000                                                   # a gap longer than the 10 s pairing window
    return fleet, msgs, times


def test_tracker_decodes_real_positions(checker_libs):
    """Aircraft flying real tracks: even/odd pairs decode to the encoded position (to CPR
    resolution), the reference position follows, surface frames decode against it — and every
    double equals the reference's."""
    fleet, msgs, times = real_position_run()
    got, tracked = _run_product("tracker_decodes_real_positions", msgs, times)
    assert tracked == len(msgs)
    # sanity of the test itself: the airborne fleet ends up where it was flown to
    by_addr = {a.addr: a for a in got.aircraft()}
    for icao, lat0, lon0, vlat, vlon in fleet:
        a = by_addr[icao]
        if a.altitude:                                                    # last frame was airborne
            assert abs(a.lat - (lat0 + vlat * 59)) < 0.02 and abs(a.lon - (lon0 + vlon * 59)) < 0.02
    assert got.reference()[2] > 100


def expiry_trace(tracker, as_msg=lambda m: m):
    """Twenty aircraft a second apart, then expiry at several clocks and time-to-live values: the
    order of the list after the updates, and per expiry the count removed and the aircraft left."""
    msgs = [_decode_frame(synth.make_frame(17, 5, (0x400000 + i).to_bytes(3, "big") + bytes([0x20, 0x10, 0x82, 0x0C, 0x30, 0xC3, 0x0C])))
            for i in range(20)]
    t0 = 1_700_000_000_000
    for k, m in enumerate(msgs):
        tracker.update(as_msg(m), t0 + 1000 * k)
    out = [[a.addr for a in tracker.aircraft()]]
    for now, ttl in ((t0 + 25_000, 60), (t0 + 25_000, 10), (t0 + 25_999, 9), (t0 + 40_000, 0)):
        out.append([tracker.expire(now, ttl), [_plain(a.as_tuple()) for a in tracker.aircraft()]])
    return out


def test_tracker_expiry_and_order(checker_libs):
    got = api.Tracker()
    tr = expiry_trace(got, _as_product)
    assert tr[0] == [0x400000 + i for i in reversed(range(20))]
    G.assert_answer("tracker_expiry_and_order", tr)
    assert got.aircraft() == []


def bad_crc_frame():
    bad = _decode_frame(bytes.fromhex("8D4840D6202CC371C32CE0576099"))       # last byte off: CRC fails, not fixable to DF17? either way
    bad.crcok = 0
    return bad


def test_tracker_ignores_bad_crc_when_checking(checker_libs):
    bad = bad_crc_frame()
    # recorded: whether the reference's tracker took the frame with and without the CRC check
    assert G.answer("tracker_ignores_bad_crc_when_checking") == [False, True]
    assert api.Tracker(1).update(_as_product(bad), 1) is None
    assert api.Tracker(0).update(_as_product(bad), 1) is not None


def first_frames_of_a_file(lat, lon, icao):
    """Three airborne position frames (even, odd, even) of one aircraft, at stream times 3, 450 and 900 ms."""
    frames = []
    for step, odd in enumerate((0, 1, 0)):
        yz, xz = _cpr_encode(lat + 0.001 * step, lon, odd)
        frames.append(_decode_frame(_position_frame(icao, 11, odd, yz, xz)))
    return frames, [3, 450, 900]                                          # first seconds of a file


def test_stream_clock_starts_at_the_epoch(checker_libs):
    """A file's stream clock (sample position / 2 MHz) starts at 0: fed to the tracker as is, the
    first airborne position of a new aircraft would be paired with the empty (time 0) slot of the
    other parity and decoded against zeros.  With MODES_STREAM_EPOCH_MS added — what the C host
    does — the first frame waits for its partner, exactly as under the reference's wall clock."""
    lat, lon, icao = 47.3, 8.5, 0x4B1601
    frames, stream_ms = first_frames_of_a_file(lat, lon, icao)
    # reference behaviour under its own (wall) clock: no position after one frame, a position after two
    # (recorded per frame: [lat, lon, SBS line] of the reference at 1_700_000_000_000 + t)
    want = G.answer("stream_clock_starts_at_the_epoch")
    assert len(want) == len(frames)
    got = api.Tracker()
    for m, t, (r_lat, r_lon, r_sbs) in zip(frames, stream_ms, want):
        g = got.update(_as_product(m), api.STREAM_EPOCH_MS + t)
        assert (g[0].lat, g[0].lon) == (r_lat, r_lon)
        assert g[1] == r_sbs                                              # SBS line
        if t == 3:
            assert (g[0].lat, g[0].lon) == (0.0, 0.0)
    assert abs(got.aircraft()[0].lat - lat) < 0.02 and abs(got.aircraft()[0].lon - lon) < 0.02
    # the hazard itself (documented in include/modes_b200.h): a clock starting at 0 pairs the first frame with nothing
    raw = api.Tracker()
    g = raw.update(_as_product(frames[0]), stream_ms[0])
    assert (g[0].lat, g[0].lon) != (0.0, 0.0)
