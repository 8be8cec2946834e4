"""CPU (-m "not gpu"): the full message text (SURVEY §8(f) item 1) against the reference binary's
own stdout, byte for byte (its sha256, recorded in tests/golden/reference_answers.json).  Messages
come from the product's resolver fed with the checker's candidate records; the text from
modes_format_message()."""
import numpy as np
import pytest

import checker as C
import golden_util as G
from dump1090_b200 import api, synth


def _product_text(data, fix=1, aggressive=0, check_crc=1):
    cands = C.oracle_scan_candidates(data, fix=fix, aggressive=aggressive, cap=400000)
    arr = np.frombuffer(b"".join(bytes(c) for c in cands), dtype=api.CANDIDATE_DTYPE) if cands \
        else np.zeros(0, dtype=api.CANDIDATE_DTYPE)
    r = api.Resolver(fix_errors=fix, aggressive=aggressive, check_crc=check_crc)
    r.run(arr, np.array([(0, arr.size)], dtype=api.TILE_DTYPE))
    return "".join(m.text(check_crc) for m in r.take_messages())


MODES1_FLAGS = [([], {}), (["--aggressive"], dict(aggressive=1)), (["--no-crc-check"], dict(check_crc=0)),
                (["--no-fix"], dict(fix=0))]


@pytest.mark.parametrize("flags,kw", MODES1_FLAGS, ids=str)
def test_text_equals_reference_on_modes1(flags, kw, checker_libs):
    data = C.modes1()
    G.assert_answer(f"text_equals_reference_on_modes1/{' '.join(flags)}", _product_text(data, **kw).encode("latin1"))


TRAFFIC_SEEDS = [51, 52]
TRAFFIC_FLAGS = ["--aggressive", "--no-crc-check"]


def text_traffic(seed):
    return synth.random_traffic(400000, 700, seed, amp_range=(30.0, 110.0), max_flips=1)


@pytest.mark.parametrize("seed", TRAFFIC_SEEDS)
def test_text_equals_reference_on_traffic(seed, checker_libs):
    """All DF / extended-squitter kinds the generator emits (ident, surface, airborne, velocity,
    heading, unknown ME types, DF18, address/parity formats)."""
    text = _product_text(text_traffic(seed), aggressive=1, check_crc=0)
    G.assert_answer(f"text_equals_reference_on_traffic/{seed}", text.encode("latin1"))


def test_text_buffer_too_small_is_safe():
    m = api.Message()
    m.msgbits, m.msgtype, m.errorbit = 112, 17, -1
    import ctypes
    buf = ctypes.create_string_buffer(8)
    n = api.lib().modes_format_message(ctypes.byref(m), 1, buf, 8)
    assert n > 8 and buf.raw[7:8] == b"\0"


def test_raw_net_line_is_uppercase():
    m = api.Message()
    m.msgbits = 56
    for k, b in enumerate(bytes.fromhex("5d4840d6abcdef")):
        m.msg[k] = b
    assert m.raw_net_line() == "*5D4840D6ABCDEF;\n"          # dump1090.c:2387 "%02X"
    assert m.raw_line() == "*5d4840d6abcdef;"               # dump1090.c:1325 "%02x"


_FULL = "8D4B969699155600E87406F5B69F"
_SHORT = "5D4840D6ABCDEF"
HEX_LINES = [f"*{_FULL};", f"  *{_FULL};\r\n", f"*{_FULL.lower()};", f"*{_SHORT};", f"\t*{_SHORT};  ", f"*{_FULL}", f"{_FULL};",
             f"*{_FULL}00;", f"*{_FULL[:-1]};", f"*{_FULL[:-2]}zz;", "*;x", "", "   ", "*", ";", f"* {_FULL};", f"*{_FULL} ;"]


def test_hex_line_parser_matches_reference(checker_libs):
    """modes_parse_hex_line accepts / discards exactly the lines decodeHexMessage does, and yields the
    frame bytes it decodes (full-length frames: the reference leaves missing bytes uninitialised).
    Recorded per line: [delivered, msgbits, the 14 message bytes] of the reference."""
    want = G.answer("hex_line_parser_matches_reference")
    assert len(want) == len(HEX_LINES)
    for line, (delivered, msgbits, msg_hex) in zip(HEX_LINES, want):
        got = api.parse_hex_line(line)
        assert (got is not None) == bool(delivered), repr(line)
        if got is not None and len(line.strip()) - 2 in (14, 28):
            nbytes = msgbits // 8
            if nbytes * 2 == len(line.strip()) - 2:          # DF length matches what the line supplied
                assert got[:nbytes] == bytes.fromhex(msg_hex)[:nbytes], repr(line)
