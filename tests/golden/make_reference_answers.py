"""Record tests/golden/reference_answers.json: the unmodified reference's side of every test
that compares with it (test_oracle, test_format_text, test_tracker, test_gpu_edges).

Run where the reference is compiled into oracle/_ref (`make oracle` with its sources present):

    python tests/golden/make_reference_answers.py              # (re)write the file
    python tests/golden/make_reference_answers.py --show KEY   # print one answer, to diff with a failing test's

Each answer is keyed by test and parameters.  Small answers are stored as they are, large ones
as golden_util.digest() of exactly what the test computes on the product's (or oracle's) side.
The inputs come from the same functions the tests call.
"""
import ctypes
import json
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent))
sys.path.insert(0, str(HERE.parent.parent))

import checker as C  # noqa: E402
import golden_util as G  # noqa: E402
import test_format_text as TF  # noqa: E402
import test_gpu_edges as TE  # noqa: E402
import test_oracle as TO  # noqa: E402
import test_tracker as TT  # noqa: E402

REF_BIN = C.ORACLE_DIR / "_ref" / "ref_dump1090"
STORED_AS_IS = {"crc_table_matches_reference", "hex_line_parser_matches_reference",
                "tracker_ignores_bad_crc_when_checking", "stream_clock_starts_at_the_epoch"}


def ref_stdout(data_or_path, flags):
    """stdout of the reference harness binary (the reference's main()) on a capture."""
    if isinstance(data_or_path, Path):
        return subprocess.run([str(REF_BIN), "--ifile", str(data_or_path), *flags], capture_output=True, check=True).stdout
    with tempfile.NamedTemporaryFile(suffix=".bin") as f:
        f.write(data_or_path.tobytes())
        f.flush()
        return subprocess.run([str(REF_BIN), "--ifile", f.name, *flags], capture_output=True, check=True).stdout


def oracle_answers(ans):
    ref = C.ref_lib()
    for kw in TO.FLAG_SETS:
        r, rs = C.ref_decode(C.modes1(), **kw)
        ans[f"oracle_equals_reference_modes1/{kw}"] = [TO._fields(r), rs]
    for seed in TO.SYNTHETIC_SEEDS:
        for kw in TO.SYNTHETIC_FLAGS:
            r, rs = C.ref_decode(TO.synthetic_traffic(seed), **kw)
            ans[f"oracle_equals_reference_synthetic/{seed}/{kw}"] = [TO._fields(r), rs]
    buf = TO.magnitude_buffer()
    out = np.empty(buf.size // 2, dtype="<u2")
    ref.ref_magnitude(buf.ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p))
    ans["magnitude_equals_reference"] = out
    ref.ref_checksum.restype = ctypes.c_uint32
    crc = []
    for b in range(88):
        msg = bytearray(14)
        msg[b >> 3] = 0x80 >> (b & 7)
        crc.append(int(ref.ref_checksum(bytes(msg), 112)))
    ans["crc_table_matches_reference"] = crc
    ans["decode_bytes_matches_reference"] = TO.decode_bytes_fields(ref, "ref_decode_bytes")


def text_answers(ans):
    for flags, _ in TF.MODES1_FLAGS:
        ans[f"text_equals_reference_on_modes1/{' '.join(flags)}"] = ref_stdout(C.modes1_path(), flags)
    for seed in TF.TRAFFIC_SEEDS:
        ans[f"text_equals_reference_on_traffic/{seed}"] = ref_stdout(TF.text_traffic(seed), TF.TRAFFIC_FLAGS)
    rows = []
    for line in TF.HEX_LINES:
        out = C.Msg()
        delivered = C.ref_lib().ref_decode_hex_line(line.encode(), 1, 0, ctypes.byref(out))
        rows.append([int(bool(delivered)), int(out.msgbits), bytes(out.msg).hex()])
    ans["hex_line_parser_matches_reference"] = rows


def tracker_answers(ans):
    ans["nl_function_matches_reference"] = [C.ref_cpr_nl(lat) for lat in TT.nl_latitudes()]
    for check_crc in (1, 0):
        msgs, times = TT.decoded_traffic(check_crc)
        ans[f"tracker_on_decoded_traffic/{check_crc}"] = TT.trace(C.RefTracker(check_crc), msgs, times)
    _, msgs, times = TT.real_position_run()
    ans["tracker_decodes_real_positions"] = TT.trace(C.RefTracker(), msgs, times)
    ans["tracker_expiry_and_order"] = TT.expiry_trace(C.RefTracker())
    bad = TT.bad_crc_frame()
    ans["tracker_ignores_bad_crc_when_checking"] = [C.RefTracker(c).update(bad, 1) is not None for c in (1, 0)]
    ref = C.RefTracker()
    frames, stream_ms = TT.first_frames_of_a_file(47.3, 8.5, 0x4B1601)
    rows = []
    for m, t in zip(frames, stream_ms):
        a, sbs = ref.update(m, 1_700_000_000_000 + t)
        rows.append([a.lat, a.lon, sbs])
    ans["stream_clock_starts_at_the_epoch"] = rows


def gpu_edge_answers(ans):
    fields = []
    for aggressive, frame in TE.hex_door_frames():
        m = C.Msg()
        C.ref_lib().ref_decode_bytes(frame, 1, aggressive, ctypes.byref(m))
        fields.append(C.msg_fields(m))
    ans["hex_door_matches_reference"] = fields
    for flags in TE.C_HOST_TEXT_FLAGS:
        ans[f"c_host_binary/{' '.join(flags)}"] = ref_stdout(C.modes1_path(), flags)


def main():
    C.build_oracle()
    if not (C.REF_SO.exists() and REF_BIN.exists()):
        raise SystemExit("oracle/_ref is not built: run `make oracle` where the reference sources are present")
    ans = {}
    for part in (oracle_answers, text_answers, tracker_answers, gpu_edge_answers):
        part(ans)
    if sys.argv[1:2] == ["--show"]:
        G.write_answer(ans[sys.argv[2]], sys.stdout.buffer)
        return
    stored = {k: v if k in STORED_AS_IS else G.digest(v) for k, v in ans.items()}
    G.ANSWERS_PATH.write_text(json.dumps(stored, indent=1, sort_keys=True) + "\n")
    print(f"{G.ANSWERS_PATH.name}: {len(stored)} answers")


if __name__ == "__main__":
    main()
