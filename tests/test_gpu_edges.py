"""-m gpu: edge cases, the hex door, the C host binary, and full-size properties."""
import hashlib
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

import checker as C
import golden_util as G
from dump1090_b200 import api, synth

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def _lines(msgs):
    return [m.raw_line() for m in msgs]


def _olines(msgs):
    return [m.hexline() for m in msgs]


@pytest.mark.parametrize("nbytes", [0, 1, 2, 477, 5000, 262143, 262144, 262145, 524288, 600001])
@pytest.mark.parametrize("drop", [0, 1])
def test_ragged_lengths(nbytes, drop, gpu_decoder_factory, checker_libs):
    """Empty, odd, one-short, exact-buffer and one-over inputs: same EOF-buffer semantics as the
    reference (dump1090.c:481-507), both outcomes of its EOF race."""
    data = synth.random_traffic(300001, 420, 17)[:nbytes]
    exp, st = C.oracle_decode(data, drop_eof=drop)
    dec = gpu_decoder_factory(drop_eof_buffer=drop)
    got = dec.decode(data)
    assert _lines(got) == _olines(exp)
    assert list(dec.stats().values()) == st


def test_frame_at_every_buffer_seam_offset(gpu_decoder_factory, checker_libs):
    """A strong DF17 frame slid across the 131072-sample buffer seam: carry-over and the two
    untested positions per buffer (j = 131070, 131071) behave as in the reference."""
    frame = synth.make_frame(17, 5, bytes.fromhex("4840d6202cc371c32ce0"))
    dec = gpu_decoder_factory()
    for start in list(range(131072 - 250, 131072 - 225)) + [130830, 130831, 130832, 130833, 130834]:
        s = synth.synth_stream(131072 + 2000, [(start, frame, 80.0, 0.7, 0.0)], sigma=1.0, seed=start)
        exp, _ = C.oracle_decode(s)
        assert _lines(dec.decode(s)) == _olines(exp), start


def test_saturated_samples(gpu_decoder_factory, checker_libs):
    """Bytes 0 and 255 (|x-127| = 127/128, squared magnitudes up to 32768) keep exact ordering."""
    frame = synth.make_frame(17, 5, bytes.fromhex("4840d6202cc371c32ce0"))
    s = synth.synth_stream(200000, [(1000 + 400 * k, frame, 150.0 + 10 * k, 0.1 * k, 0.3 * (k % 3)) for k in range(300)],
                           sigma=3.0, seed=5)
    assert s.max() == 255 and s.min() == 0
    exp, st = C.oracle_decode(s, aggressive=1)
    dec = gpu_decoder_factory(aggressive=1)
    assert _lines(dec.decode(s)) == _olines(exp)
    assert list(dec.stats().values()) == st
    assert np.array_equal(dec.magnitude(s), C.oracle_magnitude(s))


def test_reset_and_reuse(gpu_decoder_factory, checker_libs):
    dec = gpu_decoder_factory()
    a = synth.random_traffic(200000, 250, 61)
    b = C.modes1()
    ea, _ = C.oracle_decode(a)
    eb, _ = C.oracle_decode(b)
    for _ in range(2):
        assert _lines(dec.decode(a)) == _olines(ea)
        assert _lines(dec.decode(b)) == _olines(eb)


def test_output_array_equals_callback(gpu_decoder_factory, checker_libs):
    data = C.modes1()
    dec = gpu_decoder_factory()
    want = _lines(dec.decode(data))
    out = dec.set_output_array(1000)
    dec.reset(); dec.rearm_output(); dec.process(data); dec.finish()
    n = dec.output_count()
    assert [out[i].raw_line() for i in range(n)] == want
    dec.set_output_array(0)


def hex_door_frames():
    """(aggressive, frame): 120 frames of every DF with 0, 1 or 2 flipped bits, without and then with --aggressive."""
    rng = synth.Counter(7)
    for aggressive in (0, 1):
        for k in range(120):
            df = [17, 17, 18, 11, 4, 5, 20, 21, 0, 16][k % 10]
            body = bytes(rng.below(256) for _ in range(10 if df >= 16 else 3))
            frame = synth.flip_bits(synth.make_frame(df, rng.below(8), body), [rng.below(56) for _ in range(k % 3)])
            yield aggressive, frame.ljust(14, b"\0")


def test_hex_door_matches_reference(gpu_decoder_factory, checker_libs):
    """modes_decode_frame == decodeModesMessage on frame bytes (dump1090.c:2472-2502), incl. repairs.
    The reference's msg_fields of every frame are recorded in tests/golden/reference_answers.json."""
    got = []
    for aggressive, frame in hex_door_frames():
        dec = gpu_decoder_factory(aggressive=aggressive)          # fresh ICAO cache, like the harness
        got.append(C.msg_fields(dec.decode_frame(frame)))
        dec.close()
    assert len(got) == 240
    G.assert_answer("hex_door_matches_reference", got)


def test_hex_door_batch_equals_single_frames(gpu_decoder_factory, checker_libs):
    """modes_decode_frames(n) == n x modes_decode_frame, including the address cache carried from frame to frame."""
    rng = synth.Counter(11)
    frames = []
    for k in range(300):
        df = [17, 11, 17, 4, 5, 20, 18, 0][k % 8]
        icao = 0x400000 + rng.below(40)
        body = (icao.to_bytes(3, "big") + bytes(rng.below(256) for _ in range(7))) if df in (17, 18) else \
            (icao.to_bytes(3, "big") if df == 11 else bytes(rng.below(256) for _ in range(10 if df >= 16 else 3)))
        fr = synth.make_frame(df, rng.below(8), body, icao_for_ap=None if df in (11, 17, 18) else icao)
        frames.append(synth.flip_bits(fr, [rng.below(len(fr) * 8) for _ in range(k % 3)]))
    for aggressive in (0, 1):
        one = gpu_decoder_factory(aggressive=aggressive)
        many = gpu_decoder_factory(aggressive=aggressive)
        want = [C.msg_fields(one.decode_frame(f)) for f in frames]
        got = [C.msg_fields(m) for m in many.decode_frames(frames)]
        assert got == want
        assert any(m["crcok"] for m in got if m["msgtype"] in (4, 5, 20))     # address/parity replies validated by the carried cache


C_HOST_TEXT_FLAGS = [[], ["--aggressive", "--no-crc-check"], ["--onlyaddr"]]


def test_c_host_binary(checker_libs):
    """./dump1090-b200 --ifile modes1.bin --raw prints the reference's lines (SURVEY.md §4 md5 pins)."""
    exe = ROOT / "dump1090-b200"
    assert exe.exists(), "build the C host with `make`"
    f = str(C.modes1_path())
    pins = {(): (284, "4a81758c8bec"), ("--drop-eof-buffer",): (217, "7b1719f22374"),
            ("--no-fix",): (283, "ac539444a66e"), ("--no-crc-check",): (765, "a6092d178fcf"),
            ("--no-crc-check", "--aggressive"): (824, "bec25488d6b8")}
    for flags, (n, md5) in pins.items():
        out = subprocess.run([str(exe), "--ifile", f, "--raw", *flags], capture_output=True, check=True).stdout
        assert out.count(b"\n") == n and hashlib.md5(out).hexdigest().startswith(md5), flags
    # default output = the full text of displayModesMessage (dump1090.c:1314-1450): byte-identical to the
    # reference harness binary, which prints through the reference's own function (the sha256 of its
    # stdout is recorded in tests/golden/reference_answers.json)
    for flags in C_HOST_TEXT_FLAGS:
        ours = subprocess.run([str(exe), "--ifile", f, *flags], capture_output=True, check=True).stdout
        G.assert_answer(f"c_host_binary/{' '.join(flags)}", ours)
    stats = subprocess.run([str(exe), "--ifile", f, "--stats"], capture_output=True, check=True, text=True).stdout
    assert stats.splitlines()[:4] == ["546 valid preambles", "282 demodulated again after phase correction",
                                      "535 demodulated with zero errors", "276 with good crc"]


def test_c_host_sbs_and_json(gpu_decoder_factory, checker_libs):
    """./dump1090-b200 --sbs / --aircraft-json == the Python tracker over the same decoded messages."""
    exe = ROOT / "dump1090-b200"
    f = str(C.modes1_path())
    msgs = gpu_decoder_factory().decode(C.modes1())
    tr = api.Tracker(1)
    lines = []
    for m in msgs:
        g = tr.update(m, api.STREAM_EPOCH_MS + int(m.sample_pos / 2000))
        if g:
            lines.append(g[1])
    sbs = subprocess.run([str(exe), "--ifile", f, "--sbs"], capture_output=True, check=True, text=True).stdout
    assert sbs == "".join(lines)
    js = subprocess.run([str(exe), "--ifile", f, "--aircraft-json"], capture_output=True, check=True, text=True).stdout
    assert js == tr.json()


def test_full_size_properties(gpu_decoder_factory, checker_libs):
    """BASELINE.json configs[1] size (modes1.bin tiled to 1 GiB, --no-fix): prefix equality with the
    oracle, invariance to feed chunking / batch size, determinism."""
    data = synth.tile_to(C.modes1(), 1 << 30)
    dec = gpu_decoder_factory(fix_errors=0)
    out = dec.set_output_array(700000)
    dec.reset(); dec.rearm_output(); dec.process(data); dec.finish()
    n = dec.output_count()
    assert n == 425744
    pos = np.array([out[i].sample_pos for i in range(n)])
    assert np.all(np.diff(pos) > 0), "messages must come out in stream order"
    digest = hashlib.sha256(b"".join(bytes(out[i].msg) for i in range(n))).hexdigest()
    stats = dec.stats()
    # prefix: the first 256 reference buffers, checked message for message against the oracle
    k = 256
    exp, _ = C.oracle_decode(data[: k * api.BUFFER_BYTES], fix=0, drop_eof=1)
    cut = int(np.searchsorted(pos, k * api.BUFFER_SAMPLES - 240))
    assert [out[i].raw_line() for i in range(cut)] == [m.hexline() for m in exp]
    # same stream, different chunking and batch size -> identical messages and statistics
    dec2 = gpu_decoder_factory(fix_errors=0, max_batch_bytes=api.BUFFER_BYTES * 7)
    out2 = dec2.set_output_array(700000)
    dec2.reset(); dec2.rearm_output()
    step = 100 * 1000 * 1000 + 1
    for off in range(0, data.size, step):
        dec2.process(data[off: off + step])
    dec2.finish()
    assert dec2.output_count() == n
    assert hashlib.sha256(b"".join(bytes(out2[i].msg) for i in range(n))).hexdigest() == digest
    assert dec2.stats() == stats


def _periodic(period_pattern, nsamples, amp=100):
    """I/Q stream whose magnitude repeats `period_pattern` (1 = pulse, 0 = silence)."""
    pat = np.array(period_pattern, dtype=np.uint8)
    reps = -(-nsamples // pat.size)
    hi = np.tile(pat, reps)[:nsamples]
    out = np.full(2 * nsamples, 127, dtype=np.uint8)
    out[0::2] = 127 + amp * hi
    return out


@pytest.mark.parametrize("name,pattern", [
    ("candidate_every_15", [1, 0, 1, 0, 0, 0, 0, 1, 0, 1, 0, 0, 0, 0, 0]),      # > 256 candidates per tile
    ("survivor_every_7", [1, 0, 1, 0, 0, 0, 0]),                                 # > 512 ten-comparison survivors per tile
    ("candidate_every_16", [1, 0, 1, 0, 0, 0, 0, 1, 0, 1, 0, 0, 0, 0, 0, 0]),   # exactly 256 per tile
])
def test_pathological_density(name, pattern, gpu_decoder_factory, checker_libs):
    """Periodic input that makes (almost) every period a preamble: the scan kernel's dense path,
    and the automatic growth of the candidate buffers (default room: one candidate per 64 samples)."""
    import torch
    data = _periodic(pattern, 131072 * 2 + 5000)
    exp, st = C.oracle_decode(data, check_crc=0, cap=200000)
    dec = gpu_decoder_factory(check_crc=0)
    got = dec.decode(data)
    assert [m.raw_line() for m in got] == [m.hexline() for m in exp]
    assert list(dec.stats().values()) == st
    # candidate records, byte for byte
    nbuf = data.size // api.BUFFER_BYTES + 1
    padded = np.full(nbuf * api.BUFFER_BYTES, 127, dtype=np.uint8)
    padded[: data.size] = data
    want = C.oracle_scan_candidates(data, cap=200000)
    want_arr = np.frombuffer(b"".join(bytes(c) for c in want), dtype=api.CANDIDATE_DTYPE)
    d = torch.from_numpy(padded).cuda()
    dec.detect_device(d.data_ptr(), nbuf)
    cands, tiles = dec.detect_fetch(nbuf)
    order = np.concatenate([np.arange(o, o + c) for o, c in tiles]).astype(int)
    assert order.size == want_arr.size
    assert np.array_equal(cands.view(np.uint8).reshape(-1, 56)[order], want_arr.view(np.uint8).reshape(-1, 56))


def test_caller_buffers_overflow_is_reported(gpu_decoder_factory):
    import torch
    data = _periodic([1, 0, 1, 0, 0, 0, 0, 1, 0, 1, 0, 0, 0, 0, 0], 131072)
    d = torch.from_numpy(data).cuda()
    small = torch.zeros(100 * 56, dtype=torch.uint8, device="cuda")
    tiles = torch.zeros(api.tiles_for(1) * 8, dtype=torch.uint8, device="cuda")
    dec = gpu_decoder_factory()
    dec.detect_device(d.data_ptr(), 1, None, small.data_ptr(), 100, tiles.data_ptr())
    with pytest.raises(RuntimeError, match="capacity exceeded"):
        dec.detect_wait()


@pytest.mark.parametrize("n_gpus,batch_buffers", [(2, 1), (3, 2), (2, 256)])
def test_multi_gpu_context(n_gpus, batch_buffers, gpu_decoder_factory, checker_libs):
    """modes_config.n_gpus > 1: the streaming decode deals its batches to several GPUs (devices are
    reused round-robin when the box has fewer) and resolves each group of batches exactly; messages,
    fields and statistics equal the oracle's, whatever the batch size and the feeding pattern."""
    data = synth.random_traffic(131072 * 11 + 4321, 2400, 91, n_aircraft=18)
    for kw in (dict(), dict(aggressive=1, check_crc=0)):
        exp, st = C.oracle_decode(data, aggressive=kw.get("aggressive", 0), check_crc=kw.get("check_crc", 1), cap=100000)
        dec = gpu_decoder_factory(n_gpus=n_gpus, max_batch_bytes=batch_buffers * api.BUFFER_BYTES, **kw)
        got = dec.decode(data)
        assert _lines(got) == _olines(exp)
        assert [C.msg_fields(m, with_pos=True) for m in got] == [C.msg_fields(m, with_pos=True) for m in exp]
        assert list(dec.stats().values()) == st
        assert _lines(dec.decode(data, chunk=300001)) == _olines(exp)


def test_c_host_multi_gpu(checker_libs):
    """./dump1090-b200 --gpus 2: same lines as one GPU (SURVEY.md §4 md5 pins)."""
    exe = ROOT / "dump1090-b200"
    f = str(C.modes1_path())
    for flags, (n, md5) in {(): (284, "4a81758c8bec"), ("--no-crc-check", "--aggressive"): (824, "bec25488d6b8")}.items():
        out = subprocess.run([str(exe), "--ifile", f, "--raw", "--gpus", "2", "--chunk", "300000", *flags], capture_output=True, check=True).stdout
        assert out.count(b"\n") == n and hashlib.md5(out).hexdigest().startswith(md5), flags


def test_two_gpu_fused_gather(checker_libs):
    """With two or more GPUs on the box: the sharded decode with the record gather fused into the
    kernels (CUDA-IPC peer stores into rank 0's HBM) equals the oracle (scripts/multi_gpu_parity.py)."""
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29577", str(ROOT / "scripts" / "multi_gpu_parity.py")],
                         capture_output=True, text=True, cwd=str(ROOT), timeout=600)
    assert "MULTI_GPU_PARITY PASS" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


@pytest.mark.parametrize("snr_db", [0, 6, 10, 15])
def test_low_snr_detect_rate_identical(snr_db, gpu_decoder_factory, checker_libs):
    """BASELINE.json configs[4] in miniature: injected DF17 at low SNR, --aggressive; the GPU must make
    exactly the oracle's decisions (same messages, same repairs), not merely a similar detect rate."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("snr_sweep", ROOT / "scripts" / "snr_sweep.py")
    sweep = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(sweep)
    data, truth = sweep.stream_at(float(snr_db), 400, 2000 + snr_db)
    exp, st = C.oracle_decode(data, aggressive=1, cap=8192)
    dec = gpu_decoder_factory(aggressive=1)
    got = dec.decode(data)
    assert [C.msg_fields(m) for m in got] == [C.msg_fields(m) for m in exp]
    assert list(dec.stats().values()) == st


def test_sleeping_host_wait_gives_the_same_messages(gpu_decoder_factory, checker_libs):
    """modes_set_host_wait(1): contexts created afterwards wait on cudaEventBlockingSync events."""
    L = api.lib()
    a = synth.random_traffic(131072 * 5 + 999, 900, 67)
    want, st = C.oracle_decode(a)
    assert L.modes_set_host_wait(1) == 0
    try:
        dec = gpu_decoder_factory(max_batch_bytes=2 * api.BUFFER_BYTES)
        for _ in range(2):
            assert _lines(dec.decode(a)) == _olines(want)
        assert list(dec.stats().values()) == st
        n_buf = a.size // api.BUFFER_BYTES + 1                # the stream plus the no-signal EOF buffer
        padded = np.full(n_buf * api.BUFFER_BYTES, 127, dtype=np.uint8)
        padded[: a.size] = a
        dec.detect_host(padded.ctypes.data, n_buf, None)
        cands, tiles = dec.detect_fetch(n_buf)
        res = api.Resolver()
        res.run(cands, tiles)
        assert _lines(res.take_messages()) == _olines(want)
        assert int(tiles["count"].sum()) == cands.size > 0
    finally:
        assert L.modes_set_host_wait(0) == 0
