"""A receiver pool created with gpu_resolve = 1 (modes_pool_*): the order-dependent half runs on the
device, one warp per receiver with that receiver's address cache resident in HBM.  Every receiver's
messages, fields, stream positions and statistics must equal a decode of its stream alone, and the
output array, receiver_of[] and the statistics must equal the host pool path's byte for byte, on any
sequence of calls."""
import ctypes

import numpy as np
import pytest

import checker as C
from dump1090_b200 import api, synth
from test_pool import BUF, _check, _expect, _schedule, _streams

FLAGS = [dict(), dict(aggressive=1), dict(fix=0), dict(check_crc=0)]
AP_FORMATS = {0, 4, 5, 16, 20, 21}          # address/parity replies: accepted only for an address in the cache


def _ids(kw):
    return "-".join(f"{a}{b}" for a, b in kw.items()) or "default"


def _cfg(kw):
    return dict(fix_errors=kw.get("fix", 1), aggressive=kw.get("aggressive", 0), check_crc=kw.get("check_crc", 1))


def test_host_half_refused_when_resolving_on_device():
    """modes_pool_resolve would replay with the host caches, which such a pool never updates."""
    with api.ReceiverPool(3, gpu_resolve=1) as pool:
        with pytest.raises(RuntimeError, match="resolves on the device"):
            pool.resolve([0], np.zeros(0, api.CANDIDATE_DTYPE), np.zeros(api.tiles_for(2), api.TILE_DTYPE))


def _run(ops, n_rx, gpu_resolve, max_batch=0, cap=20000, **cfg):
    """Run a call sequence on one pool: what every collect put in the output array (structs and
    receiver_of, as bytes), every receiver's messages through the sink, its statistics and buffers."""
    size = ctypes.sizeof(api.Message)
    with api.ReceiverPool(n_rx, max_batch=max_batch, gpu_resolve=gpu_resolve, **cfg) as pool:
        out, out_rx = pool.set_output_array(cap)
        arrays = []

        def took():
            n = pool.output_count()
            assert n <= cap, "output array too small for the test"
            arrays.append((ctypes.string_at(out, n * size), out_rx[:n].tobytes()))

        for op, *a in ops:
            if op == "reset":
                pool.reset(*a)
            elif op == "submit":
                pool.submit(*a)
            else:
                pool.rearm_output()
                if op == "ingest":
                    pool.ingest(*a)
                else:
                    pool.collect()
                took()
        msgs = [[bytes(m) for m in pool.take(r)] for r in range(n_rx)]
        return dict(arrays=arrays, msgs=msgs, stats=[pool.stats(r) for r in range(n_rx)],
                    buffers=[pool.buffers(r) for r in range(n_rx)])


def _same_as_host_path(ops, n_rx, **kw):
    host, dev = _run(ops, n_rx, 0, **kw), _run(ops, n_rx, 1, **kw)
    assert sum(len(m) for m in host["msgs"]) > 0
    for key in ("buffers", "stats", "msgs"):
        assert dev[key] == host[key], key
    assert len(dev["arrays"]) == len(host["arrays"])
    for k, (d, h) in enumerate(zip(dev["arrays"], host["arrays"])):
        assert d[1] == h[1], f"receiver_of of call {k}"
        assert d[0] == h[0], f"structs of call {k}"
    return dev


@pytest.mark.gpu
@pytest.mark.parametrize("kw", FLAGS, ids=_ids)
def test_device_resolve_matches_single_stream_decodes(kw, checker_libs):
    n_rx, n_buf = 7, 3
    streams = _streams(n_rx, n_buf)
    nxt = [0] * n_rx
    with api.ReceiverPool(n_rx, max_batch=5, gpu_resolve=1, **_cfg(kw)) as pool:
        for ids in _schedule(n_rx, n_buf, seed=4):
            for lo in range(0, len(ids), 5):                            # at most max_batch receivers per call
                part = ids[lo: lo + 5]
                pool.ingest(part, [streams[r][nxt[r] * BUF: (nxt[r] + 1) * BUF] for r in part])
                for r in part:
                    nxt[r] += 1
        assert [pool.buffers(r) for r in range(n_rx)] == [n_buf] * n_rx
        _check(pool, streams, kw)


@pytest.mark.gpu
def test_device_resolve_equals_host_path_at_256_receivers(checker_libs):
    """The receivers workload's shape: receiver r reads the tiled capture r buffers in, two batches
    in flight, all buffers of a call at one stride in host memory."""
    n_rx, steps = 256, 3
    data = np.resize(C.modes1(), (n_rx + steps) * BUF)
    ids = list(range(n_rx))

    def batch(k):
        return ids, [data[(r + k) * BUF: (r + k + 1) * BUF] for r in ids]

    ops = [("submit", *batch(0))]
    for k in range(1, steps):
        ops += [("submit", *batch(k)), ("collect",)]
    ops += [("collect",)]
    dev = _same_as_host_path(ops, n_rx, cap=n_rx * 400, fix_errors=0)
    exp, exp_stats = C.oracle_decode(data[: steps * BUF], fix=0, drop_eof=1)
    got0 = [api.Message.from_buffer_copy(b) for b in dev["msgs"][0]]
    assert [m.raw_line() for m in got0] == [m.hexline() for m in exp]
    assert list(dev["stats"][0].values()) == exp_stats


@pytest.mark.gpu
def test_caches_are_per_receiver_and_persist_across_batches(checker_libs):
    """Receiver B joins receiver A's stream at buffer 2: address/parity replies of aircraft A heard
    announced earlier are A's messages, and not B's until B has heard the aircraft itself."""
    n_buf = 4
    s = synth.random_traffic(n_buf * 131072, 80 * n_buf, seed=11, n_aircraft=20)
    with api.ReceiverPool(2, gpu_resolve=1) as pool:
        for k in range(n_buf):
            ids = [0, 1] if k >= 2 else [0]
            pool.ingest(ids, [s[k * BUF: (k + 1) * BUF]] * len(ids))
        got_a, got_b = pool.take(0), pool.take(1)
        stats_a, stats_b = list(pool.stats(0).values()), list(pool.stats(1).values())
    lines_a, fields_a, want_stats_a = _expect(s, {})
    lines_b, fields_b, want_stats_b = _expect(s[2 * BUF:], {})

    def replies(lines, fields, since):
        return {ln for ln, f in zip(lines, fields) if f["sample_pos"] >= since and f["msgtype"] in AP_FORMATS}

    assert replies(lines_a, fields_a, 2 * 131072) - replies(lines_b, fields_b, 0), "the streams do not tell the caches apart"
    assert [m.raw_line() for m in got_a] == lines_a and [C.msg_fields(m, with_pos=True) for m in got_a] == fields_a
    assert [m.raw_line() for m in got_b] == lines_b and [C.msg_fields(m, with_pos=True) for m in got_b] == fields_b
    assert (stats_a, stats_b) == (want_stats_a, want_stats_b)


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(), dict(check_crc=0)], ids=_ids)
def test_pipeline_and_lifecycle_equal_host_path(kw, checker_libs):
    n_rx, n_buf = 5, 3
    st = _streams(n_rx, n_buf)

    def buf(r, k, stream=None):
        return st[r if stream is None else stream][k * BUF: (k + 1) * BUF]

    ops = []
    # two batches in flight, receivers in both of them
    ops += [("submit", [0, 1, 2], [buf(r, 0) for r in (0, 1, 2)])]
    for k in range(1, n_buf):
        ops += [("submit", [2, 0, 1], [buf(r, k) for r in (2, 0, 1)]), ("collect",)]
    ops += [("collect",)]
    # all buffers of a call in one host block (constant distance): the strided upload
    ops += [("reset", r) for r in range(n_rx)]
    for k in range(n_buf):
        block = np.stack([buf(r, k) for r in range(n_rx)])
        ops += [("ingest", list(range(n_rx)), [block[r] for r in range(n_rx)])]
    # reset between calls: receiver 3 starts its stream again
    ops += [("reset", 3), ("ingest", [3, 4], [buf(3, 0), buf(4, 0)]), ("ingest", [3], [buf(3, 1)])]
    # reset of a receiver whose batch is still in flight: it takes effect for that batch
    ops += [("reset", 0), ("submit", [0, 1], [buf(0, 0), buf(1, 0)]), ("reset", 1),
            ("submit", [1, 0], [buf(1, 1), buf(0, 1)]), ("collect",), ("collect",)]
    # a receiver that starts a new stream
    ops += [("reset", 2)] + [("ingest", [2], [buf(2, k, stream=4)]) for k in range(n_buf)]
    _same_as_host_path(ops, n_rx, **_cfg(kw))


@pytest.mark.gpu
def test_dense_batch_is_repeated_before_the_caches_are_touched(checker_libs):
    """A buffer denser than the candidate buffers of a batch (one candidate per 64 samples): the
    detection is repeated with larger buffers, and the device resolve then runs once, as usual."""
    from test_gpu_edges import _periodic
    dense = _periodic([1, 0, 1, 0, 0, 0, 0, 1, 0, 1, 0, 0, 0, 0, 0], 3 * 131072)
    st = _streams(1, 3)[0]
    ops = [("ingest", [0, 1], [dense[:BUF], st[:BUF]]),
           ("ingest", [0], [dense[BUF: 2 * BUF]]),                     # alone in its batch: over capacity
           ("ingest", [1, 0], [st[BUF: 2 * BUF], dense[2 * BUF:]])]
    _same_as_host_path(ops, 2, cap=60000, check_crc=0)
