"""Host-only timing of the sequential resolve (modes_resolve.cpp) on records produced by the
oracle's candidate scan: no GPU needed.  usage: python scripts/resolve_probe.py [MiB] [shards]"""
import sys, time, pathlib
import numpy as np
ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
import checker as C
from dump1090_b200 import api, synth

mib = int(sys.argv[1]) if len(sys.argv) > 1 else 256
n_sh = int(sys.argv[2]) if len(sys.argv) > 2 else 8
C.build_oracle()
src = C.modes1()
data = synth.tile_to(src, mib << 20)
t0 = time.time()
cands = C.oracle_scan_candidates(data, fix=0, cap=4_000_000)
arr = np.frombuffer(b"".join(bytes(c) for c in cands), dtype=api.CANDIDATE_DTYPE)
print(f"oracle scan: {len(arr)} candidates in {time.time()-t0:.1f}s", flush=True)
n_buf = (mib << 20) // (2 * 131072)
g = (arr["t"] + 2) // api.TILE_SAMPLES
n_tiles = api.tiles_for(n_buf)
cnt = np.bincount(g, minlength=n_tiles).astype(np.uint32)
off = np.concatenate([[0], np.cumsum(cnt)[:-1]]).astype(np.uint32)
tiles = np.zeros(n_tiles, dtype=api.TILE_DTYPE)
tiles["offset"] = off; tiles["count"] = cnt
if len(sys.argv) > 3 and sys.argv[3] == "scatter":
    # the GPU appends tiles in completion order: scatter the tiles' record runs through the array
    rng = np.random.default_rng(5)
    order = np.argsort(np.arange(n_tiles) + rng.integers(0, 6000, n_tiles))      # locally scrambled, globally increasing
    new_off = np.zeros(n_tiles, dtype=np.uint32)
    new_off[order] = np.concatenate([[0], np.cumsum(cnt[order])[:-1]])
    src = np.repeat(off, cnt) + (np.arange(len(arr)) - np.repeat(off, cnt))
    dst = np.repeat(new_off, cnt) + (np.arange(len(arr)) - np.repeat(off, cnt))
    scattered = np.zeros_like(arr)
    scattered.view(np.uint8).reshape(-1, 56)[dst] = arr.view(np.uint8).reshape(-1, 56)[src]
    arr = scattered
    tiles["offset"] = new_off

for shards in (1, n_sh):
    r = api.Resolver(fix_errors=0, aggressive=0, check_crc=1)
    out = r.set_output_array(shards * 600_000 * mib // 1024 + 1000)
    sh = [(arr.copy(), tiles.copy(), k * n_buf) for k in range(shards)]          # distinct memory per shard
    best = 1e9
    for it in range(3):
        r.reset_state(); r.rearm_output()
        t0 = time.perf_counter()
        r.run_shards(sh) if shards > 1 else r.run(arr, tiles)
        dt = time.perf_counter() - t0
        best = min(best, dt)
    print(f"shards={shards}: {r.output_count()} messages, best {best*1e3:.1f} ms "
          f"({shards*len(arr)/best/1e6:.1f} M candidates/s)", flush=True)
