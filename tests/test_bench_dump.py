"""bench.py --dump-outputs: the last timed step's planes and RGBA of a fixed sample of streams, written as float arrays,
are exactly the oracle's pictures of those streams, and the same on every run with the same arguments."""
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import oracle_decode_stream
from h263_rs_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, H = 352, 288
NAMES = ("stream_ids", "y", "cb", "cr", "rgba")


def bench_dump(out, impl, streams, steps, warmup):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", impl, "--streams", str(streams), "--steps", str(steps),
           "--warmup", str(warmup), "--skip-extras", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return {n: np.load(os.path.join(out, n + ".npy")) for n in NAMES}


@pytest.mark.parametrize("impl", ["reference", pytest.param("ours", marks=pytest.mark.gpu)])
def test_dump_is_the_oracle_picture_of_the_last_step(tmp_path, impl):
    streams, steps, warmup = 24, 2, 1
    got = bench_dump(tmp_path / "a", impl, streams, steps, warmup)
    ids = got["stream_ids"].astype(np.int64)
    assert got["stream_ids"].dtype == np.float64 and all(got[n].dtype == np.float32 for n in NAMES[1:])
    assert len(ids) == 16 and len(set(ids.tolist())) == 16 and ids.min() >= 0 and ids.max() < streams
    assert got["rgba"].shape == (16, H, W, 4) and got["cb"].shape == (16, H // 2, W // 2)
    for k, s in enumerate(ids):
        # bench.py's workload: stream s is generated with seed s, every fourth one with full-range vectors
        packets = synth.make_stream(W, H, 1 + warmup + steps, int(s), mv_mode=0 if s % 4 else 1)
        ref = oracle_decode_stream(packets)[-1]
        assert np.array_equal(got["y"][k].reshape(-1), ref["y"]) and np.array_equal(got["rgba"][k].reshape(-1), ref["rgba"]), s
        assert np.array_equal(got["cb"][k].reshape(-1), ref["cb"]) and np.array_equal(got["cr"][k].reshape(-1), ref["cr"]), s
    again = bench_dump(tmp_path / "b", impl, streams, steps, warmup)
    for n in NAMES:
        assert np.array_equal(got[n], again[n]), n
