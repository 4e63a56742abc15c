"""``bench.py --dump-outputs`` on the GPU: the N-best it writes for its last timed pass is what ``BeamDecoder.decode_batch``
returns for the same utterances, batches and weights."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dump_outputs_equal_a_direct_decode(cuda, tmp_path):
    import bench
    from e2e_asr_pytorch_b200 import shard
    n_utts, out = 24, tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--n-utts", str(n_utts),
           "--no-cpu-baseline", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 2 and line["nbest_complete"] is True
    d = {k: np.load(str(out / (k + ".npy"))) for k in ("tokens", "token_scores", "lengths", "mean_scores", "nbest", "utterance_ids")}
    assert d["utterance_ids"].tolist() == list(range(n_utts))
    dec, _, _ = bench.build_models(cuda)
    lengths = bench.workload_lengths(1, n_utts)
    shards = shard.plan_shards(lengths, 1, bench.MAX_RATIO)
    checked = 0
    for ids in shard.make_batches(shards[0], lengths, 4096, 0):              # the bench's batches (its default arguments)
        feat, fl = bench.make_features(ids, lengths, pin=False)
        tok, sc, ln, avg, n = dec.decode_batch(feat.to(cuda), fl.to(cuda), return_arrays=True)
        for row, u in enumerate(ids):
            assert d["nbest"][u] == int(n[row]) > 0, u
            for k in range(int(n[row])):
                m = int(ln[row, k])
                assert d["lengths"][u, k] == m and d["mean_scores"][u, k] == float(avg[row, k]), (u, k)
                assert d["tokens"][u, k, :m].tolist() == tok[row, k, :m].tolist(), (u, k)
                assert np.array_equal(d["token_scores"][u, k, :m], sc[row, k, :m].numpy()), (u, k)
                assert not d["tokens"][u, k, m:].any() and not d["token_scores"][u, k, m:].any()
            checked += 1
    assert checked == n_utts
