"""The encoder of config/librispeech_asr.yaml (no VGG, four BLSTM layers of 320 units, the second dropping every other
frame) on the packed device path against the route it took before (forward_ragged: cuDNN over 128-utterance padded
chunks).

    python tools/bench_encoder_subsample.py [--utts 2620] [--repeats 3] [--decode-rounds 2] [--out DIR]

Model: synth.ASR_MODEL_CFG with vgg: 0 and sample_rate [1, 2, 1, 1], random init; the 4x1024 RNNLM of synth.LM_MODEL_CFG.
Utterances: synth.devclean_lengths, sorted by decreasing length and encoded / decoded as ONE batch, as bench.py batches
them.
Encoder: BatchedStepper.encode with the packed routing (Encoder.forward_ragged_packed) and with the old one (the
encoder's packed_supported patched to refuse), alternating, CUDA events, ``--repeats`` times; max |packed - ragged| over
the rows t < enc_len.
Decode: BeamDecoder.decode_batch (beam 8, RNNLM weight 0.5, CTC weight 0.5) with either routing, alternating; utts/s and
the number of utterances whose 1-best differs between the two.
Memory: torch.cuda.max_memory_allocated over one packed decode next to shard.estimate_decode_bytes(..., time_reduction=2,
front_reduction=1), the estimate decode_dataset sizes its batches by.
The card's name and power limit are read in the same run.
"""
import argparse
import copy
import json
import os
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_gru import card  # noqa: E402


def yaml_encoder_cfg():
    from e2e_asr_pytorch_b200 import synth
    cfg = copy.deepcopy(synth.ASR_MODEL_CFG)
    cfg["encoder"].update({"vgg": 0, "sample_rate": [1, 2, 1, 1], "sample_style": "drop"})
    return cfg


def encoder_bench(asr, feats, lens, repeats):
    from e2e_asr_pytorch_b200.decode import _Fp32Math
    from e2e_asr_pytorch_b200.stepper import BatchedStepper
    enc = asr.encoder
    st = BatchedStepper(asr, None, split_gemm=True)
    supported = enc.packed_supported
    assert supported()

    def run(packed):
        enc.packed_supported = supported if packed else (lambda: False)
        try:
            return st.encode(feats, lens)
        finally:
            enc.packed_supported = supported
    times = {"packed": [], "ragged": []}
    with torch.no_grad(), _Fp32Math():
        a, la = run(True)
        b, lb = run(False)
        torch.cuda.synchronize()
        assert torch.equal(la, lb)
        t = min(a.shape[1], b.shape[1])
        m = torch.arange(t, device=a.device)[None, :] < la[:, None]
        diff = float((a[:, :t] - b[:, :t]).abs()[m].max())
        del a, b, m
        for _ in range(repeats):
            for arm in ("packed", "ragged"):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                out = run(arm == "packed")
                e1.record()
                torch.cuda.synchronize()
                times[arm].append(e0.elapsed_time(e1))
                del out
    res = {"utts": int(lens.numel()), "input_frames": int(lens.sum()), "longest": int(lens.max()),
           "packed_ms": min(times["packed"]), "ragged_ms": min(times["ragged"]),
           "packed_ms_all": times["packed"], "ragged_ms_all": times["ragged"],
           "max_abs_diff_rows_below_enc_len": diff}
    res["speedup"] = res["ragged_ms"] / res["packed_ms"]
    torch.cuda.empty_cache()
    return res


def decode_bench(asr, lm, feats, lens, rounds, warm, dev):
    from e2e_asr_pytorch_b200 import BeamDecoder, shard
    import yaml
    decs = {}
    with tempfile.TemporaryDirectory(prefix="e2e_bench_sub_") as tmp:
        torch.save({"model": lm.state_dict()}, os.path.join(tmp, "lm.pth"))
        with open(os.path.join(tmp, "lm.yaml"), "w") as f:
            from e2e_asr_pytorch_b200 import synth
            yaml.safe_dump({"model": synth.LM_MODEL_CFG}, f)
        for arm in ("packed", "ragged"):
            decs[arm] = BeamDecoder(copy.deepcopy(asr), None, 8, 0.01, 0.2, lm_path=os.path.join(tmp, "lm.pth"),
                                    lm_config=os.path.join(tmp, "lm.yaml"), lm_weight=0.5, ctc_weight=0.5).to(dev)
    decs["ragged"].asr.encoder.packed_supported = lambda: False
    for arm in decs:
        decs[arm].decode_batch(feats[:warm], lens[:warm])
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    rates = {arm: [] for arm in decs}
    first, peak = {}, None
    for r in range(rounds):
        for arm in decs:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = decs[arm].decode_batch(feats, lens, return_arrays=True)
            torch.cuda.synchronize()
            rates[arm].append(int(lens.numel()) / (time.perf_counter() - t0))
            if peak is None:                                  # the first pass is the packed one
                peak = torch.cuda.max_memory_allocated()
            first.setdefault(arm, out)
    a, b = first["packed"], first["ragged"]
    differ = 0
    for u in range(a[0].shape[0]):
        la, lb = int(a[2][u, 0]), int(b[2][u, 0])
        differ += int(la != lb or not torch.equal(a[0][u, 0, :la], b[0][u, 0, :lb]))
    d = decs["packed"]
    est = shard.estimate_decode_bytes(int(lens.numel()), int(lens.max()), d.asr.vocab_size, d.beam_size,
                                      d.ctc_beam_size if d.apply_ctc else 0, feat_dim=int(feats.shape[2]),
                                      time_reduction=d.asr.encoder.sample_rate, front_reduction=1)
    return {"utts": int(lens.numel()), "rounds": rounds, "utts_per_s_packed": rates["packed"],
            "utts_per_s_ragged": rates["ragged"], "speedup": max(rates["packed"]) / max(rates["ragged"]),
            "utterances_with_different_1best": differ,
            "peak_allocated_bytes": peak, "allocated_before_bytes": base,
            "peak_above_resident_bytes": peak - base + int(feats.numel()) * 4,
            "estimate_decode_bytes": est, "estimate_covers_peak": est >= peak}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=2620)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--decode-rounds", type=int, default=2)
    ap.add_argument("--warm-utts", type=int, default=256)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    from e2e_asr_pytorch_b200 import synth
    dev = torch.device("cuda:0")
    results = {"card": card()}
    print(json.dumps(results), flush=True)
    asr = synth.build_asr(31, yaml_encoder_cfg(), seed=0)
    lm = synth.build_lm(31, seed=1)
    lengths = synth.devclean_lengths(a.utts)
    order = np.argsort(-lengths, kind="stable")
    feats, lens = synth.padded_batch(order, lengths[order])
    feats, lens = feats.to(dev), lens.to(dev)
    enc_asr = copy.deepcopy(asr).to(dev)
    results["encoder"] = encoder_bench(enc_asr, feats, lens, a.repeats)
    print(json.dumps(results["encoder"]), flush=True)
    del enc_asr
    torch.cuda.empty_cache()
    if a.decode_rounds > 0:
        results["decode"] = decode_bench(asr, lm, feats, lens, a.decode_rounds, min(a.warm_utts, a.utts), dev)
        print(json.dumps(results["decode"]), flush=True)
    results["card_after"] = card()
    print(json.dumps({"card_after": results["card_after"]}), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "bench_encoder_subsample.json"), "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
