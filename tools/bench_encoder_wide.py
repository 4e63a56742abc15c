"""Encoders with recurrent layers wider than 384 units (VGG + four BLSTM layers of H = 512 and of H = 1024 units per
direction) on the packed device path, whose recurrence then runs in the thread-block cluster form of csrc/lstm_seq.cu,
against the route such encoders took before (forward_ragged: cuDNN over 128-utterance padded chunks).

    python tools/bench_encoder_wide.py [--hidden 512 1024] [--utts 2620] [--repeats 3] [--decode-rounds 2] [--out DIR]

Model: synth.WIDE_ASR_CFG (synth.ASR_MODEL_CFG with dim [H]*4 and a 512-wide speller), random init; the 4x1024 RNNLM of
synth.LM_MODEL_CFG.  Utterances: synth.devclean_lengths, sorted by decreasing length and encoded / decoded as ONE batch,
as bench.py batches them.
Encoder and decode: tools/bench_encoder_subsample.py's measurements (CUDA events around BatchedStepper.encode with either
routing, alternating; max |packed - ragged| over the rows t < enc_len; beam 8 + RNNLM 0.5 + CTC 0.5 decodes with either
routing, alternating, utts/s and the number of differing 1-bests; peak torch.cuda.max_memory_allocated of a packed
decode).  The memory estimate is the one decode_dataset sizes its batches by (results.decode_bytes_fn).
The card's name and power limit are read in the same run.
"""
import argparse
import copy
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_encoder_subsample import decode_bench, encoder_bench  # noqa: E402
from tools.bench_gru import card  # noqa: E402


def wide_cfg(hidden):
    from e2e_asr_pytorch_b200 import synth
    cfg = copy.deepcopy(synth.WIDE_ASR_CFG)
    cfg["encoder"]["dim"] = [int(hidden)] * 4
    return cfg


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--hidden", type=int, nargs="+", default=[512, 1024])
    ap.add_argument("--utts", type=int, default=2620)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--decode-rounds", type=int, default=2)
    ap.add_argument("--warm-utts", type=int, default=256)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    from e2e_asr_pytorch_b200 import results as R, synth
    dev = torch.device("cuda:0")
    out = {"card": card(), "hidden": {}}
    print(json.dumps(out), flush=True)
    lm = synth.build_lm(31, seed=1)
    lengths = synth.devclean_lengths(a.utts)
    order = np.argsort(-lengths, kind="stable")
    feats, lens = synth.padded_batch(order, lengths[order])
    feats, lens = feats.to(dev), lens.to(dev)
    for h in a.hidden:
        asr = synth.build_asr(31, wide_cfg(h), seed=0)
        res = {"encoder_dims": [h] * 4, "decoder_dim": synth.WIDE_ASR_CFG["decoder"]["dim"]}
        enc_asr = copy.deepcopy(asr).to(dev)
        res["encoder"] = encoder_bench(enc_asr, feats, lens, a.repeats)
        print(json.dumps({"hidden": h, "encoder": res["encoder"]}), flush=True)
        del enc_asr
        torch.cuda.empty_cache()
        if a.decode_rounds > 0:
            d = decode_bench(asr, lm, feats, lens, a.decode_rounds, min(a.warm_utts, a.utts), dev)
            # decode_bench's estimate is that of an encoder without a front end; this one has the VGG front end and
            # a width above the estimate's default
            from e2e_asr_pytorch_b200 import BeamDecoder
            est_dec = BeamDecoder(asr, None, 8, 0.01, 0.2, ctc_weight=0.5)
            d["estimate_decode_bytes"] = R.decode_bytes_fn(est_dec, int(feats.shape[2]))(int(lens.numel()), int(lens.max()))
            d["estimate_covers_peak"] = d["estimate_decode_bytes"] >= d["peak_allocated_bytes"]
            d["estimate_enc_dim"] = max(640, R.encoder_width(asr.encoder))
            res["decode"] = d
            print(json.dumps({"hidden": h, "decode": d}), flush=True)
        out["hidden"][str(h)] = res
        del asr
        torch.cuda.empty_cache()
    out["card_after"] = card()
    print(json.dumps({"card_after": out["card_after"]}), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "bench_encoder_wide.json"), "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
