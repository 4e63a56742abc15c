"""Beam sizes up to 64 on the B200: decode throughput of the cfg3 model (V = 10000, max_len_ratio 0.07, RNNLM 0.5, CTC 0.5,
random init) across beams, the (3b) combine/prune step of the wide kernel against the narrow one, the prefix kernel's share
of a beam-64 step, and the beam-64 peak allocation against shard.estimate_decode_bytes.

    python tools/bench_wide_beam.py [--beams 8 16 32 48 64] [--utts 2620] [--out DIR]

Decodes: synth.devclean_lengths(utts), longest first, in the memory-budgeted batches decode_dataset would form
(results.decode_bytes_fn, 80 % of the free memory); each beam warms up on the 32 shortest utterances, then decodes the set
once with coarse phase marks (encode, steps, finalize summed over the batches).
(3b): one utterance batch of U = 128 with V = 10000, C = int(1.5 B), CTC + LM on, CUDA events around 50 launches after 5.
Prefix share: the first batch at beam 64 decoded again with an event pair around every prefix launch.
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np
import torch
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_gru import card  # noqa: E402

VOCAB, MIN_RATIO, MAX_RATIO, LM_W, CTC_W = 10000, 0.0, 0.07, 0.5, 0.5


def make_decoder(asr, lm_path, lm_cfg, beam, dev):
    from e2e_asr_pytorch_b200 import BeamDecoder
    return BeamDecoder(asr, None, beam, MIN_RATIO, MAX_RATIO, lm_path=lm_path, lm_config=lm_cfg, lm_weight=LM_W,
                       ctc_weight=CTC_W).to(dev)


def decode_set(dec, lengths, batches, dev, phases=True):
    from e2e_asr_pytorch_b200 import synth
    dec.profile_phases = "coarse" if phases else False
    ph = {}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for ids in batches:
        feat, fl = synth.padded_batch(ids, lengths[ids])
        dec.phase_ms = {}                                   # decode_batch adds to it
        dec.decode_batch(feat.to(dev), fl.to(dev), return_arrays="device")
        for k, v in dec.phase_ms.items():
            ph[k] = ph.get(k, 0.0) + v
    torch.cuda.synchronize()
    return time.perf_counter() - t0, ph


def combine_step_ms(beam, narrow, dev, U=128, reps=50):
    from e2e_asr_pytorch_b200 import ops
    rng = np.random.default_rng(beam)
    C = int(1.5 * beam)
    buf = ops.BeamBuffers(U, beam, C, 1000, torch.full((U,), 1000), torch.full((U,), 1000), dev)
    buf.n_live.fill_(beam)
    buf.n_active.fill_(beam)
    att = torch.from_numpy(rng.standard_normal((U * beam, VOCAB)).astype(np.float32) * 3).to(dev)
    lm = torch.from_numpy(rng.standard_normal((U * beam, VOCAB)).astype(np.float32) * 2).to(dev)
    ops.beam_candidates(att, U, beam, VOCAB, C, buf.n_active, buf.att_stats, buf.cand)
    buf.psi.copy_(torch.from_numpy(-rng.random(tuple(buf.psi.shape)).astype(np.float32) * 8))
    keep = ops.BEAM_NARROW_MAX
    ops.BEAM_NARROW_MAX = 32 if narrow else 0
    try:
        for s in range(5):
            ops.beam_combine_prune(buf, att, lm, VOCAB, 5 + s, CTC_W, LM_W, 1.5)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in range(reps):
            ops.beam_combine_prune(buf, att, lm, VOCAB, 10 + s, CTC_W, LM_W, 1.5)
        e1.record()
        torch.cuda.synchronize()
    finally:
        ops.BEAM_NARROW_MAX = keep
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--beams", type=int, nargs="+", default=[8, 16, 32, 48, 64])
    ap.add_argument("--utts", type=int, default=2620)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    from e2e_asr_pytorch_b200 import results as R, shard, synth
    dev = torch.device("cuda:0")
    out = {"card": card(), "utts": a.utts, "model": "cfg3: synth.build_asr(10000) + build_lm(10000), beam B, ctc 0.5, lm 0.5, "
           "max_len_ratio 0.07, random init", "decode": {}}
    print(json.dumps({"card": out["card"]}), flush=True)
    asr, lm = synth.build_asr(VOCAB, seed=0), synth.build_lm(VOCAB, seed=1)
    tmp = tempfile.mkdtemp(prefix="e2e_wide_beam_")
    lm_path, lm_cfg = os.path.join(tmp, "lm.pth"), os.path.join(tmp, "lm.yaml")
    torch.save({"model": lm.state_dict()}, lm_path)
    yaml.safe_dump({"model": synth.LM_MODEL_CFG}, open(lm_cfg, "w"))
    lengths = synth.devclean_lengths(a.utts)
    idx = list(range(a.utts))
    shortest = sorted(idx, key=lambda i: lengths[i])[:32]

    # (3b) per step
    out["combine_prune_ms"] = {"U": 128, "V": VOCAB,
                               "B32_narrow": combine_step_ms(32, True, dev), "B32_wide": combine_step_ms(32, False, dev),
                               "B64_wide": combine_step_ms(64, False, dev)}
    print(json.dumps({"combine_prune_ms": out["combine_prune_ms"]}), flush=True)

    for beam in a.beams:
        dec = make_decoder(asr, lm_path, lm_cfg, beam, dev)
        free = torch.cuda.mem_get_info(dev)[0]
        bytes_fn = R.decode_bytes_fn(dec, synth.FEAT_DIM)
        batches = shard.make_batches(idx, lengths, max_utts=4096, max_bytes=int(0.8 * free), bytes_fn=bytes_fn)
        decode_set(dec, lengths, [shortest], dev, phases=False)                 # warm-up
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        secs, ph = decode_set(dec, lengths, batches, dev)
        rec = {"utts_per_s": a.utts / secs, "seconds": secs, "batches": len(batches),
               "phases_ms": {k: round(v, 3) for k, v in ph.items()}}
        if beam == max(a.beams):
            # peak of the set's decode (its first batch holds the longest utterances and is the largest) against the
            # estimate of that batch, which is what sized it
            first = batches[0]
            kw = {k: v for k, v in bytes_fn.keywords.items() if k not in ("vocab", "beam", "n_cand")}
            n_cand = bytes_fn.keywords["n_cand"]
            l_max = int(max(lengths[i] for i in first))
            est = shard.estimate_decode_bytes(len(first), l_max, VOCAB, beam, n_cand, **kw)
            out["memory"] = {"n_utts": len(first), "l_max": l_max, "vocab": VOCAB, "beam": beam, "n_cand": n_cand,
                             "estimate_kwargs": kw, "estimate_bytes": int(est),
                             "peak_bytes": int(torch.cuda.max_memory_allocated(dev)), "allocated_before_bytes": int(base),
                             "what": "peak torch.cuda.max_memory_allocated over the whole set's decode (models included); "
                                     "estimate of the first (largest) batch"}
            # the prefix kernel's share of a step: the first batch again with an event pair around every prefix launch
            dec.profile_prefix = True
            dec.prefix_events = []
            _, ph1 = decode_set(dec, lengths, [first], dev)
            pre = sum(e0.elapsed_time(e1) for e0, e1, _, _ in dec.prefix_events)
            dec.profile_prefix = False
            rec["prefix_share"] = {"prefix_ms": pre, "steps_ms": ph1.get("steps"), "share": pre / ph1["steps"] if ph1.get("steps") else None,
                                   "batch_utts": len(first), "note": "events around each prefix launch slow the steps slightly"}
        out["decode"][str(beam)] = rec
        print(json.dumps({"beam": beam, **rec}), flush=True)
        del dec
        torch.cuda.empty_cache()
    out["card_after"] = card()
    print(json.dumps({"memory": out.get("memory"), "card_after": out["card_after"]}), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "r07_wide_beam.json"), "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
