"""What decoding with the word-embedding fusion plug-in costs on the device path.

    python tools/bench_emb_fusion.py [--utts 2620] [--repeats 2] [--out DIR]

Workloads (bench.py's models and decode settings, random init): cfg2 (V = 31) and cfg3 (V = 10000, max_len_ratio 0.07,
memory-budgeted batches as tools/bench_config.py sizes them), beam 8 + RNNLM (weight 0.5) + CTC (weight 0.5), the
synth.devclean_lengths set, each decoded without the plug-in and with it (E = 300; a fixed lambda = 0.3 with a fixed
temperature 1, and a per-entry learnable lambda and temperature).  Features are device resident; each variant is
decoded once to warm up and ``--repeats`` times timed (CUDA events), alternating variants.

Per step, at the rows of the first decode steps (utterances x beam): CUDA-event time of the plug-in's GEMMs (emb_net +
table product, stepper.EmbFusion.logits), of the fusion kernel (e2e_emb_fuse_candidates) and, for scale, of char_trans
and of the kernel it replaces (e2e_beam_candidates).  The kernel's bytes: 12 per row entry (both logit rows read, the
fused row written) + 4 per candidate + 8 of statistics, over its time, as a fraction of the HBM bandwidth measured in
the same run (a device-to-device copy of 4 GiB).  At V = 31 the kernel's 5 MB of inputs sit in L2, so that fraction is
nominal there.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_gru import card  # noqa: E402

BEAM, CTC_W, LM_W, MIN_RATIO, E_DIM = 8, 0.5, 0.5, 0.01, 300
WORKLOADS = {"cfg2": (31, 0.2), "cfg3": (10000, 0.07)}
FUSION = {"off": None, "fixed": dict(fuse=0.3, temperature=1.0), "learnable": dict(fuse=-2, temperature=-2)}


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def hbm_peak_gbs(dev):
    a = torch.empty(1 << 30, dtype=torch.float32, device=dev)
    b = torch.empty_like(a)
    ms = timed(lambda: b.copy_(a), 20)
    del a, b
    return 2 * 4 * (1 << 30) / ms / 1e6


def step_parts(asr, emb, rows, vocab, dev):
    """CUDA-event ms of one step's plug-in GEMMs and fusion kernel (and of char_trans / (3a)) at ``rows`` rows."""
    from e2e_asr_pytorch_b200 import ops
    from e2e_asr_pytorch_b200.decode import _Fp32Math
    from e2e_asr_pytorch_b200.stepper import EmbFusion
    fus = EmbFusion(emb)
    n_cand, u = int(1.5 * BEAM), rows // BEAM
    g = torch.Generator(device=dev).manual_seed(0)
    top = torch.randn(rows, asr.dec_dim, device=dev, generator=g)
    n_live = torch.full((u,), BEAM, dtype=torch.int32, device=dev)
    stats = torch.empty(rows, 2, device=dev)
    cand = torch.empty(rows, n_cand, dtype=torch.int32, device=dev)
    out = torch.empty(rows, vocab, device=dev)
    with torch.no_grad(), _Fp32Math():
        dec_logits = asr.decoder.char_trans(top).contiguous()
        emb_logits = fus.logits(top).contiguous()
        t_gemm = timed(lambda: fus.logits(top), 20)
        t_char = timed(lambda: asr.decoder.char_trans(top), 20)
        t_kern = timed(lambda: ops.emb_fuse_candidates(dec_logits, emb_logits, u, BEAM, vocab, n_cand, fus.scale, fus.lam, fus.eps,
                                                       n_live, out, stats, cand), 50)
        t_cand = timed(lambda: ops.beam_candidates(dec_logits, u, BEAM, vocab, n_cand, n_live, stats, cand), 50)
    flop = 2 * rows * (asr.dec_dim * emb.emb_net[0].out_features + emb.emb_net[0].out_features * E_DIM + E_DIM * vocab)
    nbytes = rows * (12 * vocab + 4 * n_cand + 8)
    return {"rows": rows, "emb_gemms_ms": t_gemm, "emb_gemms_tflops": flop / t_gemm / 1e9, "char_trans_ms": t_char,
            "fuse_kernel_ms": t_kern, "beam_candidates_ms": t_cand, "fuse_kernel_bytes": nbytes,
            "fuse_kernel_gbs": nbytes / t_kern / 1e6}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=2620)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--workloads", default="cfg2,cfg3")
    ap.add_argument("--out", default="", help="directory for emb_fusion.json (default: the JSON line on stdout only)")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a B200"
    import yaml
    from e2e_asr_pytorch_b200 import BeamDecoder, shard, synth
    dev = torch.device("cuda", 0)
    result = {"card": card(), "hbm_copy_gbs": hbm_peak_gbs(dev), "workloads": {}}
    lengths = synth.devclean_lengths(a.utts)
    for name in a.workloads.split(","):
        vocab, max_ratio = WORKLOADS[name]
        asr = synth.build_asr(vocab, seed=0)
        lm = synth.build_lm(vocab, seed=1)
        tmp = tempfile.mkdtemp(prefix="e2e_emb_bench_")
        torch.save({"model": lm.state_dict()}, os.path.join(tmp, "lm.pth"))
        yaml.safe_dump({"model": synth.LM_MODEL_CFG}, open(os.path.join(tmp, "lm.yaml"), "w"))
        if vocab > 31:
            import functools
            fn = functools.partial(shard.estimate_decode_bytes, vocab=vocab, beam=BEAM, n_cand=int(1.5 * BEAM))
            batches = shard.make_batches(range(len(lengths)), lengths, 4096, None, int(0.8 * 178e9), fn)
        else:
            batches = shard.make_batches(range(len(lengths)), lengths, 4096)
        feats = []
        for b in batches:
            f, l = synth.padded_batch(b, [lengths[i] for i in b])
            feats.append((f.to(dev), l.to(dev)))
        decs = {}
        for kind, kw in FUSION.items():
            emb = synth.build_emb(vocab, asr.dec_dim, E_DIM, seed=3, **kw) if kw else None
            decs[kind] = BeamDecoder(asr, emb, BEAM, MIN_RATIO, max_ratio, lm_path=os.path.join(tmp, "lm.pth"),
                                     lm_config=os.path.join(tmp, "lm.yaml"), lm_weight=LM_W, ctc_weight=CTC_W).to(dev)
        times = {k: [] for k in decs}

        def one(kind):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for f, l in feats:
                decs[kind].decode_batch(f, l, return_arrays="device")
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1)
        for kind in decs:
            one(kind)
        for _ in range(a.repeats):
            for kind in decs:
                times[kind].append(one(kind))
        rec = {"vocab": vocab, "max_len_ratio": max_ratio, "utterances": len(lengths), "batches": len(batches), "decode": {}}
        for kind in decs:
            ms = float(np.median(times[kind]))
            rec["decode"][kind] = {"ms": times[kind], "utts_per_s": len(lengths) / (ms / 1e3)}
        rows = min(len(lengths), 4096) * BEAM
        rec["per_step"] = {}
        for kind in ("fixed", "learnable"):
            part = step_parts(asr, decs[kind].emb_decoder, rows, vocab, dev)
            part["fuse_kernel_frac_of_hbm"] = part["fuse_kernel_gbs"] / result["hbm_copy_gbs"]
            rec["per_step"][kind] = part
        result["workloads"][name] = rec
        print(json.dumps({name: rec}), flush=True)
        del decs, feats
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "emb_fusion.json"), "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
