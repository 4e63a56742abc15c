"""Multi-head location-aware attention: the fused step against the plain PyTorch multi-head step it replaces, and the
whole-decode rate of a multi-head full-size model with the fused kernel on and off.

    python tools/bench_heads.py [--heads 1,2,4] [--vproj 0] [--utts 2620] [--frames 180] [--beam 8] [--steps 20]
                                [--decode-heads 4] [--decode-utts 2620] [--decode-rounds 2] [--out DIR]

Step: the batched stepper's attention step (BatchedStepper._attend: keys / values / alignments laid out as a decode
lays them out, merge_head included for H > 1) at the bench shape (2620 utterances x 180 frames, beam 8, A = 300,
K = 10, W = 201, E = 640), timed with CUDA events over ``--steps`` steps after a warm-up, fused and plain alternating.
Decode: BeamDecoder.decode_batch on the full-size model (synth.ASR_MODEL_CFG with num_head = H, beam 8 + RNNLM, joint
CTC) over cfg2 lengths (synth.devclean_lengths), fused_attention on and off alternating, ``--decode-rounds`` passes
each after one warm-up pass each.  The card's name and power limit are printed with the numbers.
"""
import argparse
import copy
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = ""
    return q or torch.cuda.get_device_name(0)


def step_bench(heads, v_proj, utts, frames, beam, steps, dev):
    from e2e_asr_pytorch_b200 import synth
    from e2e_asr_pytorch_b200.decode import _Fp32Math
    from e2e_asr_pytorch_b200.stepper import BatchedStepper
    cfg = copy.deepcopy(synth.ASR_MODEL_CFG)
    cfg["attention"].update({"num_head": heads, "v_proj": bool(v_proj)})
    asr = synth.build_asr(31, cfg, seed=0).to(dev)
    g = torch.Generator().manual_seed(0)
    enc = torch.randn(utts, frames, 640, generator=g).to(dev)
    enc_len = torch.full((utts,), frames, dtype=torch.long, device=dev)
    a_dim = cfg["attention"]["dim"]
    query = torch.tanh(torch.randn(utts * beam, heads * a_dim, generator=g)).to(dev)
    res = {}
    with torch.no_grad(), _Fp32Math():
        st = {name: BatchedStepper(asr, None, fused_attention=fused) for name, fused in (("fused", True), ("plain", False))}
        for name, s in st.items():
            s.start(enc, enc_len, beam)
            assert s.fused_step == (name == "fused"), name
            for _ in range(3):
                s._attend(query, utts)
        torch.cuda.synchronize()
        times = {name: [] for name in st}
        for _ in range(2):                               # alternate the two paths
            for name, s in st.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(steps):
                    s._attend(query, utts)
                e1.record()
                torch.cuda.synchronize()
                times[name].append(e0.elapsed_time(e1) / steps)
        a_f, c_f = st["fused"]._attend(query, utts)
        a_p, c_p = st["plain"]._attend(query, utts)
        res = {"heads": heads, "v_proj": int(bool(v_proj)), "utts": utts, "frames": frames, "beam": beam,
               "fused_ms": min(times["fused"]), "plain_ms": min(times["plain"]), "fused_ms_all": times["fused"],
               "plain_ms_all": times["plain"], "max_abs_diff_attn": float((a_f.reshape(a_p.shape) - a_p).abs().max()),
               "max_abs_diff_context": float((c_f - c_p).abs().max())}
        res["speedup"] = res["plain_ms"] / res["fused_ms"]
        # device time of each fused kernel, in a profiled run of its own after the timed ones
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(steps):
                st["fused"]._attend(query, utts)
            torch.cuda.synchronize()
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA and "attention_" in ev.name:
                k = "energy_kernel_us" if "energy" in ev.name else "softmax_context_kernel_us"
                res[k] = res.get(k, 0.0) + ev.device_time / steps
    del st
    torch.cuda.empty_cache()
    return res


def decode_bench(heads, v_proj, utts, rounds, max_utts, dev):
    import tempfile
    import numpy as np
    import yaml
    from e2e_asr_pytorch_b200 import BeamDecoder, shard, synth
    cfg = copy.deepcopy(synth.ASR_MODEL_CFG)
    cfg["attention"].update({"num_head": heads, "v_proj": bool(v_proj)})
    asr = synth.build_asr(31, cfg, seed=0)
    lm = synth.build_lm(31, seed=1)
    decs = {}
    with tempfile.TemporaryDirectory(prefix="e2e_bench_heads_") as tmp:
        torch.save({"model": lm.state_dict()}, os.path.join(tmp, "lm.pth"))
        with open(os.path.join(tmp, "lm.yaml"), "w") as f:
            yaml.safe_dump({"model": synth.LM_MODEL_CFG}, f)
        for fused in (True, False):                      # one decoder per setting: each keeps its own stepper and graphs
            d = BeamDecoder(asr, None, 8, 0.01, 0.2, lm_path=os.path.join(tmp, "lm.pth"), lm_config=os.path.join(tmp, "lm.yaml"),
                            lm_weight=0.5, ctc_weight=0.5).to(dev)
            d.fused_attention = fused
            decs[fused] = d
    lengths = synth.devclean_lengths(utts)
    batches = shard.make_batches(np.arange(utts), lengths, max_utts)
    data = [tuple(x.to(dev) for x in synth.padded_batch(b, lengths[b])) for b in batches]

    def one_pass(fused):
        dec = decs[fused]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        outs = [dec.decode_batch(f, l, return_arrays=True) for f, l in data]
        torch.cuda.synchronize()
        assert dec._stepper[2].fused_step == fused
        return time.perf_counter() - t0, outs

    rates = {True: [], False: []}
    first = {}
    for fused in (True, False):
        _, first[fused] = one_pass(fused)                # warm-up (and the outputs compared below)
    for _ in range(rounds):
        for fused in (True, False):
            dt, _ = one_pass(fused)
            rates[fused].append(utts / dt)
    same = sum(int(torch.equal(a[0][:, 0], b[0][:, 0]) and torch.equal(a[2][:, 0], b[2][:, 0])) for a, b in zip(first[True], first[False]))
    return {"heads": heads, "v_proj": int(bool(v_proj)), "utts": utts, "batches": len(batches), "rounds": rounds,
            "utts_per_s_fused": rates[True], "utts_per_s_plain": rates[False],
            "batches_with_identical_1best_arrays": same}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--heads", default="1,2,4")
    ap.add_argument("--vproj", type=int, default=0)
    ap.add_argument("--utts", type=int, default=2620)
    ap.add_argument("--frames", type=int, default=180)
    ap.add_argument("--beam", type=int, default=8)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--decode-heads", type=int, default=4)
    ap.add_argument("--decode-utts", type=int, default=2620)
    ap.add_argument("--decode-rounds", type=int, default=2)
    ap.add_argument("--decode-max-utts", type=int, default=1024)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    dev = torch.device("cuda:0")
    results = {"card": card()}
    print(json.dumps(results), flush=True)
    results["step"] = []
    for h in (int(x) for x in a.heads.split(",") if x):
        r = step_bench(h, a.vproj, a.utts, a.frames, a.beam, a.steps, dev)
        results["step"].append(r)
        print(json.dumps(r), flush=True)
    one = [r for r in results["step"] if r["heads"] == 1 and "energy_kernel_us" in r]
    if one:                                              # measured energy-kernel time over H = 1, beside (1+H)/2
        results["energy_kernel_ratio"] = {r["heads"]: {"measured": r["energy_kernel_us"] / one[0]["energy_kernel_us"],
                                                       "mufu_estimate": (1 + r["heads"]) / 2} for r in results["step"]}
        print(json.dumps({"energy_kernel_ratio": results["energy_kernel_ratio"]}), flush=True)
    if a.decode_heads > 0 and a.decode_utts > 0:
        r = decode_bench(a.decode_heads, a.vproj, a.decode_utts, a.decode_rounds, a.decode_max_utts, dev)
        results["decode"] = r
        print(json.dumps(r), flush=True)
    results["card_after"] = card()
    print(json.dumps({"card_after": results["card_after"]}))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "bench_heads.json"), "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
