"""GRU models on the device path against the plain path they used before: the RNNLM step, the encoder recurrence and a
whole decode.

    python tools/bench_gru.py [--rows 20960,512,64] [--steps 20] [--repeats 3] [--enc-utts 2620] [--decode-utts 2620]
                              [--decode-rounds 2] [--out DIR]

RNNLM step: one step of a 4x1024 GRU LM (synth.LM_MODEL_CFG with module: GRU), tabled layer 0, rows gathered through a
parent index as in a decode.  Arms: the fused GRU stack (stepper._FusedLstm over the nn.GRU: split kernel, split-bf16
GEMMs, GRU cell kernel; CUDA-graph replay up to 4096 rows), the plain stepper._Rnn GRU step (fp32 F.linear + element-wise
ops + index_select of the states, embedding lookup included) and the fused LSTM stack of the same size.  CUDA events
over ``--steps`` steps, the arms alternating, ``--repeats`` times.
Encoder: one bidirectional GRU layer (H = 320, input 640, projection) over the utterances of synth.devclean_lengths after
the front end's 4x reduction: RecurrentLayer.forward_packed (split GEMM + persistent GRU kernel) against forward_ragged
(cuDNN GRU over 128-utterance padded chunks, as BatchedStepper.encode runs it), alternating.
Decode: BeamDecoder.decode_batch of a full-size all-GRU model (encoder, speller and RNNLM; beam 8, LM weight 0.5, joint
CTC 0.5) over devclean lengths.  The device path is the decoder as it stands; the plain arm is the routing GRU models had
before the GRU kernels: _Rnn stacks for the speller and the LM and the encoder through forward_ragged.  The number of
utterances whose 1-best differs between the two paths is reported.  The card's name and power limit are printed with the
numbers.
"""
import argparse
import copy
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
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


def _timed(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def lm_step_bench(rows, steps, repeats, dev):
    from e2e_asr_pytorch_b200 import synth
    from e2e_asr_pytorch_b200.decode import _Fp32Math
    from e2e_asr_pytorch_b200.stepper import _FusedLstm, _Rnn
    cfg = copy.deepcopy(synth.LM_MODEL_CFG)
    lm_lstm = synth.build_lm(31, cfg, seed=1).to(dev)
    cfg["module"] = "GRU"
    lm_gru = synth.build_lm(31, cfg, seed=1).to(dev)
    g = torch.Generator().manual_seed(0)
    tok = torch.randint(0, 31, (rows,), generator=g).to(dev)
    parent = torch.randint(0, rows, (rows,), generator=g).to(dev)
    res = {"rows": rows}
    with torch.no_grad(), _Fp32Math():
        arms = {}
        for name, lm in (("fused_gru", lm_gru), ("fused_lstm", lm_lstm)):
            st = _FusedLstm(lm.rnn, lm.emb.weight.detach())
            st.use_graphs = True
            st.start(rows, dev)

            def step(st=st):
                st.step(rows, tok=tok)
                st.reorder(parent)
            arms[name] = step
        plain = _Rnn(lm_gru.rnn, True, lm_gru.emb.weight.detach())
        state = [plain.zeros(rows, dev)]

        def plain_step():
            _, new = plain.step(lm_gru.emb(tok), state[0], rows, tok=tok)
            state[0] = _Rnn.gather(new, parent)
        arms["plain_gru"] = plain_step
        for fn in arms.values():                          # warm-up: library algorithms, graph capture of both parities
            for _ in range(4):
                fn()
        torch.cuda.synchronize()
        times = {k: [] for k in arms}
        for _ in range(repeats):
            for k, fn in arms.items():
                times[k].append(_timed(fn, steps))
        # the fused and the plain GRU step agree (one step from the same states)
        fused = _FusedLstm(lm_gru.rnn, lm_gru.emb.weight.detach())
        fused.start(rows, dev)
        top_f = fused.step(rows, tok=tok)
        top_p, _ = plain.step(lm_gru.emb(tok), plain.zeros(rows, dev), rows, tok=tok)
        res["max_abs_diff_fused_vs_plain"] = float((top_f - top_p).abs().max())
    for k, v in times.items():
        res[k + "_ms"] = min(v)
        res[k + "_ms_all"] = v
    res["plain_over_fused_gru"] = res["plain_gru_ms"] / res["fused_gru_ms"]
    res["fused_gru_over_fused_lstm"] = res["fused_gru_ms"] / res["fused_lstm_ms"]
    del arms, plain, state, fused
    torch.cuda.empty_cache()
    return res


def encoder_bench(utts, repeats, dev):
    from e2e_asr_pytorch_b200 import synth
    from e2e_asr_pytorch_b200.decode import _Fp32Math
    from e2e_asr_pytorch_b200.model import Encoder, RecurrentLayer, reference_init_
    torch.manual_seed(0)
    layer = RecurrentLayer(640, "GRU", 320, True, 0.0, False, 1, "drop", True)
    layer.apply(reference_init_)
    layer.eval().to(dev)
    assert layer.packed_supported()
    lens = np.sort(synth.devclean_lengths(utts) // 4)[::-1].copy()
    t_len = torch.as_tensor(lens)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(int(t_len.sum()), 640, generator=g).to(dev)
    off = (torch.cumsum(t_len, 0) - t_len).to(torch.int32).to(dev)
    first, rows = Encoder._groups(t_len)
    g_first = torch.tensor(first, dtype=torch.int32, device=dev)
    g_rows = torch.tensor(rows, dtype=torch.int32, device=dev)
    lens32 = t_len.to(torch.int32).to(dev)
    mask_all = torch.arange(int(t_len.max()), device=dev)[None, :] < t_len.to(dev)[:, None]
    chunks = []                                           # forward_ragged's input: 128-utterance padded chunks
    for lo in range(0, utts, 128):
        hi = min(utts, lo + 128)
        xc = x.new_zeros((hi - lo, int(t_len[lo]), 640))
        xc[mask_all[lo:hi, :int(t_len[lo])]] = x[int(off[lo]):int(off[hi - 1]) + int(t_len[hi - 1])]
        chunks.append((xc, t_len[lo:hi].to(dev), mask_all[lo:hi, :int(t_len[lo])]))

    def packed():
        return layer.forward_packed(x, off, lens32, g_first, g_rows)

    def ragged():
        return torch.cat([layer.forward_ragged(xc, lc)[0][m] for xc, lc, m in chunks], dim=0)
    with torch.no_grad(), _Fp32Math():
        a, b = packed(), ragged()
        torch.cuda.synchronize()
        diff = float((a - b).abs().max())
        times = {"packed": [], "ragged": []}
        for _ in range(repeats):
            times["packed"].append(_timed(packed, 1))
            times["ragged"].append(_timed(ragged, 1))
    res = {"utts": utts, "frames": int(t_len.sum()), "hidden": 320, "groups": len(first),
           "packed_ms": min(times["packed"]), "ragged_cudnn_ms": min(times["ragged"]),
           "packed_ms_all": times["packed"], "ragged_cudnn_ms_all": times["ragged"], "max_abs_diff": diff}
    res["speedup"] = res["ragged_cudnn_ms"] / res["packed_ms"]
    del chunks, x
    torch.cuda.empty_cache()
    return res


def decode_bench(utts, rounds, warm_utts, dev):
    from e2e_asr_pytorch_b200 import BeamDecoder, shard, synth
    from e2e_asr_pytorch_b200.stepper import BatchedStepper, _FusedLstm, _Rnn
    import yaml
    cfg = copy.deepcopy(synth.ASR_MODEL_CFG)
    cfg["encoder"]["module"] = "GRU"
    cfg["decoder"]["module"] = "GRU"
    lm_cfg = dict(synth.LM_MODEL_CFG, module="GRU")
    asr = synth.build_asr(31, cfg, seed=0)
    lm = synth.build_lm(31, lm_cfg, seed=1)
    decs = {}
    with tempfile.TemporaryDirectory(prefix="e2e_bench_gru_") as tmp:
        torch.save({"model": lm.state_dict()}, os.path.join(tmp, "lm.pth"))
        with open(os.path.join(tmp, "lm.yaml"), "w") as f:
            yaml.safe_dump({"model": lm_cfg}, f)
        for arm in ("device", "plain"):                   # one model copy per arm: the plain arm's encoder is re-routed
            d = BeamDecoder(copy.deepcopy(asr), None, 8, 0.01, 0.2, lm_path=os.path.join(tmp, "lm.pth"),
                            lm_config=os.path.join(tmp, "lm.yaml"), lm_weight=0.5, ctc_weight=0.5).to(dev)
            decs[arm] = d
    p = decs["plain"]
    p.asr.encoder.packed_supported = lambda: False        # encoder through forward_ragged (cuDNN GRU)
    knobs = (p.split_gemm, p.fused_attention, p.lm_split, p.vgg_split, p.step_graphs)
    st = BatchedStepper(p.asr, p.lm, p.split_gemm, p.fused_attention, p.lm_split, p.vgg_split, p.step_graphs)
    st.dec = _Rnn(p.asr.decoder.layers, p.split_gemm)     # the speller and LM stacks as plain GRU steps
    st.lm_rnn = _Rnn(p.lm.rnn, p.split_gemm, p.lm.emb.weight.detach())
    p._stepper = (dev, knobs, st)
    lengths = synth.devclean_lengths(utts)
    batches = shard.make_batches(np.arange(utts), lengths, 4096)
    data = [tuple(x.to(dev) for x in synth.padded_batch(b, lengths[b])) for b in batches]
    warm = tuple(x.to(dev) for x in synth.padded_batch(np.arange(warm_utts), lengths[:warm_utts]))

    def one_pass(arm):
        dec = decs[arm]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        outs = [dec.decode_batch(f, l, return_arrays=True) for f, l in data]
        torch.cuda.synchronize()
        s = dec._stepper[2]
        assert s.dec_fused == s.lm_fused == (arm == "device")
        return time.perf_counter() - t0, outs

    for arm in decs:
        decs[arm].decode_batch(*warm)
    rates = {arm: [] for arm in decs}
    first = {}
    for r in range(rounds):
        for arm in decs:
            dt, outs = one_pass(arm)
            rates[arm].append(utts / dt)
            first.setdefault(arm, outs)
    differ = 0
    for a, b in zip(first["device"], first["plain"]):
        for u in range(a[0].shape[0]):
            la, lb = int(a[2][u, 0]), int(b[2][u, 0])
            differ += int(la != lb or not torch.equal(a[0][u, 0, :la], b[0][u, 0, :lb]))
    return {"utts": utts, "batches": len(batches), "rounds": rounds, "utts_per_s_device": rates["device"],
            "utts_per_s_plain": rates["plain"], "speedup": max(rates["device"]) / max(rates["plain"]),
            "utterances_with_different_1best": differ}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", default="20960,512,64")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--enc-utts", type=int, default=2620)
    ap.add_argument("--decode-utts", type=int, default=2620)
    ap.add_argument("--decode-rounds", type=int, default=2)
    ap.add_argument("--decode-warm-utts", type=int, default=512)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    dev = torch.device("cuda:0")
    results = {"card": card()}
    print(json.dumps(results), flush=True)
    results["lm_step"] = []
    for rows in (int(x) for x in a.rows.split(",") if x):
        r = lm_step_bench(rows, a.steps, a.repeats, dev)
        results["lm_step"].append(r)
        print(json.dumps(r), flush=True)
    if a.enc_utts > 0:
        results["encoder"] = encoder_bench(a.enc_utts, a.repeats, dev)
        print(json.dumps(results["encoder"]), flush=True)
    if a.decode_utts > 0:
        results["decode"] = decode_bench(a.decode_utts, a.decode_rounds, min(a.decode_warm_utts, a.decode_utts), dev)
        print(json.dumps(results["decode"]), flush=True)
    results["card_after"] = card()
    print(json.dumps({"card_after": results["card_after"]}))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "bench_gru.json"), "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
