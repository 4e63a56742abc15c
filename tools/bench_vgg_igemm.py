"""A/B micro-benchmark of the VGG convolutions on one encoder chunk, both paths in one process on the same weights and
activations: the tcgen05 implicit split GEMM (csrc/conv_igemm.cu) against unfold + three library GEMMs + epilogue kernel.

    python tools/bench_vgg_igemm.py [--utts 128] [--frames 720] [--steps 10] [--out FILE.jsonl]

Per layer (128->128 pooled, 128->256, 256->256 pooled) it prints one JSON line with
  - layer_ms: the whole layer on each path (unfold: VGGFrontEnd._conv_split; igemm: ops.conv3x3_igemm with its epilogue),
  - core_ms / core_tflops: the GEMM work alone — the three library GEMMs on an operand unfolded beforehand, and the
    implicit GEMM with the raw epilogue (its split of the input included) — as bf16 tensor-core work
    (2 * pixels * Cout * 9C * 6 partial products) per second, next to MEASURED_PEAKS.json's bf16 rate if that file exists,
  - equal: whether the two paths' outputs are bit-identical.
A last line times the whole front end (forward_masked_split) with conv_path "unfold" and "igemm" (the implicit GEMM for
the layers VGGFrontEnd routes to it).  The GPU name and power limit go in every line.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _gpu():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
        return q.stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        return torch.cuda.get_device_name()


def _bf16_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except (OSError, ValueError):
        return None
    for k, v in peaks.items():
        if "bf16" in k.lower():
            return v
    return None


def _time(fn, steps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=128, help="utterances per encoder chunk (stepper.encode uses 128)")
    ap.add_argument("--frames", type=int, default=720, help="feature frames of the longest utterance")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    from e2e_asr_pytorch_b200 import ops
    from e2e_asr_pytorch_b200.model import VGGFrontEnd, reference_init_
    from e2e_asr_pytorch_b200.decode import _Fp32Math
    dev = torch.device("cuda:0")
    gpu, peak = _gpu(), _bf16_peak()
    torch.manual_seed(0)
    vgg = VGGFrontEnd(160)
    vgg.apply(reference_init_)
    vgg.eval().to(dev)
    g = torch.Generator().manual_seed(1)
    lens = torch.sort(torch.randint(a.frames // 2, a.frames + 1, (a.utts,), generator=g) // 4 * 4, descending=True)[0]
    lens[0] = a.frames // 4 * 4
    feat = torch.randn(a.utts, int(lens[0]), 160, generator=g)
    for i, l in enumerate(lens):
        feat[i, int(l):] = 0
    feat, lens = feat.to(dev), lens.to(dev)
    lines = []
    convs = [m for m in vgg.extractor if isinstance(m, torch.nn.Conv2d)]
    with torch.no_grad(), _Fp32Math():
        own = lens // 4 * 4
        v1, v2 = own.to(torch.int32).contiguous(), (own // 2).to(torch.int32).contiguous()
        x = ops.conv1_direct(feat, convs[0].weight.detach().float().contiguous(), convs[0].bias.detach().float().contiguous(),
                             v1, vgg.freq_dim)
        for conv, valid, pool in ((convs[1], v1, True), (convs[2], v2, False), (convs[3], v2, True)):
            n, h, w, c = x.shape
            k, total, cout = 9 * c, n * h * w, conv.out_channels
            res = {"bench": "vgg_igemm_layer", "gpu": gpu, "layer": "%d->%d%s" % (c, cout, " pool" if pool else ""),
                   "utts": n, "H": h, "W": w}
            lin, wsplit = vgg._split_weights(conv), vgg._igemm_weights(conv)
            bias = conv.bias.detach().float().contiguous()
            vgg.conv_path = "unfold"
            run = {"unfold": lambda: vgg._conv_split(x, valid, conv, pool=pool),
                   "igemm": lambda: ops.conv3x3_igemm(x, valid, wsplit, bias, "pool" if pool else "relu")}
            outs = {}
            for path in ("unfold", "igemm"):
                res.setdefault("layer_ms", {})[path] = _time(run[path], a.steps)
                outs[path] = run[path]()
            res["equal"] = bool(torch.equal(outs["unfold"], outs["igemm"]))
            blk = max(1, min(total, vgg.A_BYTES // (3 * k * 2)))
            am = torch.empty((blk, 3 * k), dtype=torch.bfloat16, device=dev)
            ops.conv3x3_unfold_split(x, valid, 0, blk, am)
            ym = torch.empty((blk, cout), dtype=torch.float32, device=dev)

            def library():
                torch.mm(am, lin.b2, out_dtype=torch.float32, out=ym)
                torch.addmm(ym, am[:, :2 * k], lin.b1, out_dtype=torch.float32, out=ym)
                torch.addmm(ym, am[:, :k], lin.b0, out_dtype=torch.float32, out=ym)
            flop = 2.0 * cout * k * 6
            t_lib = _time(library, a.steps)
            t_ig = _time(lambda: ops.conv3x3_igemm(x, valid, wsplit, None, "raw"), a.steps)
            res["core_ms"] = {"library_gemms_%d_rows" % blk: t_lib, "igemm_raw_%d_rows" % total: t_ig}
            res["core_tflops"] = {"library": flop * blk / t_lib / 1e9, "igemm": flop * total / t_ig / 1e9}
            res["core_rate_vs_library"] = res["core_tflops"]["igemm"] / res["core_tflops"]["library"]
            res["measured_bf16_peak"] = peak
            del am, ym
            lines.append(res)
            print(json.dumps(res), flush=True)
            x = outs["igemm"]
        fe = {"bench": "vgg_igemm_front_end", "gpu": gpu, "utts": a.utts, "frames": int(lens[0])}
        outs = {}
        for path in ("unfold", "igemm"):
            vgg.conv_path = path
            fe.setdefault("ms_per_chunk", {})[path] = _time(lambda: vgg.forward_masked_split(feat, lens), a.steps)
            outs[path] = vgg.forward_masked_split(feat, lens)[0]
        fe["equal"] = bool(torch.equal(outs["unfold"], outs["igemm"]))
        lines.append(fe)
        print(json.dumps(fe), flush=True)
    if a.out:
        with open(a.out, "a") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
