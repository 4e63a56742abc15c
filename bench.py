#!/usr/bin/env python
"""bench.py — beam-8 + RNNLM joint CTC/attention decode throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): char (31-token) VGG+BLSTM CTC-attention model with
librispeech_asr.yaml dims + random-init 4x1024 RNNLM, beam 8, ctc_weight 0.5, lm_weight 0.5,
2620 synthetic utterances with a dev-clean-like length distribution per GPU (weak scaling:
N GPUs decode N x 2620 utterances, sharded by utterance, one all-gather of the N-best).
A "step" is one pass of the hot path over that whole set.

Prints ONE JSON line (rank 0).  ``value`` = utterances/s with the features already resident in
HBM; ``e2e`` = the same through BeamDecoder.decode_batch_from_host with pinned HOST features (the
valid frames copied inside the timed region, pipelined under the encoder; the ragged N-best packed
on the device, gathered and read back to pinned host memory).  ``roofline`` describes the fused
prefix-score step kernel, timed live with CUDA events around every launch; ``phases_ms`` is the
per-phase breakdown of a pass (max over ranks); ``nbest_parity`` compares the run's own N-best of
the 16 bench-set utterances in tests/golden/beam_nbest_fullsize.npz with the reference's;
``sharded_equals_single`` (N > 1) is the bit-for-bit check of the gathered result against rank 0's
own decode of the last rank's shard.  ``--dump-outputs DIR`` writes the N-best arrays of the last timed pass
(``dump_outputs``); inputs and weights are seeded, so runs with the same arguments decode the same data.
``--impl reference`` times the UNMODIFIED reference on the host cores: its decode path byte-compiled
into oracle/_ref by __graft_entry__.build() (oracle/ref_stage.py), driven through
bin/test_asr.py::beam_decode and joblib.Parallel on a length-stratified sample of the same set.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BEAM, CTC_W, LM_W, MIN_RATIO, MAX_RATIO, VOCAB = 8, 0.5, 0.5, 0.01, 0.2, 31
N_UTTS = 2620
METRIC = "beam-8+LM joint CTC/attn decode utts/sec"
MEDIAN_NOTE = ", the workload's median length"
GOLDEN_APPLIES = True      # tests/golden/beam_nbest_fullsize.npz holds utterances of THIS workload (tools/bench_config.py clears it)


def kernel_source_sha():
    """Hash of the sources the prefix-score kernels are built from: an ncu capture is only quoted while it matches."""
    import hashlib
    h = hashlib.sha256()
    for f in ("prefix_lazy.cu", "prefix_score.cu", "common.cuh", "softplus_poly.inc", "softplus_lut.inc"):
        with open(os.path.join(ROOT, "e2e-asr-pytorch_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def load_traffic():
    """DRAM bytes per prefix-score launch, averaged over the launches of one timed pass of this same command under ncu
    (profiles/r02_prefix_traffic_inbench.json; tools/summarize_ncu.py made it).  The file carries the hash of the kernel
    sources it was captured from: a capture of another kernel version is not quoted (null)."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_prefix_traffic_inbench.json")))
        if d.get("kernel_source_sha") != kernel_source_sha():
            return None, "profiles/r02_prefix_traffic_inbench.json is of another kernel version (stale): not quoted"
        return float(d["dram_bytes_per_launch"]), "profiles/r02_prefix_traffic_inbench.json (ncu dram__bytes_read+write, mean over the launches of a pass)"
    except Exception:
        return None, None


def load_peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------
def workload_lengths(world, n_utts=N_UTTS):
    from e2e_asr_pytorch_b200 import synth
    # replica r uses the same length distribution with its own seed (cfg5: "8 x 2620 utts")
    return np.concatenate([synth.devclean_lengths(n_utts, seed=2 + r) for r in range(world)])


def build_models(device):
    from e2e_asr_pytorch_b200 import BeamDecoder, synth
    import tempfile
    import yaml
    asr = synth.build_asr(VOCAB, seed=0)
    lm = synth.build_lm(VOCAB, seed=1)
    tmp = tempfile.mkdtemp(prefix="e2e_bench_")
    torch.save({"model": lm.state_dict()}, os.path.join(tmp, "lm.pth"))
    yaml.safe_dump({"model": synth.LM_MODEL_CFG}, open(os.path.join(tmp, "lm.yaml"), "w"))
    dec = BeamDecoder(asr, None, BEAM, MIN_RATIO, MAX_RATIO, lm_path=os.path.join(tmp, "lm.pth"),
                      lm_config=os.path.join(tmp, "lm.yaml"), lm_weight=LM_W, ctc_weight=CTC_W)
    if device is not None:
        dec = dec.to(device)
    return dec, asr, lm


def make_features(ids, lengths, pin):
    """Host features of the utterances ``ids`` (seeded per utterance), zero padded."""
    from e2e_asr_pytorch_b200 import synth
    return synth.padded_batch(ids, [lengths[i] for i in ids], pin=pin)


def golden_parity(tok, sc, ln, avg, nn, tie_tol=5e-4, score_tol=2e-4):
    """The bench's own N-best of the utterances of its set that tests/golden/beam_nbest_fullsize.npz holds (decoded there
    by the UNMODIFIED reference, tools/make_golden.py) against the reference's: identical 1-best, or a tie by the
    REFERENCE's scores (the device 1-best is in the reference N-best within tie_tol of its best)."""
    path = os.path.join(ROOT, "tests", "golden", "beam_nbest_fullsize.npz")
    if not os.path.exists(path):
        return None
    g = np.load(path, allow_pickle=False)
    out = {"identical": 0, "ties": 0, "not_in_reference_nbest": 0, "n": 0, "max_score_diff": 0.0}
    for c in range(int(g["n_cases"])):
        u, n_frames = int(g["case%d_utt" % c]), int(g["case%d_len" % c])
        if u >= tok.shape[0]:
            continue                                   # a fixture outside the bench set (the short ones of the tests)
        out["n"] += 1
        m = int(ln[u, 0])
        mine = tok[u, 0, :m].tolist()
        ref = [(g["case%d_tok%d" % (c, j)].tolist(), float(g["case%d_avg%d" % (c, j)])) for j in range(int(g["case%d_nbest" % c]))]
        if mine == ref[0][0]:
            out["identical"] += 1
            out["max_score_diff"] = max(out["max_score_diff"], abs(float(avg[u, 0]) - ref[0][1]))
        elif any(mine == r[0] and abs(r[1] - ref[0][1]) < tie_tol for r in ref):
            out["ties"] += 1
        else:
            out["not_in_reference_nbest"] += 1         # the search paths diverged early (runner-up gaps of this random-init workload are
    out["tie_tol"] = tie_tol                            # 1e-5 .. 7e-4); tests/test_gpu_fullsize_golden.py audits these by rescoring
    return out


DUMP_BYTES = 64 * 1000 * 1000


def dump_outputs(out_dir, tok, sc, ln, avg, n, budget=DUMP_BYTES):
    """Write the N-best arrays of a pass (what ``BeamDecoder.decode_batch(..., return_arrays=True)`` returns, indexed by
    utterance) to ``out_dir`` as float32 .npy files: ``tokens`` and ``token_scores`` [U, beam, width], ``lengths`` and
    ``mean_scores`` [U, beam], ``nbest`` [U], plus ``utterance_ids`` (float64) naming each row.  Entries a caller never
    reads (past a hypothesis' length, hypotheses past the N-best count) are written as 0, so two builds can be compared
    array for array.  If all rows would take more than ``budget`` bytes, a fixed seeded sample of utterances is written,
    in id order."""
    tok, sc, ln, avg, n = (t.cpu().numpy() for t in (tok, sc, ln, avg, n))
    n_utts, beam, width = tok.shape
    row_bytes = 4 * (2 * beam * width + 2 * beam + 1) + 8
    room = budget - 6 * 1024                                      # the six .npy headers
    ids = np.arange(n_utts)
    if n_utts * row_bytes > room:
        ids = np.sort(np.random.default_rng(0).choice(n_utts, room // row_bytes, replace=False))
    hyp = np.arange(beam)[None, :] < n[ids, None]
    pos = hyp[:, :, None] & (np.arange(width)[None, None, :] < ln[ids, :, None])
    arrays = {"tokens": np.where(pos, tok[ids], 0), "token_scores": np.where(pos, sc[ids], 0),
              "lengths": np.where(hyp, ln[ids], 0), "mean_scores": np.where(hyp, avg[ids], 0), "nbest": n[ids]}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))
    np.save(os.path.join(out_dir, "utterance_ids.npy"), ids.astype(np.float64))
    return ids


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch.distributed as dist
    from e2e_asr_pytorch_b200 import shard, ops
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, "--gpus %d but WORLD_SIZE=%d (launch with torch.distributed.run)" % (args.gpus, world)
    assert torch.cuda.is_available(), "the B200 arm has no CPU path"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    dec, asr, lm = build_models(dev)
    dec.fast_math = bool(args.fast_math)
    dec.skip_dead_rows = not args.write_dead_rows
    dec.profile_prefix = True
    if args.lm_split:
        dec.lm_split = args.lm_split
    if args.vgg_split:
        dec.vgg_split = args.vgg_split
    if args.prefix_math:
        dec.prefix_math = args.prefix_math
    lengths = workload_lengths(world, args.n_utts)
    n_total = len(lengths)
    shards = shard.plan_shards(lengths, world, MAX_RATIO)
    batches = shard.make_batches(shards[rank], lengths, args.max_utts, args.max_padded_frames)
    cap = int(np.ceil(lengths.max() * MAX_RATIO)) + 1
    rows = max(len(s) for s in shards)
    rsize = shard.ragged_size(shards, lengths, BEAM, MAX_RATIO)

    host = [make_features(b, lengths, pin=True) for b in batches]            # pinned host buffers
    resident = [(f.to(dev), l.to(dev)) for f, l in host]                      # HBM-resident copies
    h2d_bytes = sum(f.numel() * 4 + l.numel() * 8 for f, l in host)
    if args.ragged_h2d:                                                        # only the valid frames are copied
        h2d_bytes = sum(int(l.sum()) * f.shape[2] * 4 + l.numel() * 8 for f, l in host)
    in_bytes = sum(f.numel() * 4 for f, _ in resident)
    # N-best of this rank's shard: packed ON THE DEVICE into the ragged gather buffer, all-gathered where it lies,
    # read back once into pinned host memory (shard.RaggedPacker / gather_nbest)
    packer = shard.RaggedPacker(shards[rank], lengths, BEAM, MAX_RATIO, rsize, dev)
    dec.profile_phases = "coarse"
    phase_ev = []

    def one_pass(from_host):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        ev[0].record()
        packer.reset()
        for b, hb, rb in zip(batches, host, resident):
            if from_host and args.ragged_h2d:
                part = dec.decode_batch_from_host(hb[0], hb[1], dev, return_arrays="device")   # valid frames only cross the bus
            else:
                if from_host:
                    feat, fl = hb[0].to(dev, non_blocking=True), hb[1].to(dev, non_blocking=True)
                else:
                    feat, fl = rb
                part = dec.decode_batch(feat, fl, return_arrays="device")
            ev[1].record()
            packer.pack(b, *part)
        ev[2].record()
        full = shard.gather_nbest(packer.buf, marks=(ev[3], ev[4]))           # the one collective (no-op at N=1) + the read-back
        phase_ev.append(ev)
        return packer.buf, full

    def timed(from_host, steps, warmup):
        for _ in range(warmup):
            one_pass(from_host)
        dec.prefix_events = []
        dec.phase_ms = {}
        del phase_ev[:]
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        l0 = ops.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            local_buf, full = one_pass(from_host)
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        # per-phase device-clock time of a pass (CUDA events at the phase boundaries), max over ranks
        names = ["encode", "ctc_posterior", "steps", "finalize", "pack", "gather", "d2h", "other"]
        ph = dict(dec.phase_ms)
        ph["pack"] = sum(e[1].elapsed_time(e[2]) for e in phase_ev)
        ph["gather"] = sum(e[2].elapsed_time(e[3]) for e in phase_ev)
        ph["d2h"] = sum(e[3].elapsed_time(e[4]) for e in phase_ev)
        ph["other"] = e0.elapsed_time(e1) - sum(ph.get(k, 0.0) for k in names[:-1])      # feature copy, sort / index set-up, host gaps
        vals = torch.tensor([e0.elapsed_time(e1)] + [ph.get(k, 0.0) / steps for k in names], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        clocks = sampler.stop() if rank == 0 else None
        phases = {k: round(float(v), 3) for k, v in zip(names, vals[1:].tolist())}
        return float(vals[0].item()), ops.launch_count() - l0, clocks, local_buf, full, phases

    ms, launches, clocks, local_buf, full, phases = timed(False, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        # unpacked here: the e2e leg below reads back into the same pinned host buffer
        dump_outputs(args.dump_outputs, *shard.unpack_nbest_ragged(full, shards, lengths, BEAM, MAX_RATIO, rsize))
    # prefix-score kernel: per-launch CUDA-event durations collected inside the timed region
    ev = dec.prefix_events
    k_ms = [a.elapsed_time(b) for a, b, _, _ in ev]
    units_formula = float(sum(u for _, _, u, _ in ev))
    units_rows = float(sum(r for _, _, _, r in ev))
    k_total_ms = float(sum(k_ms))
    bytes_per_unit = 12.0 + 12.0 / dec.ctc_beam_size
    peak, peak_src = load_peaks()
    traffic, traffic_src = load_traffic()
    if args.n_utts != N_UTTS:
        traffic, traffic_src = None, None          # the capture is of the full workload
    achieved = units_formula * bytes_per_unit / (k_total_ms * 1e-3) / 1e9 if k_total_ms > 0 else 0.0
    achieved_rows = units_rows * bytes_per_unit / (k_total_ms * 1e-3) / 1e9 if k_total_ms > 0 else 0.0
    dec.profile_prefix = False

    e2e_ms, _, _, _, _, e2e_phases = timed(True, args.steps, 1)
    stats_units = units_formula / max(1, args.steps)

    # ---- result checks, outside the timed regions ----------------------------------------------------------------
    try:
        tok, sc, ln, avg, nn = shard.unpack_nbest_ragged(full, shards, lengths, BEAM, MAX_RATIO, rsize)
        ok = True
    except AssertionError:
        ok = False
    parity = golden_parity(tok, sc, ln, avg, nn) if (ok and rank == 0 and args.n_utts == N_UTTS and GOLDEN_APPLIES) else None
    sharded_equal = None
    if world > 1 and ok:
        # N-GPU == 1-GPU: rank 0 decodes the LAST rank's shard itself (same batches) and compares with what the gather
        # delivered for those utterances, bit for bit
        if rank == 0:
            other = world - 1
            o_batches = shard.make_batches(shards[other], lengths, args.max_utts, args.max_padded_frames)
            sharded_equal = True
            for ob in o_batches:
                f, l = make_features(ob, lengths, pin=False)
                t2, s2, l2, a2, n2 = dec.decode_batch(f.to(dev), l.to(dev), return_arrays=True)
                idx = torch.as_tensor(np.asarray(ob, dtype=np.int64))
                w = t2.shape[2]
                same = (torch.equal(tok[idx][:, :, :w], t2) and torch.equal(ln[idx], l2) and torch.equal(nn[idx], n2)
                        and torch.equal(sc[idx][:, :, :w].contiguous().view(torch.int32), s2.contiguous().view(torch.int32))
                        and torch.equal(avg[idx].contiguous().view(torch.int32), a2.contiguous().view(torch.int32)))
                sharded_equal = sharded_equal and bool(same)
        dist.barrier()

    if rank != 0:
        # every rank leaves through the same barrier as rank 0 (a rank that returned early left rank 0 waiting
        # in its last barrier until the NCCL watchdog aborted it)
        dist.barrier()
        dist.destroy_process_group()
        return
    line = {
        "metric": METRIC, "value": n_total * args.steps / (ms * 1e-3), "unit": "utts/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "cfg2: char V=31 VGG+BLSTM CTC-attention (librispeech_asr.yaml dims, vgg=1) + 4x1024 RNNLM, "
                               "beam 8, ctc 0.5, lm 0.5, max_len_ratio 0.2, %d utts/GPU dev-clean-like lengths, random init" % args.n_utts,
                   "utterances": n_total, "batches_per_gpu": len(batches), "max_utts_per_batch": args.max_utts,
                   "prefix_fast_math": bool(args.fast_math), "prefix_math": "mufu" if args.fast_math else dec.prefix_math, "skip_dead_rows": not args.write_dead_rows,
                   "h2d": "pinned host features, valid frames only, one copy per utterance on a copy stream, pipelined under the encoder "
                          "in 128-utterance chunks (BeamDecoder.decode_batch_from_host)" if args.ragged_h2d else "padded [U,Lmax,D] tensor, one copy",
                   "lm_gemm_operands": dec.lm_split, "vgg_gemm_operands": dec.vgg_split,
                   "l2": "inputs (%.1f GB features + GB-scale prefix states per batch) exceed the 126 MB L2; no flush needed" % (in_bytes / 1e9),
                   "parallelism": "utterance shards x%d, one all-gather of the ragged N-best buffer (packed on the device, one pinned read-back)" % world},
        "e2e": {"value": n_total * args.steps / (e2e_ms * 1e-3), "unit": "utts/s",
                "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(full.numel() * 4), "phases_ms": e2e_phases},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": "prefix_score_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "traffic_unit": "bytes per launch", "traffic_source": traffic_src,
                     "algorithmic_bytes_per_launch": units_formula * bytes_per_unit / max(1, len(ev)),
                     "peak_source": peak_src,
                     "bytes_per_cand_frame": bytes_per_unit, "cand_frames_per_step": stats_units,
                     "kernel_ms_per_step": k_total_ms / max(1, args.steps), "launches_per_step": len(ev) / max(1, args.steps),
                     "kernel_share_of_step": k_total_ms / ms,
                     "achieved_computed_rows_only": achieved_rows, "frac_computed_rows_only": achieved_rows / peak,
                     "cand_frames_per_s": units_formula / (k_total_ms * 1e-3) if k_total_ms > 0 else 0.0},
        "phases_ms": phases,
        "nbest_complete": bool(ok), "nbest_parity": parity, "sharded_equals_single": sharded_equal,
    }
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline(args, sample_utts=args.cpu_sample)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# CPU arm: the UNMODIFIED reference (oracle/_ref: its decode path byte-compiled by oracle/ref_stage.py; imported from
# /root/reference where that exists), driven the way bin/test_asr.py drives it — a deep copy of the BeamDecoder inside
# functools.partial(beam_decode, ...), utterances fanned out with joblib.Parallel (bin/test_asr.py:108-109,138-139).
# ------------------------------------------------------------------------------------------------
def cpu_model_name():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def stratified_sample(lengths, n):
    """Utterance ids at the quantile midpoints (k + 0.5) / n of the sorted lengths of the set (BASELINE.md §3)."""
    order = np.argsort(np.asarray(lengths), kind="stable")
    pos = np.minimum(((np.arange(n) + 0.5) / n * len(order)).astype(np.int64), len(order) - 1)
    return [int(order[p]) for p in pos]


def cand_frames(n_frames):
    steps = int(np.ceil(n_frames * MAX_RATIO))
    return (1 + (steps - 1) * BEAM) * int(1.5 * BEAM) * (n_frames // 4) if steps > 0 else 0


class ReferenceCpu:
    """The reference's BeamDecoder on the host, with the bench's weights and decode settings."""

    def __init__(self):
        import copy
        import tempfile
        import yaml
        from functools import partial
        from oracle import refload
        from e2e_asr_pytorch_b200 import synth
        self.refload = refload
        ref = refload.load()
        self.kind = ref.kind
        test_asr = refload.load_test_asr()
        rasr = ref.ASR(synth.FEAT_DIM, VOCAB, True, **copy.deepcopy(synth.ASR_MODEL_CFG)).eval()
        rasr.load_state_dict(synth.build_asr(VOCAB, seed=0).state_dict())          # same weights as the B200 arm
        tmp = tempfile.mkdtemp(prefix="e2e_ref_")
        torch.save({"model": synth.build_lm(VOCAB, seed=1).state_dict()}, os.path.join(tmp, "lm.pth"))
        yaml.safe_dump({"model": synth.LM_MODEL_CFG}, open(os.path.join(tmp, "lm.yaml"), "w"))
        dec = ref.BeamDecoder(rasr, None, BEAM, MIN_RATIO, MAX_RATIO, lm_path=os.path.join(tmp, "lm.pth"),
                              lm_config=os.path.join(tmp, "lm.yaml"), lm_weight=LM_W, ctc_weight=CTC_W)
        self.func = partial(test_asr.beam_decode, model=copy.deepcopy(dec), device="cpu")   # bin/test_asr.py:108-109

    @staticmethod
    def data(uid, n):
        from e2e_asr_pytorch_b200 import synth
        return (["utt%d" % uid], synth.utterance(uid, n)[None], torch.LongTensor([n]), torch.zeros(1, 1, dtype=torch.long))

    def run(self, jobs, n_jobs, threads):
        """jobs: [(utterance id, frames)], decoded longest first.  ``threads``: torch intra-op threads per worker
        (None = the library default, as shipped).  Returns (wall seconds, results)."""
        from joblib import Parallel, delayed
        jobs = sorted(jobs, key=lambda j: -j[1])
        t0 = time.time()
        res = Parallel(n_jobs=n_jobs, initializer=self.refload.worker_init, initargs=(None, threads))(
            delayed(self.func)(self.data(u, n)) for u, n in jobs)
        return time.time() - t0, res


def _port_worker(job):
    uid, n = job
    import torch as th
    th.set_num_threads(1)
    from oracle import beam_oracle as BO
    from e2e_asr_pytorch_b200 import synth
    global _PORT_MODELS
    try:
        asr, lm = _PORT_MODELS
    except NameError:
        asr, lm = synth.build_asr(VOCAB, seed=0), synth.build_lm(VOCAB, seed=1)
        _PORT_MODELS = (asr, lm)
    with th.no_grad():
        nb = BO.decode_utterance(asr, synth.utterance(uid, n)[None], th.LongTensor([n]), BEAM, MIN_RATIO, MAX_RATIO, lm=lm,
                                 lm_weight=LM_W, ctc_weight=CTC_W)
    return ("utt%d" % uid, [b.ids for b in nb], [])


class PortCpu:
    """Fallback when oracle/_ref did not reach this machine: the oracle PORT of the reference (oracle/beam_oracle.py with the
    product's model.py modules), one utterance per forked worker process.  ``kind`` = "port" in the JSON line."""
    kind = "port"

    def run(self, jobs, n_jobs, threads):
        import multiprocessing as mp
        jobs = sorted(jobs, key=lambda j: -j[1])
        with mp.get_context("fork").Pool(n_jobs) as pool:
            t0 = time.time()
            res = pool.map(_port_worker, jobs, chunksize=1)
            return time.time() - t0, res


def cpu_arm():
    """The unmodified reference if it can be imported here (oracle/_ref or /root/reference), else the oracle port."""
    try:
        return ReferenceCpu()
    except Exception as e:
        sys.stderr.write("bench.py: the staged reference is not importable (%s); timing the oracle port instead\n" % (e,))
        return PortCpu()


def cpu_prefix_only(kind, frames=640, budget_s=3.0):
    """Kernel-level figure of the CPU arm (SURVEY §8d "cheap_compute-only timing"): the reference's numpy
    ``CTCPrefixScore.cheap_compute`` (src/ctc.py:68-108) alone, one core, a chain of calls on a median-length utterance
    with the bench's C = 12 candidates — the unit (candidate-frames per second) of ``roofline.cand_frames_per_s``."""
    if kind == "port":
        from oracle.ctc_prefix_oracle import PrefixScorerOracle as CTCPrefixScore
    else:
        from oracle import refload
        CTCPrefixScore = refload.load().CTCPrefixScore
    T, C = frames // 4, int(1.5 * BEAM)
    g = torch.Generator().manual_seed(7)
    x = torch.log_softmax(torch.randn(1, T, VOCAB, generator=g), -1)
    sc = CTCPrefixScore(x)
    rng = np.random.default_rng(7)
    calls, t0 = 0, time.time()
    while time.time() - t0 < budget_s:                                            # one decode after the other until the budget is spent
        r, prefix = sc.init_state(), []
        while time.time() - t0 < budget_s and len(prefix) < T // 5:               # max_len_ratio 0.2 of L = 4 T
            cands = [int(c) for c in rng.permutation(VOCAB - 1)[:C] + 1]
            for _ in range(BEAM):                                                 # the beam's hypotheses share the step
                psi, r_new = sc.cheap_compute(prefix, r, cands)
                calls += 1
            prefix, r = prefix + [cands[0]], r_new[0]
    wall = time.time() - t0
    return {"cand_frames_per_s": calls * C * T / wall, "cores": 1,
            "sample": "%d cheap_compute calls (T = %d frames, C = %d, prefixes of 0..%d tokens) in %.1f s" % (calls, T, C, T // 5 - 1, wall)}


def cpu_baseline(args, sample_utts=None):
    """Bounded CPU figure printed beside the B200 line: one median-length utterance per core."""
    cores = len(os.sched_getaffinity(0))
    procs = max(1, min(cores, args.cpu_procs or cores))
    n_jobs = sample_utts or procs
    ref = cpu_arm()
    frames = args.cpu_frames or 640
    jobs = [(100000 + k, frames) for k in range(n_jobs)]
    ref.run([(200000 + k, 80) for k in range(procs)], procs, 1)                   # spawns the workers, imports, first touch
    wall, _ = ref.run(jobs, procs, 1)
    return {"value": n_jobs / wall, "unit": "utts/s", "cores": procs, "kind": "reference" if ref.kind != "port" else "port", "cpu": cpu_model_name(),
            "sample": "%d synthetic utts of %d input frames (%.1f s audio%s) each; the unmodified reference BeamDecoder (%s) through "
                      "bin/test_asr.py::beam_decode and joblib.Parallel(n_jobs=%d), 1 torch thread per worker, %.1f s wall; the CPU cost "
                      "grows ~L^2, so the median length flatters the CPU by ~1.8x against the workload's mean cost — "
                      "`bench.py --impl reference` decodes a length-stratified sample of the set itself"
                      % (n_jobs, frames, frames / 100.0, MEDIAN_NOTE if frames == 640 else "",
                         {"staged": "oracle/_ref", "live": "/root/reference", "port": "NOT AVAILABLE HERE: oracle port, oracle/beam_oracle.py"}[ref.kind], procs, wall),
            "cand_frames_per_s": sum(cand_frames(n) for _, n in jobs) / wall,
            "prefix_only": cpu_prefix_only(ref.kind)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0))
    procs = max(1, min(cores, args.cpu_procs or cores))
    lengths = workload_lengths(1, N_UTTS)                                         # the cfg2 set of one GPU
    per_step = max(1, (args.cpu_sample or 64) // max(1, args.steps))
    if args.cpu_frames:                                                           # smoke runs: utterances of one given length
        jobs = [(100000 + k, args.cpu_frames) for k in range(per_step * args.steps)]
    else:
        jobs = [(i, int(lengths[i])) for i in stratified_sample(lengths, per_step * args.steps)]
    ref = cpu_arm()
    for _ in range(max(1, args.warmup)):                                          # workers up, modules imported, caches warm
        ref.run([(200000 + k, 80) for k in range(procs)], procs, 1)
    # best effort: one worker per core, one torch thread each; the K steps' samples are ONE joblib.Parallel region
    # (the reference iterates a whole data set the same way), so no core idles at a step boundary
    wall, res = ref.run(jobs, procs, 1)
    assert len(res) == len(jobs) and all(len(r[1]) > 0 for r in res)
    value = len(jobs) / wall
    units = sum(cand_frames(n) for _, n in jobs)
    lens = sorted(n for _, n in jobs)
    what = "synthetic utterances of one fixed length" if args.cpu_frames else \
        "utterances of the cfg2 set at the quantile midpoints of its length distribution"
    sample = ("%d %s (%d..%d input frames, mean %d; same ids, features and weights as the B200 arm), %d per step, decoded by the "
              "unmodified reference (%s: src/decode.py BeamDecoder + src/ctc.py CTCPrefixScore) through bin/test_asr.py::beam_decode "
              "and joblib.Parallel(n_jobs=%d), 1 torch thread per worker, longest first"
              % (len(jobs), what, lens[0], lens[-1], int(np.mean(lens)), per_step,
                 {"staged": "oracle/_ref", "live": "/root/reference", "port": "NOT AVAILABLE HERE: oracle port, oracle/beam_oracle.py"}[ref.kind], procs))
    shipped = None
    if not args.no_as_shipped and ref.kind != "port":
        # as shipped (script/test.sh:15): --njobs 4, torch threads left at the library default; on a smaller stratified sample
        if args.cpu_frames:
            sjobs = [(300000 + k, args.cpu_frames) for k in range(args.as_shipped_sample)]
        else:
            sjobs = [(i, int(lengths[i])) for i in stratified_sample(lengths, args.as_shipped_sample)]
        env_threads = os.environ.pop("OMP_NUM_THREADS", None)                     # torchrun exports OMP_NUM_THREADS=1
        try:
            swall, sres = ref.run(sjobs, 4, None)
        finally:
            if env_threads is not None:
                os.environ["OMP_NUM_THREADS"] = env_threads
        shipped = {"value": len(sjobs) / swall, "unit": "utts/s", "n_jobs": 4, "torch_threads": "library default",
                   "sample": "%d utterances at the quantile midpoints of the same set (%d..%d frames), %.1f s wall"
                             % (len(sjobs), min(n for _, n in sjobs), max(n for _, n in sjobs), swall)}
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "utts/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "cfg2: char V=31 VGG+BLSTM CTC-attention (librispeech_asr.yaml dims, vgg=1) + 4x1024 RNNLM, "
                               "beam 8, ctc 0.5, lm 0.5, max_len_ratio 0.2, dev-clean-like lengths, random init; bounded sample: " + sample},
        "cpu_baseline": {"value": value, "unit": "utts/s", "cores": procs, "kind": "reference" if ref.kind != "port" else "port", "cpu": cpu_model_name(),
                         "sample": sample, "cand_frames_per_s": units / wall, "wall_s": wall, "as_shipped": shipped,
                         "prefix_only": cpu_prefix_only(ref.kind)},
        "e2e": {"value": value, "unit": "utts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n-utts", type=int, default=N_UTTS, help="utterances per GPU (profiling runs only; the metric is quoted on 2620)")
    ap.add_argument("--max-utts", type=int, default=4096)
    ap.add_argument("--max-padded-frames", type=int, default=0)
    ap.add_argument("--fast-math", type=int, default=0)
    ap.add_argument("--write-dead-rows", action="store_true")
    ap.add_argument("--lm-split", default="", choices=["", "bf16x3", "fp16x2"],
                    help="operand format of the RNNLM's recurrent GEMMs (default: the decoder's, bf16x3)")
    ap.add_argument("--vgg-split", default="", choices=["", "bf16x3", "fp16x2"],
                    help="operand format of the VGG convolution GEMMs (default: the decoder's, bf16x3)")
    ap.add_argument("--prefix-math", default="", choices=["", "lut", "poly", "poly_estrin"],
                    help="log-add-exp evaluator of the prefix-score kernel (default: the decoder's, lut)")
    ap.add_argument("--ragged-h2d", action="store_true", help="(default now; kept for old command lines)")
    ap.add_argument("--padded-h2d", action="store_true",
                    help="e2e leg: copy the zero-padded [U,Lmax,D] tensor in one piece before decode_batch instead of the valid frames "
                         "only, pipelined under the encoder (BeamDecoder.decode_batch_from_host, the default)")
    ap.add_argument("--ragged-gather", action="store_true", help="(default now; kept for old command lines)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-procs", type=int, default=0)
    ap.add_argument("--cpu-sample", type=int, default=0)
    ap.add_argument("--cpu-frames", type=int, default=0, help="length of the CPU sample's utterances (default: 640 = the workload's median for the "
                    "cpu_baseline leg; the reference arm decodes a length-stratified sample of the set unless a length is given)")
    ap.add_argument("--no-as-shipped", action="store_true", help="reference arm: skip the as-shipped (--njobs 4) measurement")
    ap.add_argument("--as-shipped-sample", type=int, default=8, help="reference arm: utterances of the as-shipped measurement")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="B200 arm: write the N-best of the last timed pass to DIR/<name>.npy (float arrays, at most 64 MB; "
                         "a fixed seeded sample of the utterances when the whole set is larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the B200 arm's outputs")
    args.ragged_h2d = not args.padded_h2d
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
