"""Host-side logic on the CPU: drop-in interface surface, batched stepper vs the per-hypothesis
module protocol, utterance sharding and the N-best all-gather (gloo, world_size 2)."""
import os
import socket
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_beam_decoder_constructor_surface(tmp_path):
    import yaml
    from e2e_asr_pytorch_b200 import BeamDecoder, Hypothesis, synth
    asr = synth.build_asr(31, synth.TINY_ASR_CFG)
    lm = synth.build_lm(31, synth.TINY_LM_CFG)
    torch.save({"model": lm.state_dict()}, str(tmp_path / "lm.pth"))
    yaml.safe_dump({"model": synth.TINY_LM_CFG}, open(str(tmp_path / "lm.yaml"), "w"))
    dec = BeamDecoder(asr, None, 8, 0.01, 0.2, lm_path=str(tmp_path / "lm.pth"), lm_config=str(tmp_path / "lm.yaml"),
                      lm_weight=0.5, ctc_weight=0.5)
    assert (dec.beam_size, dec.min_len_ratio, dec.max_len_ratio) == (8, 0.01, 0.2)
    assert dec.apply_ctc and dec.ctc_w == 0.5 and dec.ctc_beam_size == 12        # int(1.5*8), decode.py:34
    assert dec.apply_lm and dec.lm_w == 0.5 and not dec.apply_emb
    msg = dec.create_msg()
    assert msg[0].startswith("Decode spec| Beam size = 8") and len(msg) == 3
    for k, v in lm.state_dict().items():
        assert torch.equal(dec.lm.state_dict()[k], v)
    import copy, pickle
    pickle.loads(pickle.dumps(copy.deepcopy(dec)))                                # bin/test_asr.py:108,138 deep-copies + pickles
    with pytest.raises(AssertionError):                                           # decode.py:32
        asr2 = synth.build_asr(31, dict(synth.TINY_ASR_CFG, ctc_weight=0.0))
        BeamDecoder(asr2, None, 2, 0.01, 0.2, ctc_weight=0.5)
    h = Hypothesis([5, 6, 1], [-1.0, -2.0, -3.0], -2.0)
    assert h.outIndex == [5, 6, 1] and float(h.avgScore()) == -2.0 and len(h.output_scores) == 3


@pytest.mark.parametrize("mode,v_proj,variant", [("loc", False, ""), ("dot", False, ""), ("loc", True, ""),
                                                 ("loc", False, "yaml_encoder"), ("loc", False, "gru"), ("loc", False, "concat_ln")])
def test_batched_stepper_matches_per_hypothesis_modules(mode, v_proj, variant):
    """The batched model step against the modules called one hypothesis at a time, as the reference does (decode.py:105-123,
    144-151): location-aware and scaled-dot attention (config key attention.mode), with and without the value projection."""
    import copy
    from e2e_asr_pytorch_b200 import synth
    from e2e_asr_pytorch_b200.stepper import BatchedStepper
    cfg = copy.deepcopy(synth.TINY_ASR_CFG)
    cfg["attention"]["mode"], cfg["attention"]["v_proj"] = mode, v_proj
    if variant == "yaml_encoder":         # config/librispeech_asr.yaml as written: no VGG, the second layer drops every other frame
        cfg["encoder"].update({"vgg": 0, "sample_rate": [1, 2], "sample_style": "drop"})
    elif variant == "gru":                # GRU encoder layers and a 2-layer GRU speller
        cfg["encoder"]["module"] = "GRU"
        cfg["decoder"].update({"module": "GRU", "layer": 2})
    elif variant == "concat_ln":          # frame concatenation instead of dropping, layer norm on (the reference's projection
        # layer is Linear(rnn_out, rnn_out) and cannot follow a concatenation, module.py:1037-1038,1078-1079: proj off)
        cfg["encoder"].update({"sample_rate": [2, 1], "sample_style": "concat", "layer_norm": [True, True], "proj": [False, False]})
    asr = synth.build_asr(31, cfg, seed=0, peak=4.0)
    lm = synth.build_lm(31, synth.TINY_LM_CFG, seed=1)
    lens, beam = [64, 120, 92], 3
    feat, fl = synth.padded_batch([3, 4, 5], lens)
    with torch.no_grad():
        st = BatchedStepper(asr, lm)
        enc, enc_len = st.encode(feat, fl)
        st.start(enc, enc_len, beam)
        a1, l1 = st.step(torch.zeros(len(lens) * beam, dtype=torch.long))
        st.reorder((torch.arange(len(lens))[:, None] * beam).expand(len(lens), beam).contiguous())     # every child from slot 0
        toks = [5, 7, 9]
        a2, l2 = st.step(torch.tensor(toks * len(lens)))
        for u, n in enumerate(lens):
            e, el = asr.encoder(feat[u:u + 1, :n], fl[u:u + 1])                  # exact batch-1 encode
            assert torch.allclose(e[0], enc[u, :int(el)], atol=2e-6)
            asr.attention.reset_mem()
            asr.set_state(asr.decoder.init_state(1), None)
            _, ctx = asr.attention(asr.decoder.get_query(), e, el)
            lg, _ = asr.decoder(torch.cat([asr.pre_embed(torch.LongTensor([0])), ctx], -1))
            lmo, lmh = lm(torch.LongTensor([[0]]), torch.ones([1]), hidden=None)
            assert torch.allclose(lg[0], a1[u * beam], atol=2e-6) and torch.allclose(lmo[0, 0], l1[u * beam], atol=2e-6)
            dstate, pa = asr.decoder.get_state(), getattr(asr.attention.att_layer, "prev_att", None)
            for b, tk in enumerate(toks):
                asr.set_state(dstate, pa)
                _, ctx2 = asr.attention(asr.decoder.get_query(), e, el)
                lg2, _ = asr.decoder(torch.cat([asr.pre_embed(torch.LongTensor([tk])), ctx2], -1))
                lmo2, _ = lm(torch.LongTensor([[tk]]), torch.ones([1]), hidden=lmh)
                assert torch.allclose(lg2[0], a2[u * beam + b], atol=3e-6)
                assert torch.allclose(lmo2[0, 0], l2[u * beam + b], atol=3e-6)


def test_shard_plan_is_balanced_and_complete():
    from e2e_asr_pytorch_b200 import shard, synth
    lengths = synth.devclean_lengths(2620)
    assert lengths.min() >= 150 and lengths.max() <= 3300 and np.all(lengths % 4 == 0)
    for world in (1, 2, 4, 8):
        parts = shard.plan_shards(lengths, world)
        allidx = np.sort(np.concatenate(parts))
        assert np.array_equal(allidx, np.arange(len(lengths)))
        cost = [shard.utterance_cost(lengths[p]).sum() for p in parts]
        assert max(cost) / (sum(cost) / world) < 1.01
    batches = shard.make_batches(np.arange(100), lengths[:100], max_utts=16)
    assert sorted(sum(batches, [])) == list(range(100)) and all(len(b) <= 16 for b in batches)
    firsts = [lengths[b[0]] for b in batches]
    assert firsts == sorted(firsts, reverse=True)


def _fake_decode(lengths, beam, ratio):
    def fn(batch):
        n = len(batch)
        cap = int(np.ceil(max(lengths[i] for i in batch) * ratio)) + 1
        tok = torch.zeros((n, beam, cap), dtype=torch.int32)
        sc = torch.zeros((n, beam, cap))
        ln = torch.zeros((n, beam), dtype=torch.int32)
        avg = torch.zeros((n, beam))
        for k, i in enumerate(batch):
            m = int(np.ceil(lengths[i] * ratio))
            for b in range(beam):
                tok[k, b, :m] = torch.arange(m, dtype=torch.int32) + 100 * i + b
                sc[k, b, :m] = -0.5 * (b + 1) - 1e-3 * i
                ln[k, b], avg[k, b] = m, -0.5 * (b + 1) - 1e-3 * i
        return tok, sc, ln, avg, torch.full((n,), beam, dtype=torch.int32)
    return fn


def test_pack_unpack_roundtrip_single_rank():
    from e2e_asr_pytorch_b200 import shard
    lengths = np.array([40, 80, 64, 120, 44])
    tok, sc, ln, avg, n = shard.decode_sharded(_fake_decode(lengths, 3, 0.2), lengths, 3, 0.2, max_utts=2)
    want = _fake_decode(lengths, 3, 0.2)(list(range(5)))
    assert torch.equal(tok, want[0]) and torch.equal(sc, want[1]) and torch.equal(ln, want[2])
    assert torch.equal(avg, want[3]) and torch.equal(n, want[4])


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gloo_worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from e2e_asr_pytorch_b200 import shard
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    lengths = np.array([40, 80, 64, 120, 44, 200, 52, 96, 100])
    res = shard.decode_sharded(_fake_decode(lengths, 3, 0.2), lengths, 3, 0.2, rank=rank, world_size=world, max_utts=2)
    torch.save(res, os.path.join(out_dir, "rank%d.pt" % rank))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_decode_allgather_gloo_world2(tmp_path):
    """N>1 path on the CPU: two gloo ranks decode disjoint shards, one all-gather, and every
    rank ends with the single-rank result in utterance order."""
    import torch.multiprocessing as mp
    from e2e_asr_pytorch_b200 import shard
    port = _free_port()
    mp.spawn(_gloo_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    lengths = np.array([40, 80, 64, 120, 44, 200, 52, 96, 100])
    want = shard.decode_sharded(_fake_decode(lengths, 3, 0.2), lengths, 3, 0.2)
    for r in range(2):
        got = torch.load(str(tmp_path / ("rank%d.pt" % r)))
        for a, b in zip(got, want):
            assert torch.equal(a, b)


def test_recurrent_kernel_grouping_covers_every_utterance_once():
    """Encoder._groups (CTA -> utterance grouping of e2e_lstm_sequence): consecutive, complete, at most 16 rows,
    long utterances in small groups."""
    from e2e_asr_pytorch_b200.model import Encoder
    for lens in ([825, 700, 610, 599, 400, 301, 300, 299] + [180] * 37 + [3, 1], [5], [650] * 9):
        first, rows = Encoder._groups(torch.tensor(lens))
        assert first[0] == 0 and sum(rows) == len(lens)
        assert all(f2 == f1 + r1 for f1, r1, f2 in zip(first, rows, first[1:]))
        assert all(1 <= r <= 16 for r in rows)
        for f, r in zip(first, rows):
            assert r <= (4 if lens[f] >= 600 else (8 if lens[f] >= 300 else 16))


def test_f16x2_split_error_budget_against_float64():
    """stepper.SplitLinearF16 (the opt-in 2-piece fp16 operand format of the RNNLM GEMMs), restated with fp32 matmuls of
    its own pieces: the operands' representation error (2^-22) stays below the fp32 accumulation error of the
    product itself, the weight scale puts the largest weight in [2^13, 2^14), and nothing overflows fp16."""
    import torch
    from e2e_asr_pytorch_b200.stepper import SplitLinearF16, _split2_f16, F16_ACT_SCALE
    g = torch.Generator().manual_seed(0)
    x = torch.tanh(torch.randn(192, 2048, generator=g) * 2)
    x[0, :3] = torch.tensor([1.0, -1.0, 1e-7])
    w = (torch.rand(1024, 2048, generator=g) * 2 - 1) / 32
    lin = SplitLinearF16(w)
    assert 2.0 ** 13 <= float(w.abs().max()) * lin.w_scale < 2.0 ** 14
    assert lin.b0.dtype == torch.float16 and torch.isfinite(lin.b1.float()).all()
    a1, a2 = _split2_f16(x, F16_ACT_SCALE)
    assert torch.isfinite(a1.float()).all() and float(a1.float().abs().max()) <= 2.0 ** 14
    back = (a1.double() + a2.double()) / F16_ACT_SCALE
    assert float((back - x.double()).abs().max()) <= 2.0 ** -22
    want = x.double() @ w.double().t()
    y = (torch.cat([a1, a2], dim=1).float() @ lin.b1.float() + a1.float() @ lin.b0.float()) * lin.out_scale
    exact_acc = (torch.cat([a1, a2], dim=1).double() @ lin.b1.double() + a1.double() @ lin.b0.double()) * lin.out_scale
    e_repr = float((exact_acc - want).abs().max())
    e_split = float((y.double() - want).abs().max())
    e_fp32 = float(((x @ w.t()).double() - want).abs().max())
    assert e_repr < 0.5 * e_fp32, (e_repr, e_fp32)
    assert e_split <= 2.0 * e_fp32 + 1e-7, (e_split, e_fp32)


def test_memory_budget_splits_a_subword_set_and_keeps_the_char_set_whole():
    """shard.estimate_decode_bytes / make_batches(max_bytes=...): BASELINE cfg2 (char vocabulary, 2620 utterances) stays
    ONE batch under a B200's 180 GB (it is measured as one, DESIGN.md §3), cfg3 (10k subword vocabulary: 86 GB of
    posteriors plus as many logits at Tmax = 825) is split, every utterance lands in exactly one batch, and a single
    utterance is never refused."""
    import functools
    from e2e_asr_pytorch_b200 import shard, synth
    lengths = synth.devclean_lengths(2620, seed=2)
    budget = int(0.8 * 178e9)
    char = functools.partial(shard.estimate_decode_bytes, vocab=31, beam=8, n_cand=12)
    sub = functools.partial(shard.estimate_decode_bytes, vocab=10000, beam=8, n_cand=12)
    whole = char(2620, int(lengths.max()))
    assert 20e9 < whole < budget, whole
    assert sub(2620, int(lengths.max())) > 178e9
    one = shard.make_batches(np.arange(2620), lengths, 4096, 0, budget, char)
    assert len(one) == 1 and len(one[0]) == 2620
    parts = shard.make_batches(np.arange(2620), lengths, 4096, 0, budget, sub)
    assert len(parts) >= 2
    assert sorted(i for b in parts for i in b) == list(range(2620))
    for b in parts:
        assert sub(len(b), int(lengths[b].max())) <= budget
        assert all(lengths[b[k]] >= lengths[b[k + 1]] for k in range(len(b) - 1))       # longest first inside a batch
    tiny = shard.make_batches(np.arange(3), lengths[:3], 4096, 0, 1, sub)               # absurd budget: one utterance per batch
    assert [len(b) for b in tiny] == [1, 1, 1]
    assert char(10, 800) < char(11, 800) < char(11, 1600)                                # monotone in both arguments


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm timed next to the B200 one) on a tiny bounded sample: one JSON line with the
    result keys, no GPU needed, rank != 0 exits silently.  It times the unmodified reference where that can be imported
    (oracle/refload.py) and otherwise the oracle port, which it must then name as such."""
    import json, os, subprocess, sys
    from oracle import refload
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
           "--cpu-sample", "2", "--cpu-frames", "40", "--cpu-procs", "2", "--as-shipped-sample", "1"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "utts/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": "utts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["cores"] == 2 and d["gpu_launches"] == 0
    assert "unmodified reference" in d["cpu_baseline"]["sample"] and "quantile" not in d["cpu_baseline"]["sample"]   # fixed-length smoke sample
    if refload.available() or refload.staged_available():
        assert d["cpu_baseline"]["kind"] == "reference"
        assert d["cpu_baseline"]["as_shipped"]["n_jobs"] == 4 and d["cpu_baseline"]["as_shipped"]["value"] > 0
    else:
        # the as-shipped leg runs the reference's own settings, so it needs the reference itself
        assert d["cpu_baseline"]["kind"] == "port" and "oracle port" in d["cpu_baseline"]["sample"]
        assert d["cpu_baseline"]["as_shipped"] is None
    po = d["cpu_baseline"]["prefix_only"]                          # SURVEY §8d: cheap_compute alone, the kernel-level CPU figure
    assert po["cores"] == 1 and 1e4 < po["cand_frames_per_s"] < 1e9 and "cheap_compute" in po["sample"]
    quiet = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=root, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert quiet.returncode == 0 and quiet.stdout.strip() == ""


def test_bench_dump_outputs_zeroes_unread_entries_and_samples_under_the_budget(tmp_path):
    """bench.dump_outputs (--dump-outputs): float arrays only, what a caller reads is written as it is and the rest is 0, and
    over the byte budget a seeded sample of the utterances (the same every time, in id order) keeps the files under it."""
    import bench
    g = torch.Generator().manual_seed(0)
    U, B, W = 50, 3, 7
    tok = torch.randint(2, 31, (U, B, W), generator=g, dtype=torch.int32)
    sc = -torch.rand(U, B, W, generator=g)
    ln = torch.randint(1, W + 1, (U, B), generator=g, dtype=torch.int32)
    avg = -torch.rand(U, B, generator=g)
    n = torch.randint(0, B + 1, (U,), generator=g, dtype=torch.int32)
    names = ["lengths", "mean_scores", "nbest", "token_scores", "tokens", "utterance_ids"]
    assert bench.dump_outputs(str(tmp_path / "all"), tok, sc, ln, avg, n).tolist() == list(range(U))
    assert sorted(os.listdir(str(tmp_path / "all"))) == [k + ".npy" for k in names]
    d = {k: np.load(str(tmp_path / "all" / (k + ".npy"))) for k in names}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert d["tokens"].shape == d["token_scores"].shape == (U, B, W) and d["nbest"].tolist() == n.tolist()
    for u in range(U):
        for k in range(B):
            m = int(ln[u, k]) if k < int(n[u]) else 0
            assert d["tokens"][u, k, :m].tolist() == tok[u, k, :m].tolist() and not d["tokens"][u, k, m:].any()
            assert np.array_equal(d["token_scores"][u, k, :m], sc[u, k, :m].numpy()) and not d["token_scores"][u, k, m:].any()
            assert d["lengths"][u, k] == m and d["mean_scores"][u, k] == (avg[u, k].item() if k < int(n[u]) else 0.0)
    budget = 6 * 1024 + 20 * (4 * (2 * B * W + 2 * B + 1) + 8)
    a = bench.dump_outputs(str(tmp_path / "a"), tok, sc, ln, avg, n, budget=budget)
    b = bench.dump_outputs(str(tmp_path / "b"), tok, sc, ln, avg, n, budget=budget)
    assert len(a) == 20 and a.tolist() == b.tolist() == sorted(set(a.tolist()))
    assert sum(os.path.getsize(str(tmp_path / "a" / f)) for f in os.listdir(str(tmp_path / "a"))) <= budget
    assert np.load(str(tmp_path / "a" / "utterance_ids.npy")).tolist() == a.tolist()
    assert np.array_equal(np.load(str(tmp_path / "a" / "tokens.npy")), d["tokens"][a])


def test_ragged_nbest_buffer_layout_and_size():
    """shard.pack_nbest_ragged / unpack_nbest_ragged: round trip in any decode order, lost utterances and over-long
    hypotheses are detected, and for the bench workload the buffer is > 4x smaller than the rectangular one."""
    from e2e_asr_pytorch_b200 import shard, synth
    lengths = np.array([40, 80, 64, 120, 44, 200, 52])
    beam, ratio = 3, 0.2
    shards = shard.plan_shards(lengths, 2, ratio)
    size = shard.ragged_size(shards, lengths, beam, ratio)
    bufs = []
    for ids in shards:
        order = list(ids[::-1])                                   # decode order != layout order
        out = _fake_decode(lengths, beam, ratio)(order)
        bufs.append(shard.pack_nbest_ragged(order, *out, ids, lengths, beam, ratio, size))
        assert bufs[-1].shape == (size,)
    tok, sc, ln, avg, n = shard.unpack_nbest_ragged(torch.cat(bufs), shards, lengths, beam, ratio, size)
    want = _fake_decode(lengths, beam, ratio)(list(range(len(lengths))))
    for a, b in zip((tok, sc, ln, avg, n), want):
        assert torch.equal(a, b)
    # a shard that did not decode one of its utterances is noticed
    ids = shards[0]
    part = _fake_decode(lengths, beam, ratio)(list(ids[1:]))
    holed = shard.pack_nbest_ragged(list(ids[1:]), *part, ids, lengths, beam, ratio, size)
    with pytest.raises(AssertionError):
        shard.unpack_nbest_ragged(torch.cat([holed, bufs[1]]), shards, lengths, beam, ratio, size)
    # a hypothesis longer than the layout allows is an error, not a truncation
    bad = list(_fake_decode(lengths, beam, ratio)([int(ids[0])]))
    bad[0] = torch.nn.functional.pad(bad[0], (0, 8)); bad[1] = torch.nn.functional.pad(bad[1], (0, 8)); bad[2] = bad[2] + 5
    with pytest.raises(ValueError):
        shard.pack_nbest_ragged([int(ids[0])], *bad, ids, lengths, beam, ratio, size)
    # the bench workload: ragged vs rectangular bytes per rank
    big = synth.devclean_lengths(2620, seed=2)
    one = shard.plan_shards(big, 1, 0.2)
    cap = int(np.ceil(big.max() * 0.2)) + 1
    assert shard.ragged_size(one, big, 8, 0.2) * 4.0 < 2620 * shard.row_width(8, cap) * 4 / 4.0


def test_empty_shard_decodes_to_nothing_without_a_device():
    """decode_batch_from_host on an empty shard returns before any device work (a rank with no utterances)."""
    from e2e_asr_pytorch_b200 import BeamDecoder, synth
    dec = BeamDecoder(synth.build_asr(31, synth.TINY_ASR_CFG, seed=0), None, 4, 0.01, 0.2, ctc_weight=0.5)
    feat, fl = torch.zeros(0, 0, synth.FEAT_DIM), torch.zeros(0, dtype=torch.long)
    assert dec.decode_batch_from_host(feat, fl, "cuda:0") == []
    tok, sc, ln, avg, n = dec.decode_batch_from_host(feat, fl, "cuda:0", return_arrays=True)
    assert tok.shape == (0, 4, 1) and sc.shape == (0, 4, 1) and ln.shape == (0, 4) and avg.shape == (0, 4) and n.shape == (0,)
    assert dec.last_stats["utterances"] == 0 and dec.last_h2d_bytes == 0


def test_shard_pack_unpack_property():
    """Property test (hypothesis) of the multi-GPU host logic: for any lengths, beam, ratio and world size — including more
    ranks than utterances — the shards partition the set, every rank's ragged buffer has the common size, and packing each
    shard in any batch order then unpacking the concatenation returns every utterance's N-best in utterance order."""
    from hypothesis import given, settings, strategies as st
    from e2e_asr_pytorch_b200 import shard

    @settings(max_examples=40, deadline=None)
    @given(st.lists(st.integers(min_value=1, max_value=60), min_size=1, max_size=12), st.integers(1, 4), st.integers(1, 5),
           st.sampled_from([0.07, 0.2, 0.5]), st.integers(0, 1000))
    def check(quarter_lengths, beam, world, ratio, seed):
        lengths = np.array(quarter_lengths) * 4
        shards = shard.plan_shards(lengths, world, ratio)
        assert len(shards) == world
        assert sorted(int(i) for s in shards for i in s) == list(range(len(lengths)))
        size = shard.ragged_size(shards, lengths, beam, ratio)
        rng = np.random.default_rng(seed)
        bufs = []
        for ids in shards:
            order = [int(i) for i in rng.permutation(np.asarray(ids, dtype=np.int64))]
            if order:
                out = _fake_decode(lengths, beam, ratio)(order)
            else:
                out = (torch.zeros((0, beam, 1), dtype=torch.int32), torch.zeros((0, beam, 1)), torch.zeros((0, beam), dtype=torch.int32),
                       torch.zeros((0, beam)), torch.zeros((0,), dtype=torch.int32))
            buf = shard.pack_nbest_ragged(order, *out, ids, lengths, beam, ratio, size)
            assert buf.shape == (size,)
            bufs.append(buf)
        tok, sc, ln, avg, n = shard.unpack_nbest_ragged(torch.cat(bufs), shards, lengths, beam, ratio, size)
        want = _fake_decode(lengths, beam, ratio)(list(range(len(lengths))))
        for a, b in zip((tok, sc, ln, avg, n), want):
            assert torch.equal(a, b)

    check()
