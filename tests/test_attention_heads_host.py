"""Multi-head attention (attention.num_head > 1) without a device: the batched stepper against the modules called one
hypothesis at a time, the CPU checker of e2e_attention_loc_heads against model.Attention, the memory estimate, and
the argument validation and shape query of the new entry points."""
import copy
import ctypes

import pytest
import torch


@pytest.mark.parametrize("heads", [2, 4])
@pytest.mark.parametrize("mode,v_proj", [("loc", False), ("loc", True), ("dot", False), ("dot", True)])
def test_batched_stepper_multi_head_matches_per_hypothesis_modules(heads, mode, v_proj):
    """Two steps with a reorder over three utterances of different lengths: every head of a hypothesis must attend its
    own utterance's values (model.Attention at batch 1), which a batched value.repeat(num_head, 1, 1) would not do."""
    from e2e_asr_pytorch_b200 import synth
    from e2e_asr_pytorch_b200.stepper import BatchedStepper
    cfg = copy.deepcopy(synth.TINY_ASR_CFG)
    cfg["attention"].update({"mode": mode, "v_proj": v_proj, "num_head": heads})
    asr = synth.build_asr(31, cfg, seed=0, peak=4.0)
    lm = synth.build_lm(31, synth.TINY_LM_CFG, seed=1)
    lens, beam = [64, 120, 92], 3
    feat, fl = synth.padded_batch([3, 4, 5], lens)
    with torch.no_grad():
        st = BatchedStepper(asr, lm, fused_attention=True)          # on the CPU the fused kernel is never chosen
        enc, enc_len = st.encode(feat, fl)
        st.start(enc, enc_len, beam)
        assert not st.fused_step
        if mode == "loc":
            assert st.prev_att.shape == (len(lens) * beam, heads, enc.shape[1])
        a1, l1 = st.step(torch.zeros(len(lens) * beam, dtype=torch.long))
        st.reorder((torch.arange(len(lens))[:, None] * beam).expand(len(lens), beam).contiguous())     # every child from slot 0
        toks = [5, 7, 9]
        a2, l2 = st.step(torch.tensor(toks * len(lens)))
        for u, n in enumerate(lens):
            e, el = asr.encoder(feat[u:u + 1, :n], fl[u:u + 1])
            asr.attention.reset_mem()
            asr.set_state(asr.decoder.init_state(1), None)
            _, ctx = asr.attention(asr.decoder.get_query(), e, el)
            lg, _ = asr.decoder(torch.cat([asr.pre_embed(torch.LongTensor([0])), ctx], -1))
            assert torch.allclose(lg[0], a1[u * beam], atol=2e-6)
            dstate, pa = asr.decoder.get_state(), getattr(asr.attention.att_layer, "prev_att", None)
            for b, tk in enumerate(toks):
                asr.set_state(dstate, pa)
                _, ctx2 = asr.attention(asr.decoder.get_query(), e, el)
                lg2, _ = asr.decoder(torch.cat([asr.pre_embed(torch.LongTensor([tk])), ctx2], -1))
                assert torch.allclose(lg2[0], a2[u * beam + b], atol=3e-6)


@pytest.mark.parametrize("v_proj", [False, True])
def test_heads_oracle_matches_model_attention(v_proj):
    """The checker of e2e_attention_loc_heads against model.Attention (H = 3) at batch 1, over two steps."""
    from e2e_asr_pytorch_b200.model import Attention
    from tests._attention_heads_oracle import loc_attention_full_heads
    torch.manual_seed(0)
    h, a, e_dim, q_dim, t = 3, 8, 12, 10, 23
    att = Attention(e_dim, q_dim, "loc", a, h, 0.5, v_proj, 4, 5).eval()
    enc = torch.randn(1, t, e_dim)
    enc_len = torch.tensor([19])
    lay = att.att_layer
    with torch.no_grad():
        key = torch.tanh(att.proj_k(enc)).view(1, t, h, a).permute(0, 2, 1, 3)
        value = torch.tanh(att.proj_v(enc)) if v_proj else enc
        prev = torch.zeros(1, h, t)
        prev[:, :, :19] = 1.0 / 19
        for step in range(2):
            dec = torch.randn(1, q_dim)
            want_attn, want_ctx = att(dec, enc, enc_len)
            query = torch.tanh(att.proj_q(dec))
            attn, ctx = loc_attention_full_heads(key, value, query, prev, enc_len, lay.loc_conv.weight, lay.loc_proj.weight,
                                                 lay.gen_energy.weight.reshape(-1), float(lay.gen_energy.bias), 0.5, 1, v_proj)
            assert (attn - want_attn).abs().max() < 1e-6
            assert (att.merge_head(ctx) - want_ctx).abs().max() < 1e-6
            assert (attn[:, :, 19:] == 0).all()
            prev = attn


def test_decode_estimate_grows_with_heads_and_value_projection():
    from e2e_asr_pytorch_b200 import shard
    args = (2620, 3312, 31, 8, 12)
    base = shard.estimate_decode_bytes(*args)
    assert shard.estimate_decode_bytes(*args, num_head=1, v_proj=False) == base
    h2, h4 = (shard.estimate_decode_bytes(*args, num_head=h) for h in (2, 4))
    assert base < h2 < h4
    assert shard.estimate_decode_bytes(*args, num_head=4, v_proj=True) - h4 > 20e9         # [U][T][4*640] fp32 values
    assert shard.estimate_decode_bytes(*args, v_proj=True) > base


def test_heads_entry_points_validate_arguments_without_a_device():
    from e2e_asr_pytorch_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(256)                       # non-null, aligned, never dereferenced
    ptrs = [fake] * 8
    # key_t .. w_energy, b_e, temp, n_run, B, H, T, A, K, W, E, per_head_values, hyps_per_unit, attn, ctx, stream
    ok = dict(n_run=2, B=4, H=2, T=40, A=24, K=4, W=21, E=16, pv=0, hpu=0)

    def call(ptr_list=ptrs, out=(fake, fake), **kw):
        v = dict(ok, **kw)
        return lib.e2e_attention_loc_heads(*ptr_list, 0.0, 0.5, v["n_run"], v["B"], v["H"], v["T"], v["A"], v["K"], v["W"], v["E"],
                                           v["pv"], v["hpu"], out[0], out[1], None)
    assert call(ptr_list=[None] + ptrs[1:]) == -1 and b"null pointer" in lib.e2e_last_error()
    assert call(out=(fake, None)) == -1
    for bad in (dict(n_run=0), dict(B=0), dict(H=0), dict(T=0), dict(A=-4), dict(K=0), dict(W=0), dict(E=0)):
        assert call(**bad) == -1 and b"bad size" in lib.e2e_last_error(), bad
    assert call(pv=2) == -1
    assert call(hpu=3) == -1
    for unsupported in (dict(H=5), dict(K=13), dict(A=26), dict(W=20), dict(B=33)):
        assert call(**unsupported) == -3 and b"unsupported shape" in lib.e2e_last_error(), unsupported
    assert call(out=(ctypes.c_void_p(260), fake)) == -1 and b"16-byte aligned" in lib.e2e_last_error()


def test_heads_shape_query_covers_every_beam_up_to_four_heads():
    """Full-size attention (A = 300, W = 201) with up to 12 filters: every beam 1..32 and every H <= 4 launches; the
    query refuses what the kernel cannot take."""
    from e2e_asr_pytorch_b200 import ops
    for h in range(1, 5):
        for k in (1, 4, 10, 12):
            assert all(ops.attention_loc_heads_supported(b, h, 300, k, 201) for b in range(1, 33)), (h, k)
    assert not ops.attention_loc_heads_supported(8, 5, 300, 10, 201)
    assert not ops.attention_loc_heads_supported(8, 2, 300, 13, 201)
    assert not ops.attention_loc_heads_supported(8, 2, 302, 10, 201)
    assert not ops.attention_loc_heads_supported(8, 2, 300, 10, 200)
    assert not ops.attention_loc_heads_supported(33, 2, 300, 10, 201)
    assert not ops.attention_loc_heads_supported(8, 4, 300, 10, 4001)              # the filters alone exceed shared memory
    assert not ops.attention_loc_heads_supported(0, 2, 300, 10, 201)
