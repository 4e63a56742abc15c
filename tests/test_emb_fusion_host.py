"""Embedding-fusion decoding, host side (no GPU): model.EmbeddingRegularizer against a float64 restatement of the plug-in's
formula for every kind of mixing weight and temperature, its state dict, the CPU stepper's emb_logits, the argument checks
of e2e_emb_fuse_candidates, the BeamDecoder's handling of the plug-in (pickle / deepcopy, what it refuses) and the SASS of
the kernels that share the new kernel's translation unit."""
import copy
import ctypes
import hashlib
import itertools
import json
import os
import pickle
import re
import shutil
import subprocess

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))


def _formula64(emb, dec_state, dec_logit):
    """log((1 - lam) softmax(dec) + lam softmax(relu(temp) * emb_logit) + eps) in float64 from the module's parameters."""
    d = lambda t: t.detach().double()
    x = torch.relu(dec_state.double() @ d(emb.emb_net[0].weight).t() + d(emb.emb_net[0].bias))
    x = x @ d(emb.emb_net[2].weight).t() + d(emb.emb_net[2].bias)
    table = d(emb.emb_table.weight)
    if emb.fuse_normalize:
        x = x / x.norm(dim=-1, keepdim=True).clamp_min(1e-12)
        table = table / table.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    pe = torch.softmax(torch.relu(d(emb.temp)) * (x @ table.t()), dim=-1)
    pd = torch.softmax(dec_logit.double(), dim=-1)
    lam = torch.sigmoid(d(emb.fuse_lambda)) if emb.fuse_learnable else d(emb.fuse_lambda)
    return torch.log((1 - lam) * pd + lam * pe + 1e-8)


@pytest.mark.parametrize("fuse,temperature,normalize",
                         list(itertools.product([0.3, -1, -2], [2.0, -1, -2], [False, True])))
def test_module_matches_the_float64_formula(fuse, temperature, normalize):
    from e2e_asr_pytorch_b200 import synth
    vocab, dec_dim = 31, 20
    emb = synth.build_emb(vocab, dec_dim, 30, fuse=fuse, temperature=temperature, fuse_normalize=normalize, seed=5)
    g = torch.Generator().manual_seed(0)
    dec_state, dec_logit = torch.randn(6, dec_dim, generator=g), 4 * torch.randn(6, vocab, generator=g)
    with torch.no_grad():
        none, got = emb(dec_state, dec_logit, return_loss=False)
    assert none is None and got.dtype == torch.float32 and got.shape == (6, vocab)
    want = _formula64(emb, dec_state, dec_logit)
    err = (got.double() - want).abs().max().item()
    assert err < 1e-5, err
    if temperature == -2:
        assert (emb.temp < 0).any()                      # the ReLU clamps some entries
    if fuse in (-1, -2):
        assert not torch.all(emb.fuse_lambda == 0.5)     # moved away from the init value


def test_parameter_names_shapes_and_state_dict_round_trip():
    from e2e_asr_pytorch_b200 import synth
    from e2e_asr_pytorch_b200.model import EmbeddingRegularizer
    shapes = {k: tuple(v.shape) for k, v in synth.build_emb(31, 20, 30, fuse=-2, temperature=-2).state_dict().items()}
    assert shapes == {"emb_table.weight": (31, 30), "emb_net.0.weight": (25, 20), "emb_net.0.bias": (25,),
                      "emb_net.2.weight": (30, 25), "emb_net.2.bias": (30,), "fuse_lambda": (31,), "temp": (31,)}
    fixed = synth.build_emb(31, 20, 30, fuse=0.4, temperature=3.0)
    assert dict(fixed.named_buffers()).keys() == {"fuse_lambda", "temp"} and not fixed.fuse_learnable
    assert float(fixed.fuse_lambda) == pytest.approx(0.4) and float(fixed.temp) == 3.0
    scalar = synth.build_emb(31, 20, 30, fuse=-1, temperature=-1)
    assert {k for k, _ in scalar.named_parameters()} >= {"fuse_lambda", "temp"} and scalar.fuse_lambda.shape == (1,)
    src = synth.build_emb(31, 20, 30, fuse=-2, temperature=-2, fuse_normalize=True, seed=9)
    dst = EmbeddingRegularizer(31, 20, emb_dim=30, fuse=-2, temperature=-2, fuse_normalize=True)
    dst.load_state_dict(src.state_dict())
    x, y = torch.randn(3, 20), torch.randn(3, 31)
    with torch.no_grad():
        assert torch.equal(dst(x, y)[1], src(x, y)[1])
    off = EmbeddingRegularizer(31, 20, emb_dim=30, fuse=0)
    assert not off.apply_fuse and off(x, y) == (None, None)
    with pytest.raises(NotImplementedError):
        src(x, y, return_loss=True)


def test_cpu_stepper_emb_logits_are_the_modules():
    """Step 0 of the CPU stepper for one utterance: every row's emb_logits are what the plug-in's emb_net and table give
    for the speller's output of the oracle's batch-1 module calls (recorded in its trace)."""
    from e2e_asr_pytorch_b200 import synth
    from e2e_asr_pytorch_b200.stepper import BatchedStepper
    from tests import _emb_fusion_oracle as EO
    asr = synth.build_asr(31, synth.TINY_ASR_CFG, seed=0, peak=4.0)
    for normalize in (False, True):
        emb = synth.build_emb(31, 20, 30, fuse=-2, temperature=-2, fuse_normalize=normalize)
        feat, n = synth.utterance(3, 64)[None], 64
        trace = []
        with torch.no_grad():
            EO.decode_utterance(asr, emb, feat, torch.LongTensor([n]), 2, 0.01, 0.05, trace=trace)
            st = BatchedStepper(asr, None, emb=emb)
            enc, enc_len = st.encode(feat, torch.LongTensor([n]))
            st.start(enc, enc_len, 2)
            att, lm, got = st.step(torch.zeros(2, dtype=torch.long))
        assert lm is None and got.shape == (2, 31)
        want = trace[0]["emb_logits"]
        for row in got:
            assert torch.allclose(row, want[0], rtol=1e-5, atol=1e-5), (row - want[0]).abs().max()
        assert torch.equal(st.emb.scale, torch.relu(emb.temp.detach()))
        assert torch.equal(st.emb.lam, torch.sigmoid(emb.fuse_lambda.detach()))


def test_stepper_without_the_plugin_returns_two_rows():
    from e2e_asr_pytorch_b200 import synth
    from e2e_asr_pytorch_b200.stepper import BatchedStepper
    asr = synth.build_asr(31, synth.TINY_ASR_CFG, seed=0, peak=4.0)
    st = BatchedStepper(asr, None)
    with torch.no_grad():
        enc, enc_len = st.encode(synth.utterance(3, 64)[None], torch.LongTensor([64]))
        st.start(enc, enc_len, 2)
        assert len(st.step(torch.zeros(2, dtype=torch.long))) == 2


def test_entry_point_rejects_bad_arguments_without_a_device():
    from e2e_asr_pytorch_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(256)                      # a non-null, aligned "device pointer" that is never dereferenced
    # e2e_emb_fuse_candidates(dec, ld_dec, emb, ld_emb, U, B, V, C, scale, n_scale, lam, n_lam, eps, n_live,
    #                         logp, ld_out, att_stats, cand, stream)
    names = (("dec", fake), ("ld_dec", 31), ("emb", fake), ("ld_emb", 31), ("U", 2), ("B", 4), ("V", 31), ("C", 6),
             ("scale", fake), ("n_scale", 1), ("lam", fake), ("n_lam", 31), ("eps", 1e-8), ("n_live", fake),
             ("logp", fake), ("ld_out", 31), ("stats", fake), ("cand", fake), ("stream", None))
    call = lambda **k: lib.e2e_emb_fuse_candidates(*[k.get(n, d) for n, d in names])
    for ptr in ("dec", "emb", "scale", "lam", "logp", "stats", "cand"):
        assert call(**{ptr: None}) == -1, ptr
        assert b"null pointer" in lib.e2e_last_error()
    for bad in ({"U": 0}, {"B": 0}, {"V": 0}, {"C": -1}, {"C": 32}, {"ld_dec": 30}, {"ld_emb": 30}, {"ld_out": 30}):
        assert call(**bad) == -1, bad
        assert b"bad size" in lib.e2e_last_error()
    for bad in ({"n_scale": 2}, {"n_lam": 30}, {"n_scale": 0}):
        assert call(**bad) == -1, bad
        assert b"1 or V entries" in lib.e2e_last_error()
    for eps in (0.0, -1e-8, float("inf"), float("nan")):
        assert call(eps=eps) == -1, eps
        assert b"eps" in lib.e2e_last_error()
    wide = dict(V=10000, ld_dec=10000, ld_emb=10000, ld_out=10000, n_lam=10000)
    assert call(C=256, **wide) != 0                  # the streaming selection's lists would not fit in shared memory
    assert b"C too large" in lib.e2e_last_error()


def test_wrapper_has_no_cpu_path():
    from e2e_asr_pytorch_b200 import ops, _lib
    rows, one = torch.zeros(8, 31), torch.ones(1)
    with pytest.raises(_lib.E2EError):
        ops.emb_fuse_candidates(rows, rows, 2, 4, 31, 6, one, one, 1e-8, torch.ones(2, dtype=torch.int32), rows,
                                torch.zeros(8, 2), torch.zeros(8, 6, dtype=torch.int32))


def _decoder(emb, **kw):
    from e2e_asr_pytorch_b200 import BeamDecoder, synth
    asr = synth.build_asr(31, synth.TINY_ASR_CFG, seed=0, peak=4.0)
    return BeamDecoder(asr, emb, 4, 0.01, 0.2, ctc_weight=0.5, **kw)


def test_decoder_keeps_the_plugin_and_survives_pickle_and_deepcopy():
    from e2e_asr_pytorch_b200 import synth
    emb = synth.build_emb(31, 20, 30, fuse=-2, temperature=-2)
    dec = _decoder(emb)
    assert dec.apply_emb and dec.emb_decoder is emb
    assert any("Emb. decoding" in line for line in dec.create_msg())
    for twin in (pickle.loads(pickle.dumps(dec)), copy.deepcopy(dec)):
        assert twin.apply_emb and twin._stepper is None
        x, y = torch.randn(2, 20), torch.randn(2, 31)
        with torch.no_grad():
            assert torch.equal(twin.emb_decoder(x, y)[1], emb(x, y)[1])
    plain = _decoder(None)
    assert not plain.apply_emb and not any("Emb." in line for line in plain.create_msg())


def test_decoder_refuses_what_is_not_fusion():
    from e2e_asr_pytorch_b200 import synth
    from e2e_asr_pytorch_b200.model import EmbeddingRegularizer
    bert = synth.build_emb(31, 20, 30)
    bert.use_bert = True
    with pytest.raises(NotImplementedError):
        _decoder(bert)
    with pytest.raises(ValueError, match="apply_fuse"):
        _decoder(EmbeddingRegularizer(31, 20, emb_dim=30, fuse=0))


def _sass_functions(path, cuobjdump):
    out = subprocess.run([cuobjdump, "-sass", path], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
        elif cur is not None:
            funcs[cur].append(line)
    return {k: "\n".join(v) for k, v in funcs.items()}


def _nvcc_release():
    from e2e_asr_pytorch_b200 import build
    nvcc = build._nvcc()
    if nvcc is None:
        return None, None
    m = re.search(r"release (\d+\.\d+)", subprocess.run([nvcc, "--version"], capture_output=True, text=True).stdout)
    return (m.group(1) if m else None), os.path.join(os.path.dirname(nvcc), "cuobjdump")


def test_beam_step_kernels_keep_their_sass():
    """The fusion kernel shares csrc/beam_step.cu with (3a), (3b), the final selection and the N-best pack: each of
    those compiles to the same instructions as before it joined (sha256 of the cuobjdump text, recorded with the
    compiler release it holds for)."""
    gold = json.load(open(os.path.join(HERE, "golden", "beam_step_sass_sha256.json")))
    release, cuobjdump = _nvcc_release()
    if release != gold["nvcc_release"] or not (os.path.exists(cuobjdump) or shutil.which("cuobjdump")):
        pytest.skip("the recorded SASS is of nvcc %s (found %s)" % (gold["nvcc_release"], release))
    from e2e_asr_pytorch_b200 import _lib, build
    _lib.load()
    funcs = _sass_functions(build.LIB_PATH, cuobjdump if os.path.exists(cuobjdump) else shutil.which("cuobjdump"))
    for name, sha in gold["kernels"].items():
        assert name in funcs, name
        assert hashlib.sha256(funcs[name].encode()).hexdigest() == sha, name
    assert any("emb_fuse_candidates_kernel" in k for k in funcs)
