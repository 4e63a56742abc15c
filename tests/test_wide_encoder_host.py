"""Encoder recurrent layers wider than 384 units, host side (no GPU): which layers take the packed path, the argument
checks of the cluster-form entry points e2e_lstm_sequence_wide / e2e_gru_sequence_wide, the decode memory estimate of
a wide encoder, and that the narrow recurrence kernels keep their SASS now that the cluster form shares their
translation unit."""
import ctypes
import hashlib
import itertools
import json
import os
import shutil

import pytest
import torch

from tests.test_emb_fusion_host import _nvcc_release, _sass_functions

HERE = os.path.dirname(os.path.abspath(__file__))


def _layer(h, module="LSTM", bidirection=True, rate=1, style="drop", layer_norm=False):
    from e2e_asr_pytorch_b200.model import RecurrentLayer
    return RecurrentLayer(8, module, h, bidirection, 0.0, layer_norm, rate, style, False).eval()


def test_packed_supported_takes_multiples_of_128_up_to_1024():
    """512 .. 1024 in steps of 128 take the packed path for LSTM and GRU, one or two directions, with and without
    sub-sampling and LayerNorm; sizes above 384 that are no multiple of 128, or above 1024, do not."""
    for h, module, bidir, (rate, style), ln in itertools.product([512, 640, 768, 896, 1024], ["LSTM", "GRU"], [True, False],
                                                                [(1, "drop"), (2, "drop"), (2, "concat")], [False, True]):
        assert _layer(h, module, bidir, rate, style, ln).packed_supported(), (h, module, bidir, rate, style, ln)
    for h, module in itertools.product([385, 400, 520, 1152], ["LSTM", "GRU"]):
        assert not _layer(h, module).packed_supported(), (h, module)
    from e2e_asr_pytorch_b200 import ops
    assert [h for h in range(1, 1300) if ops.sequence_supported(h) and h > 384] == [512, 640, 768, 896, 1024]


def test_wide_configs_encode_on_the_packed_path():
    from e2e_asr_pytorch_b200 import synth
    for cfg in (synth.WIDE_ASR_CFG, synth.TINY_WIDE_ASR_CFG):
        asr = synth.build_asr(31, cfg)
        assert asr.encoder.packed_supported()
        assert [l.layer.hidden_size for l in asr.encoder.layers[1:]] == cfg["encoder"]["dim"]
        assert cfg["decoder"]["dim"] == 512
    assert synth.WIDE_ASR_CFG["encoder"]["dim"] == [512] * 4 and synth.ASR_MODEL_CFG["encoder"]["dim"] == [320] * 4


@pytest.mark.parametrize("fn,n_gates", [("e2e_lstm_sequence_wide", 4), ("e2e_gru_sequence_wide", 3)])
def test_wide_entry_points_reject_bad_arguments_without_a_device(fn, n_gates):
    from e2e_asr_pytorch_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(256)                      # a non-null, aligned "device pointer" that is never dereferenced
    # (gates, pitch, out, out_pitch, frame_off, lens, g_first, g_rows, N, H, n_groups, n_dirs, fw..., bw..., stream)
    names = (("gates", fake), ("pitch", None), ("out", fake), ("out_pitch", None), ("frame_off", fake), ("lens", fake),
             ("g_first", fake), ("g_rows", fake), ("N", 3), ("H", 512), ("n_groups", 1), ("dirs", 2),
             ("b_fw", fake), ("w_fw", fake), ("goff_fw", 0), ("ooff_fw", 0),
             ("b_bw", fake), ("w_bw", fake), ("goff_bw", None), ("ooff_bw", None), ("stream", None))

    def call(**k):
        h = k.get("H", 512)
        dflt = {"pitch": 2 * n_gates * h, "out_pitch": 2 * h, "goff_bw": n_gates * h, "ooff_bw": h}
        return getattr(lib, fn)(*[k.get(n, dflt.get(n, d)) for n, d in names])

    def refused(code, what, **k):
        assert call(**k) == code, k
        msg = lib.e2e_last_error()
        assert fn.encode() in msg and what in msg, (k, msg)

    for ptr in ("gates", "out", "frame_off", "lens", "g_first", "g_rows", "w_fw"):
        refused(-1, b"null pointer", **{ptr: None})
    refused(-1, b"null pointer", w_bw=None)                                # two directions need the backward weights
    refused(-1, b"bad size", pitch=n_gates * 512 - 1, dirs=1)              # pitch < n_gates * H
    refused(-1, b"bad size", out_pitch=511)
    for dirs in (0, 3):
        refused(-1, b"bad size", dirs=dirs)
    refused(-1, b"bad size", N=0)
    refused(-1, b"bad size", n_groups=0)
    for h in (400, 520, 1000):                                             # H % 128 != 0
        refused(-3, b"hidden size %d" % h, H=h)
    refused(-3, b"hidden size 1152", H=1152)                               # H > 1024
    # the narrow entry points still refuse what only the wide ones take
    narrow = getattr(lib, fn.replace("_wide", ""))
    assert narrow(*[dict(names).get(n) if n not in ("pitch", "out_pitch", "goff_bw", "ooff_bw") else
                    {"pitch": 2 * n_gates * 512, "out_pitch": 1024, "goff_bw": n_gates * 512, "ooff_bw": 512}[n]
                    for n, _ in names]) == -3
    assert b"hidden size 512 > 384" in lib.e2e_last_error()


def test_wide_wrappers_have_no_cpu_path():
    from e2e_asr_pytorch_b200 import ops, _lib
    h = 512
    idx = torch.zeros(2, dtype=torch.int32)
    w = (torch.zeros(4 * h), torch.zeros(h, h, 4), 0, 0)
    with pytest.raises(_lib.E2EError):
        ops.lstm_sequence(torch.zeros(6, 4 * h), torch.zeros(6, h), idx, idx, idx, idx, h, w)
    with pytest.raises(_lib.E2EError):
        ops.gru_sequence(torch.zeros(6, 3 * h), torch.zeros(6, h), idx, idx, idx, idx, h, w)


def _decoder(cfg):
    from e2e_asr_pytorch_b200 import BeamDecoder, synth
    return BeamDecoder(synth.build_asr(31, cfg, seed=0), None, 8, 0.01, 0.2, ctc_weight=0.5)


def test_decode_estimate_grows_with_the_encoder_width_above_640():
    """decode_dataset sizes batches with the encoder's recurrence width when it exceeds the estimate's default 640:
    a 2 x 512 encoder's estimate is larger, by at least its output and gate buffers, and 2 x 320 or narrower encoders
    keep the estimate they had."""
    import copy
    from e2e_asr_pytorch_b200 import results, shard, synth
    args = (2620, 3300)
    default = shard.estimate_decode_bytes(*args, vocab=31, beam=8, n_cand=12, feat_dim=160)
    for cfg in (synth.ASR_MODEL_CFG, synth.TINY_ASR_CFG):
        assert results.decode_bytes_fn(_decoder(cfg), 160)(*args) == default
    assert results.encoder_width(_decoder(synth.ASR_MODEL_CFG).asr.encoder) == 640
    wide = _decoder(synth.WIDE_ASR_CFG)
    assert results.encoder_width(wide.asr.encoder) == 1024
    est = results.decode_bytes_fn(wide, 160)(*args)
    assert est == shard.estimate_decode_bytes(*args, vocab=31, beam=8, n_cand=12, feat_dim=160, enc_dim=1024)
    t = (3300 // 4 + 3) // 4 * 4
    assert est - default >= 2620 * t * (1024 - 640) * 4 * 2                   # the padded output + the packed frames
    sizes = []
    for h in (512, 768, 1024):
        cfg = copy.deepcopy(synth.TINY_ASR_CFG)
        cfg["encoder"]["dim"] = [h, h]
        sizes.append(results.decode_bytes_fn(_decoder(cfg), 160)(*args))
    assert default < sizes[0] < sizes[1] < sizes[2]


def test_nvcc_builds_the_library_for_sm_100a_with_the_wide_kernels():
    """build.py compiles the library with -gencode arch=compute_100a,code=sm_100a, and it holds both cluster kernels."""
    from e2e_asr_pytorch_b200 import _lib, build
    assert "arch=compute_100a,code=sm_100a" in build.NVCC_FLAGS
    lib = _lib.load()
    for name in ("e2e_lstm_sequence_wide", "e2e_gru_sequence_wide"):
        assert hasattr(lib, name)
    release, cuobjdump = _nvcc_release()
    tool = cuobjdump if cuobjdump and os.path.exists(cuobjdump) else shutil.which("cuobjdump")
    if tool is None:
        pytest.skip("no cuobjdump next to nvcc")
    import subprocess
    elf = subprocess.run([tool, "-lelf", build.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in elf
    funcs = _sass_functions(build.LIB_PATH, tool)
    for k in ("lstm_seq_wide_kernel", "gru_seq_wide_kernel"):
        sass = [v for n, v in funcs.items() if k in n]
        assert len(sass) == 1, k
        assert "UCGABAR_ARV" in sass[0] and "UCGABAR_WAIT" in sass[0], k       # the cluster barrier of every step
        assert "LDL" not in sass[0] and "STL" not in sass[0], k               # no spills


def test_narrow_recurrence_kernels_keep_their_sass():
    """lstm_seq_kernel and gru_seq_kernel compile to the same instructions as before the cluster form joined
    csrc/lstm_seq.cu (sha256 of the cuobjdump text, recorded with the compiler release it holds for)."""
    gold = json.load(open(os.path.join(HERE, "golden", "lstm_seq_sass_sha256.json")))
    release, cuobjdump = _nvcc_release()
    if release != gold["nvcc_release"] or not (os.path.exists(cuobjdump) or shutil.which("cuobjdump")):
        pytest.skip("the recorded SASS is of nvcc %s (found %s)" % (gold["nvcc_release"], release))
    from e2e_asr_pytorch_b200 import _lib, build
    _lib.load()
    funcs = _sass_functions(build.LIB_PATH, cuobjdump if os.path.exists(cuobjdump) else shutil.which("cuobjdump"))
    assert len(gold["kernels"]) == 2
    for name, sha in gold["kernels"].items():
        assert name in funcs, name
        assert hashlib.sha256(funcs[name].encode()).hexdigest() == sha, name
