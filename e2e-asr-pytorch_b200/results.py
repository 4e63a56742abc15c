"""Result files and scoring of the decode flow (SURVEY.md §8f row f-3).

The reference writes two tab-separated files per data split (``bin/test_asr.py:90-104,146-156``)

    *_output.csv :  idx \\t hyp \\t truth                 (1-best)
    *_beam.csv   :  idx \\t beam \\t hyp \\t truth        (every returned hypothesis, best first)

and scores them with ``eval.py`` (mean CER / WER of the 1-best, ``eval.py:14-26``) and
``eval_beam.py`` (per utterance the MINIMUM error over consecutive rows with the same ``idx`` —
an oracle over the N-best, ``eval_beam.py:28-39``).  Both scripts depend on pandas and the
``editdistance`` package; this module restates the file formats and the statistics on numpy
alone so that the B200 decode path can feed the same evaluation flow:

* :func:`decode_dataset`  — what ``Solver.exec`` + ``beam_decode`` do (``bin/test_asr.py:86-173``),
  batched: utterances are grouped by length and decoded with ``BeamDecoder.decode_batch``;
* :func:`write_results`   — ``Solver.write_hyp`` (``bin/test_asr.py:146-156``), same bytes;
* :func:`score_file` / :func:`format_report` — the numbers and the table ``eval.py`` /
  ``eval_beam.py`` print.
"""
import csv

import numpy as np

SEP = ' '   # eval.py:6


# ------------------------------------------------------------------------------------------------
# files
# ------------------------------------------------------------------------------------------------
def init_result_files(best_path, beam_path=None):
    """Headers exactly as bin/test_asr.py:91-92,103-104."""
    with open(best_path, 'w') as f:
        f.write('idx\thyp\ttruth\n')
    if beam_path is not None:
        with open(beam_path, 'w') as f:
            f.write('idx\tbeam\thyp\ttruth\n')


def write_results(results, tokenizer, best_path, beam_path=None):
    """results: iterable of (name, [hyp token ids, best first], truth token ids) — the tuples
    ``beam_decode`` returns (bin/test_asr.py:172-173).  ``tokenizer.decode(ids)`` is any of the reference's
    text encoders (src/text.py).  Appends like the reference (bin/test_asr.py:146-156)."""
    with open(best_path, 'a') as fb:
        fbeam = open(beam_path, 'a') if beam_path is not None else None
        try:
            for name, hyp_seqs, truth in results:
                hyps = [tokenizer.decode(list(h)) for h in hyp_seqs]
                tr = tokenizer.decode(list(truth))
                fb.write('\t'.join([name, hyps[0], tr]) + '\n')
                if fbeam is not None:
                    for b, hyp in enumerate(hyps):
                        fbeam.write('\t'.join([name, str(b), hyp, tr]) + '\n')
        finally:
            if fbeam is not None:
                fbeam.close()


def encoder_width(encoder):
    """The widest recurrence output of an encoder's layers (2H for a bidirectional layer of H units), 0 without any."""
    import torch
    return max([l.hidden_size * (2 if l.bidirectional else 1) for l in encoder.modules()
                if isinstance(l, (torch.nn.LSTM, torch.nn.GRU))] or [0])


def decode_bytes_fn(decoder, feat_dim):
    """``bytes_fn(n_utts, l_max)`` that decode_dataset sizes its batches by: shard.estimate_decode_bytes with the
    decoder's settings.  An encoder wider than the estimate's default 640 (two directions of 320 units) passes its own
    width, which the encoder output and the packed first layer's gates scale with; narrower ones keep the default."""
    import functools
    from . import shard
    enc = decoder.asr.encoder
    width = encoder_width(enc)
    return functools.partial(shard.estimate_decode_bytes, vocab=decoder.asr.vocab_size, beam=decoder.beam_size,
                             n_cand=decoder.ctc_beam_size if decoder.apply_ctc else 0, feat_dim=feat_dim,
                             num_head=decoder.asr.attention.num_head, v_proj=bool(decoder.asr.attention.v_proj),
                             time_reduction=getattr(enc, "sample_rate", 4),
                             front_reduction=4 if getattr(enc, "vgg", 1) else 1,
                             **({"enc_dim": width} if width > 640 else {}))


def decode_dataset(decoder, samples, device, max_utts=4096, max_padded_frames=0, max_bytes=None):
    """samples: sequence of (name, feat [L,D] float tensor, truth ids).  Returns the reference's
    result tuples (name, [hyp.outIndex ...], truth) in the order of ``samples``
    (bin/test_asr.py:138-139,159-173), decoding many utterances per ``decode_batch`` call.
    Batches are closed before their estimated footprint (shard.estimate_decode_bytes) exceeds ``max_bytes``
    (default: 80 % of the device's free memory), which is what splits a subword-vocabulary set."""
    import torch
    from . import shard
    lengths = np.array([int(s[1].shape[0]) for s in samples], dtype=np.int64)
    out = [None] * len(samples)
    if max_bytes is None and torch.device(device).type == "cuda":
        max_bytes = int(0.8 * torch.cuda.mem_get_info(device)[0])
    feat_dim = int(samples[0][1].shape[1]) if len(samples) else 160
    bytes_fn = decode_bytes_fn(decoder, feat_dim)
    for batch in shard.make_batches(np.arange(len(samples)), lengths, max_utts, max_padded_frames, max_bytes, bytes_fn):
        l_max = int(lengths[batch].max())
        feats = torch.zeros(len(batch), l_max, samples[batch[0]][1].shape[1])
        for k, i in enumerate(batch):
            feats[k, :lengths[i]] = samples[i][1]
        nbest = decoder.decode_batch(feats.to(device), torch.as_tensor(lengths[batch]).to(device))
        for k, i in enumerate(batch):
            out[i] = (samples[i][0], [h.outIndex for h in nbest[k]], list(samples[i][2]))
    return out


# ------------------------------------------------------------------------------------------------
# scoring
# ------------------------------------------------------------------------------------------------
def edit_distance(a, b):
    """Levenshtein distance between two sequences (what ``editdistance.eval`` returns)."""
    if len(a) < len(b):
        a, b = b, a
    if len(b) == 0:
        return len(a)
    ids = {}
    bi = np.fromiter((ids.setdefault(x, len(ids)) for x in b), dtype=np.int64, count=len(b))
    prev = np.arange(len(b) + 1, dtype=np.int64)
    offs = np.arange(len(b) + 1, dtype=np.int64)
    for i, x in enumerate(a, 1):
        xi = ids.get(x, -1)
        sub = prev[:-1] + (bi != xi)
        cand = np.minimum(sub, prev[1:] + 1)                    # substitution / deletion
        cur = np.empty_like(prev)
        cur[0] = i
        cur[1:] = cand
        # insertions: cur[j] = min_k<=j (cur[k] + j - k)  ->  prefix minimum of cur[k] - k, plus j
        cur = np.minimum.accumulate(cur - offs) + offs
        prev = cur
    return int(prev[-1])


def read_rows(path):
    """Rows of a result file as dicts; like ``pd.read_csv(sep='\\t', keep_default_na=False)``
    (eval.py:21): empty fields stay empty strings."""
    with open(path, newline='') as f:
        return list(csv.DictReader(f, delimiter='\t'))


def _row_errors(row):
    hyp, truth = row['hyp'], row['truth']
    cer = 100 * float(edit_distance(hyp, truth)) / len(truth)                                   # eval.py:15-16
    wer = 100 * float(edit_distance(hyp.split(SEP), truth.split(SEP))) / len(truth.split(SEP))  # eval.py:17-18
    return cer, wer


def score_file(path, beam=False):
    """Statistics of ``eval.py`` (beam=False) or ``eval_beam.py`` (beam=True) for one result file."""
    rows = read_rows(path)
    if not rows:
        raise ValueError("no rows in " + path)
    cer = np.array([_row_errors(r)[0] for r in rows])
    wer = np.array([_row_errors(r)[1] for r in rows])
    hyp_c = np.array([len(r['hyp']) for r in rows], dtype=np.float64)
    hyp_w = np.array([len(r['hyp'].split(SEP)) for r in rows], dtype=np.float64)
    tr_c = np.array([len(r['truth']) for r in rows], dtype=np.float64)
    tr_w = np.array([len(r['truth'].split(SEP)) for r in rows], dtype=np.float64)
    if beam:
        # eval_beam.py:28-39: minimum over consecutive rows with the same idx; numpy std (ddof=0)
        cers, wers, prev = [], [], ''
        for r, c, w in zip(rows, cer, wer):
            if r['idx'] == prev:
                cers[-1], wers[-1] = min(cers[-1], c), min(wers[-1], w)
            else:
                prev = r['idx']
                cers.append(c)
                wers.append(w)
        cer_u, wer_u, ddof = np.array(cers), np.array(wers), 0
    else:
        cer_u, wer_u, ddof = cer, wer, 1                         # pandas Series.std (eval.py:43): ddof=1
    std = lambda v: float(np.std(v, ddof=ddof)) if len(v) > ddof else float('nan')
    return {
        'file': path, 'rows': len(rows), 'utterances': len(cer_u),
        'truth_chars': float(tr_c.mean()), 'hyp_chars': float(hyp_c.mean()), 'chars_abs_diff': float(np.abs(tr_c - hyp_c).mean()),
        'truth_words': float(tr_w.mean()), 'hyp_words': float(hyp_w.mean()), 'words_abs_diff': float(np.abs(tr_w - hyp_w).mean()),
        'cer_mean': float(cer_u.mean()), 'cer_std': std(cer_u), 'cer_min': float(cer_u.min()), 'cer_max': float(cer_u.max()),
        'wer_mean': float(wer_u.mean()), 'wer_std': std(wer_u), 'wer_min': float(wer_u.min()), 'wer_max': float(wer_u.max()),
    }


def format_report(s):
    """The table eval.py:30-49 / eval_beam.py:44-63 print, from :func:`score_file`'s dict."""
    lines = [
        '',
        '============  Result of {} ============'.format(s['file']),
        ' -----------------------------------------------------------------------',
        '| Statics\t\t|  Truth\t|  Prediction\t| Abs. Diff.\t|',
        ' -----------------------------------------------------------------------',
        '| Avg. # of chars\t|  {:.2f}\t|  {:.2f}\t|  {:.2f}\t\t|'.format(s['truth_chars'], s['hyp_chars'], s['chars_abs_diff']),
        '| Avg. # of words\t|  {:.2f}\t|  {:.2f}\t|  {:.2f}\t\t|'.format(s['truth_words'], s['hyp_words'], s['words_abs_diff']),
        ' -----------------------------------------------------------------------',
        ' ---------------------------------------------------------------',
        '| Error Rate (%)| Mean\t\t| Std.\t\t| Min./Max.\t|',
        ' ---------------------------------------------------------------',
        '| Character\t| {:2.4f}\t| {:.2f}\t\t| {:.2f}/{:.2f}\t|'.format(s['cer_mean'], s['cer_std'], s['cer_min'], s['cer_max']),
        '| Word\t\t| {:2.4f}\t| {:.2f}\t\t| {:.2f}/{:.2f}\t|'.format(s['wer_mean'], s['wer_std'], s['wer_min'], s['wer_max']),
        ' ---------------------------------------------------------------',
        'Note : If the text unit is phoneme, WER = PER and CER is meaningless.',
    ]
    return '\n'.join(lines)


def main(argv=None):
    import argparse
    ap = argparse.ArgumentParser(description='Score a result file like eval.py (default) or eval_beam.py (--beam).')
    ap.add_argument('--file', type=str, required=True)
    ap.add_argument('--beam', action='store_true')
    a = ap.parse_args(argv)
    print(format_report(score_file(a.file, beam=a.beam)))


if __name__ == '__main__':
    main()
