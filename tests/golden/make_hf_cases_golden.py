#!/usr/bin/env python3
"""Stores what HuggingFace `transformers` computes for the CPU tests that compare against it live, so that those
comparisons also run where transformers is not installed (where it is, the tests recompute it and compare against
both). Writes tests/golden/hf_cases.npz:
  * mel_filters_80, mel_filters_128: transformers.audio_utils.mel_filter_bank (slaney, 0-8 kHz, 201 bins), [n_mel][201]
    (test_host_logic.py);
  * live_masks: the -inf masks HF's logit processors (make_rules_golden.hf_processors) leave on the seeded cases
    make_rules_golden.cases(seed=LIVE_SEED, n=N_LIVE), packed bits; d1_masks / d2_masks: the same for the inputs of
    the named-difference tests, d1_cases() / d2_cases() (test_oracle_vs_hf_rules.py).
Run (needs transformers):   python tests/golden/make_hf_cases_golden.py
"""
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)
import make_rules_golden as mrg  # noqa: E402
from tools import gen_model, ggml_io  # noqa: E402

LIVE_SEED, N_LIVE = 77, 48


def hf_mel_filters(n_mel):
    from transformers.audio_utils import mel_filter_bank
    return mel_filter_bank(num_frequency_bins=201, num_mel_filters=n_mel, min_frequency=0.0, max_frequency=8000.0,
                           sampling_rate=16000, norm="slaney", mel_scale="slaney").T


def prompt(sp):
    return [sp["sot"], sp["sot"] + 1, sp["transcribe"]]


def d1_cases(sp, n_vocab):
    """D1 (initial text not forced): a text token dominates the first sampled position."""
    logits = np.random.default_rng(1).normal(0, 1, n_vocab).astype(np.float32)
    logits[2000] += 30.0
    return [([], logits)]


def d2_cases(sp, n_vocab):
    """D2 (equal timestamp allowed): text after a timestamp pair, and after the initial timestamp."""
    logits = np.random.default_rng(2).normal(0, 1, n_vocab).astype(np.float32)
    beg = sp["beg"]
    return [([beg, 1000, beg + 40, beg + 40, 1001], logits), ([beg, 1000, 1001], logits)]


def hf_case_masks(sp, vocab, cs):
    p = prompt(sp)
    procs = mrg.hf_processors(sp, vocab, len(p))
    return np.stack([mrg.hf_mask(procs, p, hist, logits)[0] for hist, logits in cs])


def main():
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "micro.bin")
        info = gen_model.generate(path, **mrg.MODEL_ARGS)
        hp, _, vocab, _ = ggml_io.read_ggml(path)
    sp, n = info["special"], hp["n_vocab"]
    live = mrg.cases(sp, n, len(vocab) - 1, seed=LIVE_SEED, n=N_LIVE)
    out = os.path.join(HERE, "hf_cases.npz")
    np.savez_compressed(out, model_args=np.array(repr(mrg.MODEL_ARGS)),
                        mel_filters_80=hf_mel_filters(80), mel_filters_128=hf_mel_filters(128),
                        live_masks=np.packbits(hf_case_masks(sp, vocab, live), axis=1),
                        d1_masks=np.packbits(hf_case_masks(sp, vocab, d1_cases(sp, n)), axis=1),
                        d2_masks=np.packbits(hf_case_masks(sp, vocab, d2_cases(sp, n)), axis=1))
    print("wrote", out)


if __name__ == "__main__":
    main()
