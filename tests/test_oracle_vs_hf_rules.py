"""CPU tests pinning the oracle's logit rules and greedy sequencing against HuggingFace's independent
implementation of the same OpenAI rules (generation/logits_process.py:1812-2046 and
WhisperForConditionalGeneration.generate). The fixtures are produced by HF code alone
(tests/golden/make_rules_golden.py -> golden/rules_hf.npz, tests/golden/make_hf_cases_golden.py ->
golden/hf_cases.npz); when `transformers` is importable the HF side is also re-run live. The two intentional
whisper.cpp-vs-OpenAI differences (D1, D2: see make_rules_golden.py) are asserted explicitly instead of being
tolerated."""
import ast
import os
import sys

import numpy as np
import pytest

from conftest import model_file, seg_ids
from tools import ggml_io, synth_audio

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import make_hf_cases_golden as mhc  # noqa: E402
import make_rules_golden as mrg  # noqa: E402


@pytest.fixture(scope="module")
def ctx(ora):
    g = np.load(os.path.join(HERE, "golden", "rules_hf.npz"))
    args = ast.literal_eval(str(g["model_args"]))
    assert args == mrg.MODEL_ARGS
    hf = np.load(os.path.join(HERE, "golden", "hf_cases.npz"))
    assert ast.literal_eval(str(hf["model_args"])) == mrg.MODEL_ARGS
    path, info = model_file(args["size"], seed=args["seed"], script_len=args["script_len"], keyed=args["keyed"])
    hp, _, vocab, _ = ggml_io.read_ggml(path)
    o = ora.Oracle(path)
    return dict(g=g, hf=hf, path=path, info=info, sp=info["special"], vocab=vocab, n_vocab=hp["n_vocab"], o=o)


def hf_masks(ctx, key, cs):
    """HF's -inf masks for the (history, logits) cases `cs`: as stored in golden/hf_cases.npz[key] and, when
    transformers is importable, recomputed live; the oracle is held to each of them."""
    out = [np.unpackbits(ctx["hf"][key], axis=1)[:, : ctx["n_vocab"]].astype(bool)]
    assert len(out[0]) == len(cs)
    try:
        import transformers  # noqa: F401
    except ImportError:
        return out
    return out + [mhc.hf_case_masks(ctx["sp"], ctx["vocab"], cs)]


def decoder_state(hist, beg):
    """whisper.cpp's per-decoder (has_ts, seek_delta) after sampling `hist`: updated by every token
    > <|0.00|> (whisper_full_with_state's "timestamp token - update sliding window" block)."""
    has_ts, seek_delta = False, 3000
    for t in hist:
        if t > beg:
            has_ts, seek_delta = True, 2 * (t - beg)
    return has_ts, seek_delta


def oracle_mask(c, hist, logits, **kw):
    o = c["o"]
    p = o.default_params(0, **dict(dict(suppress_nst=1), **kw))
    has_ts, sd = decoder_state(hist, c["sp"]["beg"])
    lo, lp, pr = o.process_logits(p, hist, has_ts, sd, 0.0, logits)
    return np.isneginf(lo), lo, lp, pr


def test_static_suppress_set_matches_vocabulary_rule(ctx):
    """The always-suppressed ids (specials, language tokens, non-speech symbols), recomputed in Python from
    the vocabulary alone, are exactly what the oracle masks on a mid-text step."""
    sp, n = ctx["sp"], ctx["n_vocab"]
    logits = np.zeros(n, np.float32)
    logits[2000] = 20.0  # a dominant text token keeps the timestamp-mass rule out of the way
    mask, _, _, _ = oracle_mask(ctx, [sp["beg"], 1000, 1001], logits)
    want = set(mrg.static_suppress_ids(ctx["vocab"], sp)) | {sp["not_"]}
    # mid-text after <|0.00|> only: no timestamp floor (has_ts is false), nothing else is masked
    assert set(np.flatnonzero(mask).tolist()) == want
    mask0, _, _, _ = oracle_mask(ctx, [sp["beg"], 1000, 1001], logits, suppress_nst=0)
    assert set(np.flatnonzero(mask0).tolist()) == set(mrg.static_suppress_ids(ctx["vocab"], sp, False)) | {sp["not_"]}


def test_masks_match_hf_golden(ctx):
    g, sp = ctx["g"], ctx["sp"]
    cs = mrg.cases(sp, ctx["n_vocab"], len(ctx["vocab"]) - 1)
    assert len(cs) == int(g["n_cases"])
    want = np.unpackbits(g["masks"], axis=1)[:, : ctx["n_vocab"]].astype(bool)
    kinds = set()
    for i, (hist, logits) in enumerate(cs):
        got, lo, lp, pr = oracle_mask(ctx, hist, logits)
        assert np.array_equal(got, want[i]), "case %d: history %s" % (i, hist)
        # what is not masked is untouched, and the log-probabilities are the log-softmax of the survivors
        keep = ~got
        assert np.array_equal(lo[keep], logits[keep])
        shift = (lo[keep].astype(np.float64) - lp[keep])
        assert np.ptp(shift) < 1e-3                       # one shared log-sum-exp
        ref = logits[keep].astype(np.float64)
        lse = np.log(np.exp(ref - ref.max()).sum()) + ref.max()
        if abs(pr.sum() - 1.0) < 1e-3:
            assert abs(shift.mean() - lse) < 1e-3         # f32 sums over up to 51865 terms
        else:
            # whisper.cpp does not renormalise after the timestamp-mass rule removed the text tokens:
            # the probabilities are those of the timestamps BEFORE the removal (their sum = ptsum < 1)
            assert got[: sp["beg"]].all() and pr.sum() < 1.0 and shift.mean() > lse
        beg = sp["beg"]
        kinds.add((len(hist) == 0, bool(hist) and hist[-1] >= beg, len(hist) >= 2 and hist[-2] >= beg))
    assert len(kinds) >= 4  # initial, after a pair, after text, after text + one timestamp


def test_masks_match_hf_live(ctx):
    sp = ctx["sp"]
    cs = mrg.cases(sp, ctx["n_vocab"], len(ctx["vocab"]) - 1, seed=mhc.LIVE_SEED, n=mhc.N_LIVE)
    hf = hf_masks(ctx, "live_masks", cs)
    for i, (hist, logits) in enumerate(cs):
        got, _, _, _ = oracle_mask(ctx, hist, logits)
        for want in hf:
            assert np.array_equal(got, want[i])


def test_named_difference_d1_initial_text_not_forced(ctx):
    """OpenAI/HF force a timestamp at the first sampled position; whisper.cpp only through the mass rule."""
    sp, n = ctx["sp"], ctx["n_vocab"]
    cs = mhc.d1_cases(sp, n)                               # no history; a text token dominates
    got, _, _, _ = oracle_mask(ctx, *cs[0])
    beg = sp["beg"]
    for want, in hf_masks(ctx, "d1_masks", cs):
        assert want[:beg].all() and not got[2000]          # HF: no text at all; whisper.cpp: text survives
        assert np.array_equal(got[beg:], want[beg:])       # same max_initial_ts window (<= 1.00 s)
    static = np.zeros(n, bool)
    static[mrg.static_suppress_ids(ctx["vocab"], sp)] = True
    static[[sp["not_"], sp["eot"], mrg.space_id(ctx["vocab"])]] = True
    assert np.array_equal(got[:beg], static[:beg])         # and exactly the static + blank suppression below it


def test_named_difference_d2_equal_timestamp_allowed(ctx):
    """After text that follows a timestamp, HF forbids timestamps <= the last one; whisper.cpp only < it."""
    sp, n = ctx["sp"], ctx["n_vocab"]
    beg = sp["beg"]
    cs = mhc.d2_cases(sp, n)
    for masks in hf_masks(ctx, "d2_masks", cs):
        for (hist, logits), want in zip(cs, masks):
            got, _, _, _ = oracle_mask(ctx, hist, logits)
            last = max(t for t in hist if t >= beg)
            diff = np.flatnonzero(got != want)
            assert diff.tolist() == [last] and want[last] and not got[last]


def test_greedy_sequence_matches_hf_generate_golden(ctx, ora):
    """Prompt construction, the rules in context and the EOT stop: HF's greedy generate(return_timestamps=True)
    and the oracle's whisper_full restatement sample the same tokens (oracle in HF-comparable numerics:
    erf-GELU, f32 activations). HF returns every sampled token; whisper.cpp's segments drop the second
    timestamp of a pair and EOT."""
    g, sp = ctx["g"], ctx["sp"]
    o = ora.Oracle(ctx["path"], weight_round=False, act_round=ora.ACT_F32, gelu_erf=True)
    p = o.default_params(0, language="en", temperature_inc=0.0, suppress_nst=1)
    for i in range(g["hf_sequences"].shape[0]):
        seq = [int(t) for t in g["hf_sequences"][i] if t >= 0]
        if seq[: len(g["prompt"])] == g["prompt"].tolist():
            seq = seq[len(g["prompt"]):]
        kept = [t for j, t in enumerate(seq) if t != sp["eot"] and not (j > 0 and t >= sp["beg"] and seq[j - 1] == t)]
        r = o.full(synth_audio.to_f32(mrg.golden_clip(ctx["info"], i)), p)
        assert seg_ids(r) == kept
    assert len({tuple(int(t) for t in row) for row in g["hf_sequences"]}) == 3  # three clips, three transcripts
