"""CPU tests of the host-side logic around the path: synthetic asset generators, ggml format
round trip, utterance sharding and the 2-rank (gloo) gather / max-time plumbing of bench.py."""
import os
import subprocess
import sys

import numpy as np

from conftest import ROOT, load_pkg_module, model_file
from tools import ggml_io, synth_audio

sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_hf_cases_golden as mhc  # noqa: E402


def test_ggml_file_layout(micro_model):
    path, info = micro_model
    hp, filters, vocab, T = ggml_io.read_ggml(path)
    assert hp["n_vocab"] == 51865 and hp["n_audio_ctx"] == 1500 and hp["n_text_ctx"] == 448
    assert filters.shape == (80, 201) and abs(filters.sum(1).min()) > 0
    assert len(vocab) == 50257 and vocab[32] == b" "
    d = hp["n_audio_state"]
    assert T["encoder.conv1.weight"].shape == (d, 80, 3)
    assert T["encoder.conv1.bias"].shape == (d, 1)
    assert T["decoder.token_embedding.weight"].shape == (51865, d)
    assert "encoder.blocks.0.attn.key.bias" not in T
    assert info["special"]["beg"] == 50364 and info["special"]["eot"] == 50257


def test_special_tokens_large_v3_and_english_only():
    from tools import gen_model
    lv3 = gen_model.special_tokens(51866)
    assert (lv3["translate"], lv3["transcribe"], lv3["beg"], lv3["n_langs"]) == (50359, 50360, 50365, 100)
    en = gen_model.special_tokens(51864)
    assert (en["eot"], en["sot"], en["beg"]) == (50256, 50257, 50363)


def test_mel_filterbank_matches_transformers():
    """Against transformers' mel_filter_bank as stored in tests/golden/hf_cases.npz and, where transformers is
    importable, computed live."""
    from tools import gen_model
    g = np.load(os.path.join(ROOT, "tests", "golden", "hf_cases.npz"))
    try:
        import transformers  # noqa: F401
        live = True
    except ImportError:
        live = False
    for n_mel in (80, 128):
        got = gen_model.mel_filterbank(n_mel)
        for ref in [g["mel_filters_%d" % n_mel]] + ([mhc.hf_mel_filters(n_mel)] if live else []):
            assert ref.shape == (n_mel, 201) and np.abs(got - ref).max() < 1e-6


def test_synthetic_audio_is_seeded_and_shaped():
    a = synth_audio.utterance(5, 7)
    b = synth_audio.utterance(5, 7)
    c = synth_audio.utterance(5, 8)
    assert a.dtype == np.int16 and len(a) == 480000 and (a == b).all() and (a != c).any()
    assert abs(int(np.abs(a).max()) - 16383) <= 1
    d = synth_audio.durations_config4(16)
    assert all(5.0 <= x <= 30.0 for x in d) and len(set(d)) > 8
    f = synth_audio.to_f32(a)
    assert f.dtype == np.float32 and f[0] == np.float32(a[0]) / np.float32(32768.0)


def test_sharding_covers_every_utterance_once():
    dp = load_pkg_module("dispatch")
    for n, world in ((1024, 8), (256, 4), (7, 2), (3, 4)):
        seen = sorted(i for r in range(world) for i in dp.shard_utterances(n, world, r))
        assert seen == list(range(n))
    lens = synth_audio.durations_config4(256)
    parts = [dp.shard_utterances(256, 4, r, lens) for r in range(4)]
    assert sorted(i for p in parts for i in p) == list(range(256))
    sums = [sum(lens[i] for i in p) for p in parts]
    assert max(sums) - min(sums) < 30.0  # balanced to within one utterance


def test_two_rank_gather_and_max_time_gloo(tmp_path):
    script = tmp_path / "rank.py"
    script.write_text('''
import os, sys, importlib.util
import torch.distributed as dist
spec = importlib.util.spec_from_file_location("dispatch", sys.argv[1]); dp = importlib.util.module_from_spec(spec); spec.loader.exec_module(dp)
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
idx = dp.shard_utterances(10, world, rank, [float(i % 5 + 1) for i in range(10)])
local = [{"utt": i, "rank": rank} for i in idx]
out = dp.gather_results(local, idx, 10, world, rank)
t = dp.max_over_ranks(1.0 + rank, world)
if rank == 0:
    assert [o["utt"] for o in out] == list(range(10)), out
    assert {o["rank"] for o in out} == {0, 1}
    assert t == 2.0
    print("GATHER_OK")
else:
    assert out is None and t == 2.0
dist.destroy_process_group()
''')
    dispatch = os.path.join(ROOT, "sentiric-stt-whisper-service_b200", "dispatch.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29617", str(script), dispatch],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "GATHER_OK" in r.stdout, r.stdout + r.stderr


def test_bench_reference_arm_other_ranks_do_no_work():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, env=env, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""
