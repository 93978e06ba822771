#!/usr/bin/env python3
"""Benchmark of the Whisper hot path on B200 (BASELINE.json: audio-sec/sec, large-v3).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA engine
    python bench.py --impl reference --gpus N --steps K ...  # the CPU arm (oracle; see below)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results (dump_outputs):
                                                             # rank 0's windows only under --gpus > 1; not with --inproc

Workload (BASELINE.json configs[4], the configuration the metric is quoted on, per GPU):
Whisper large-v3 (128 mel), greedy, batch 64, 128 x 30 s windows per GPU per step (1024 windows
over 8 GPUs), seeded synthetic ggml weights of the "keyed" kind (tools/gen_model.py --keyed: a
~100-token timestamped transcript whose 85 text tokens are each chosen, out of 4 alternatives, by the AUDIO
through mel -> encoder -> cross attention), synthetic 16 kHz clips that spell a different seeded symbol
sequence per window (tools/synth_audio.keyed_clip). One "step" = one pass of the whole hot
path (PCM -> log-mel -> conv stem -> encoder -> cross-KV -> greedy decode -> segments) over the
rank's 128 windows. Windows are independent: ranks share nothing (weak scaling, no collective on
the data path); torch.distributed is used only for the barrier and the max-over-ranks time. The context
runs two lanes (two batches of 64 windows in flight on the GPU, weights shared; `stages.lanes`).

`value` : audio-seconds per second with the PCM already resident in HBM (device pointers in).
`e2e`   : the same through the reference-facing C-ABI call with pinned HOST buffers (H2D of the
          PCM and the D2H read-back of picks / token-timestamp energy inside the timed region).
The reference arm (`--impl reference`) times the CPU oracle (a restatement of whisper.cpp v1.8.2,
"CPU restatement, not ggml": the reference's own whisper.cpp cannot be built here, DESIGN.md) on a
bounded sample of the same workload: one window per step, all host threads.
"""
import argparse
import ctypes as C
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PKG = os.path.join(ROOT, "sentiric-stt-whisper-service_b200")

SERVICE_PARAMS = dict(  # what SttEngine::transcribe sets (stt_engine.cpp:204-243) with config.h defaults
    language="en", token_timestamps=1, suppress_nst=1, no_speech_thold=0.85, logprob_thold=-0.7,
    entropy_thold=2.40, temperature=0.0)


def load_binding():
    spec = importlib.util.spec_from_file_location("sw_binding", os.path.join(PKG, "sw_binding.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"],
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback (B200_PROFILING.md)")


KEYED_K = 4


def model_path(size, script_len):
    return "/tmp/sw_bench_%s_s%d_k%d.bin" % (size, script_len, KEYED_K)


def ensure_model(size, script_len):
    from tools import gen_model
    path = model_path(size, script_len)
    if not (os.path.exists(path) and os.path.exists(path + ".json")):
        tmp = path + ".tmp%d" % os.getpid()
        info = gen_model.generate(tmp, size, script_len=script_len, keyed=KEYED_K)
        os.replace(tmp, path)
        json.dump(dict(script=[int(t) for t in info["script"]], special=info["special"], keyed=info["keyed"]),
                  open(path + ".json", "w"))
    return path


def model_info(path):
    return json.load(open(path + ".json"))


def window_clip(info, index):
    """Window `index` of the workload: a clip that spells its own seeded symbol sequence, and the transcript
    (token ids, as the engine reports them) a correct path must therefore return for it. The bench checks
    every window of one pass against it: a fast step that does not listen to its audio cannot pass."""
    from tools import gen_model, synth_audio
    sym = synth_audio.keyed_symbols(info["keyed"], 5000 + index)
    return synth_audio.keyed_clip(info["keyed"], sym, seed=5000 + index), gen_model.keyed_expected_tokens(info, sym)


DUMP_LIMIT = 64 << 20
TOKEN_FLOATS = ("p", "plog", "pt", "ptsum", "vlen")


def dump_outputs(out_dir, windows, results):
    """Writes what a caller received from the last timed step, one array per field as out_dir/<name>.npy, so that
    two builds can be compared output for output: per window (`windows[i]` is result i's index in the workload) its
    language and decoder step count, per segment its bounds, per token its id, timestamp token, probabilities and
    times, each row tagged with its window (and segment). Token probabilities are float32 as computed; integers are
    stored exactly as float64. Above DUMP_LIMIT bytes in all, a seeded sample of whole windows is written."""
    def tables(sel):
        t = {k: [] for k in ("window_index", "window_lang_id", "window_n_decode_steps", "segment_window",
                             "segment_t0", "segment_t1", "segment_speaker_turn_next", "token_window", "token_segment",
                             "token_id", "token_tid", "token_t0", "token_t1") + tuple("token_" + f for f in TOKEN_FLOATS)}
        for i in sel:
            w, r = windows[i], results[i]
            t["window_index"].append(w)
            t["window_lang_id"].append(r["lang_id"])
            t["window_n_decode_steps"].append(r["n_decode_steps"])
            for s, seg in enumerate(r["segments"]):
                t["segment_window"].append(w)
                for k in ("t0", "t1", "speaker_turn_next"):
                    t["segment_" + k].append(seg[k])
                for tok in seg["tokens"]:
                    t["token_window"].append(w)
                    t["token_segment"].append(s)
                    for k in ("id", "tid", "t0", "t1") + TOKEN_FLOATS:
                        t["token_" + k].append(tok[k])
        floats = {"token_" + f for f in TOKEN_FLOATS}
        return {k: np.asarray(v, np.float32 if k in floats else np.float64) for k, v in t.items()}

    size = [sum(a.nbytes for a in tables([i]).values()) for i in range(len(results))]
    sel = list(range(len(results)))
    if sum(size) > DUMP_LIMIT:
        sel, total = [], 0
        for i in np.random.default_rng(0).permutation(len(results)):
            if total + size[i] > DUMP_LIMIT:
                break
            sel.append(int(i))
            total += size[i]
        sel.sort()
    os.makedirs(out_dir, exist_ok=True)
    for k, a in tables(sel).items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    print("bench.py: outputs of %d of %d windows of the last timed step written to %s" % (len(sel), len(results), out_dir),
          file=sys.stderr)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names)
                   if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=reasons, samples=len(sm))


def run_reference(args, rank, world):
    """CPU arm: the oracle on the host cores, one 30 s window of the same workload per step."""
    if rank != 0:
        return
    from oracle import ora
    from tools import synth_audio
    path = ensure_model(args.model, args.script_len)
    cores = os.cpu_count() or 1
    o = ora.Oracle(path, weight_round=False, act_round=ora.ACT_F16, threads=cores)
    beam = int(CONFIGS[args.config].get("beam", 1))
    p = o.default_params(1, beam_size=beam, **SERVICE_PARAMS) if beam > 1 else o.default_params(0, **SERVICE_PARAMS)
    times = []
    info = model_info(path)
    for s in range(args.warmup + args.steps):
        pcm = synth_audio.to_f32(window_clip(info, s)[0])
        t0 = time.perf_counter()
        r = o.full(pcm, p)
        dt = time.perf_counter() - t0
        if s >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [s], [r])
    total = sum(times)
    val = 30.0 * len(times) / total
    line = dict(
        impl="reference", metric="audio-sec/sec (RTFx)", value=val, unit="audio-sec/sec",
        n_gpus=args.gpus, steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * total / len(times),
        higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f16 weights, f32 accumulate",
        data="synthetic",
        config=dict(workload="whisper %s %s, one 30 s window per step (bounded sample of: %s)" %
                             (args.model, "beam 5" if beam > 1 else "greedy", CONFIGS[args.config]["what"]),
                    baseline_config=args.config, script_tokens=args.script_len),
        cpu_baseline=dict(value=val, unit="audio-sec/sec", cores=cores, kind="port",
                          sample="1 x 30 s window per step, %d steps; CPU restatement of whisper.cpp "
                                 "v1.8.2, not ggml" % args.steps),
        e2e=dict(value=val, unit="audio-sec/sec", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
        n_decode_steps=r["n_decode_steps"])
    print(json.dumps(line), flush=True)


CONFIGS = {
    # BASELINE.json configs[i-1]; 5 is the one the metric is quoted on (default)
    1: dict(model="tiny", script_len=60, windows=1, batch=1, beam=1,
            what="Whisper tiny greedy, ONE 30 s clip (the reference's own CPU-runnable case): the CPU arm beside it is "
                 "the headline of this line"),
    2: dict(model="base", script_len=60, windows=32, batch=32, beam=1,
            what="Whisper base, batch of 32 x 30 s windows, mel + encoder + greedy decode"),
    3: dict(model="small", script_len=60, windows=32, batch=32, beam=5,
            what="Whisper small (12 + 12 layers), beam search with 5 beams over the paged self-KV cache, 32 x 30 s windows"),
    4: dict(model="medium", script_len=60, total=256, batch=64, beam=1, ragged=True, langs=["en", "tr", "de", "ja"],
            what="Whisper medium multilingual, 256 utterances of mixed 5-30 s length (language cycled over en/tr/de/ja) "
                 "dealt to the ranks by descending length (dispatch.shard_utterances)"),
    5: dict(model="large-v3", script_len=100, windows=128, batch=64, beam=1,
            what="whisper large-v3 greedy batch-64, 128 x 30 s windows per GPU per step (BASELINE configs[4] share of one GPU)"),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=5, choices=sorted(CONFIGS),
                    help="BASELINE.json configs[N-1]; 5 (default) is the configuration the metric is quoted on")
    ap.add_argument("--model", default=None)
    ap.add_argument("--windows-per-gpu", type=int, default=None)
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--script-len", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--oracle-windows", type=int, default=3, help="windows the CPU oracle also transcribes (parity + cpu_baseline)")
    ap.add_argument("--inproc", type=int, default=0,
                    help="N > 0: ONE process, N contexts on devices 0..N-1 driven by N host threads (the in-process "
                         "dispatcher of SURVEY.md §8(e)) instead of one process per GPU; prints the same line with "
                         "mode=inproc")
    ap.add_argument("--facade", action="store_true", default=True,
                    help="(default) also measure the reference-facing class: caller threads on SttEngine::transcribe_pcm16 "
                         "with pageable vectors (host/stt_cli bench mode) -> e2e_facade")
    ap.add_argument("--no-facade", dest="facade", action="store_false")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the results of the last timed step (rank 0's windows) as "
                         "DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.inproc > 0:
        ap.error("--dump-outputs is not supported with --inproc")
    cfg = dict(CONFIGS[args.config])
    if args.model:
        cfg["model"] = args.model
    if args.batch:
        cfg["batch"] = args.batch
    if args.script_len:
        cfg["script_len"] = args.script_len
    if args.windows_per_gpu:
        cfg["windows"] = args.windows_per_gpu
        cfg.pop("total", None)
    args.model, args.batch, args.script_len = cfg["model"], cfg["batch"], cfg["script_len"]

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return 0
    if args.inproc > 0:
        return run_inproc(args, cfg)

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- model (rank 0 of the node generates the seeded file once)
    if local_rank == 0:
        ensure_model(args.model, args.script_len)
    barrier()
    path = model_path(args.model, args.script_len)
    minfo = model_info(path)

    swb = load_binding()
    from tools import gen_model, synth_audio
    disp = importlib.util.spec_from_file_location("dispatch", os.path.join(PKG, "dispatch.py"))
    dispatch = importlib.util.module_from_spec(disp)
    disp.loader.exec_module(dispatch)
    beam = int(cfg.get("beam", 1))
    eng = swb.Engine(path, device=local_rank, max_batch=args.batch, max_beams=5)
    # host sequencer workers (the Settings.n_threads knob): this rank's share of the box's cores
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    cores_here = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 4)
    n_threads = max(2, min(16, cores_here // max(1, local_world)))
    langs = cfg.get("langs", ["en"])

    def make_params(lang):
        kw = dict(SERVICE_PARAMS, language=lang)
        p = eng.default_params(1, beam_size=beam, **kw) if beam > 1 else eng.default_params(0, **kw)
        p.n_threads = n_threads  # greedy: best_of 5, temperature_inc 0.2 (defaults)
        return p
    params_by_lang = {lg: make_params(lg) for lg in langs}
    eng.set_kernel_timing(True)

    # ---- this rank's utterances: int16 PCM, pinned host copy + device copy
    if cfg.get("ragged"):
        total = int(cfg["total"])
        durs = synth_audio.durations_config4(total)
        mine = dispatch.shard_utterances(total, world, rank, lengths=durs)   # dealt by descending length
        scaling = "strong"
    else:
        W0 = int(cfg["windows"])
        durs = [30.0] * (W0 * world)
        mine = dispatch.shard_utterances(W0 * world, world, rank)            # contiguous blocks: weak scaling
        scaling = "weak"
    W = len(mine)
    n_samp = [int(round(durs[i] * 100)) * 160 for i in mine]
    offs = np.concatenate([[0], np.cumsum(n_samp)]).astype(np.int64)
    L = swb.lib()
    host = L.sw_host_alloc(int(offs[-1]) * 2)
    if not host:
        raise SystemExit("pinned allocation failed: " + swb.last_error())
    host_np = np.ctypeslib.as_array(C.cast(host, C.POINTER(C.c_int16)), shape=(int(offs[-1]),))
    want_ids, n_sure = [], []
    for j, i in enumerate(mine):
        clip, ids = window_clip(minfo, i)
        host_np[offs[j]:offs[j + 1]] = clip[: n_samp[j]]
        want_ids.append(ids)
        # tokens a clip shorter than 30 s still decides (tone slots wholly inside the audio)
        n_sure.append(len(ids) if n_samp[j] >= 480000 else gen_model.keyed_sure_prefix(minfo, n_samp[j]))
    dev = torch.from_numpy(host_np.copy()).cuda()
    ptr16 = C.POINTER(C.c_int16)
    # ONE C-ABI call per step: sw_full_batch_pcm16_lang carries a language per utterance (utterance i of
    # config 4 speaks langs[i % 4]), so mixed-language work shares device passes
    idx = list(range(W))
    groups = [dict(
        lang=langs[0], idx=idx, n=W, lens=(C.c_int * W)(*n_samp),
        langs=(C.c_char_p * W)(*[langs[mine[j] % len(langs)].encode() for j in idx]) if len(langs) > 1 else None,
        host=(ptr16 * W)(*[C.cast(host + int(offs[j]) * 2, ptr16) for j in idx]),
        dev=(ptr16 * W)(*[C.cast(dev.data_ptr() + int(offs[j]) * 2, ptr16) for j in idx]))]

    L.sw_result_token_data.restype = swb.TokenData
    parity = dict(windows=0, token_identical_to_expected=0, distinct_transcripts=0)
    seen, got_ids = set(), {}

    def step(which, check=False, keep=None):
        """One pass over the rank's windows. keep: a list that takes (window, result handle) pairs instead of
        freeing the results, for reading after the timed region."""
        n_tok = 0
        for g in groups:
            res = eng.full_batch_ptrs(g[which], g["lens"], g["n"], params_by_lang[g["lang"]], languages=g["langs"])
            for w, r in zip(g["idx"], res):
                ids = []
                for s in range(L.sw_result_n_segments(r)):
                    nt = L.sw_result_n_tokens(r, s)
                    n_tok += nt
                    if check:
                        ids += [L.sw_result_token_data(r, s, j).id for j in range(nt)]
                if check:
                    parity["windows"] += 1
                    k = n_sure[w]
                    parity["token_identical_to_expected"] += int(ids[:k] == want_ids[w][:k] and (k < len(want_ids[w]) or ids == want_ids[w]))
                    seen.add(tuple(ids))
                    got_ids[w] = ids
                if keep is not None:
                    keep.append((w, r))
                else:
                    L.sw_result_free(r)
        return n_tok

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(which, k, keep=None):
        """K steps between a barrier + device synchronize on both sides, timed with two CUDA events. The device
        is idle when the first is recorded (synchronize just before) and every step call returns only after
        its last kernel and read-back have completed (the sequencer reads the picks of every decoder step), so
        the second event, recorded behind the last step, closes the region on the device. The host clock
        around the same region is reported next to it (`host_ms_per_step`); the two must agree."""
        barrier()
        t0 = time.perf_counter()
        ev0.record()
        n_tok = 0
        for i in range(k):
            n_tok += step(which, keep=keep if i == k - 1 else None)
        ev1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        dt = ev0.elapsed_time(ev1) * 1e-3
        if world > 1:
            t = torch.tensor([dt, wall], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt, wall = float(t[0].item()), float(t[1].item())
        return dt, n_tok, wall

    for i in range(args.warmup):
        step("dev", check=(i == 0))  # untimed: every window of the first warm-up pass is checked
    eng.stats(reset=True)
    clocks = ClockSampler(local_rank)
    if rank == 0:  # one sampler per job: the line reports rank 0's GPU, and nvidia-smi polling is not free
        clocks.start()
    last = [] if args.dump_outputs and rank == 0 else None
    dt, n_tok, wall = timed("dev", args.steps, keep=last)
    st = eng.stats(reset=True)
    dt_e2e, _, wall_e2e = timed("host", args.steps)
    st_e2e = eng.stats(reset=True)
    clk = clocks.stop()
    if last is not None:
        dump_outputs(args.dump_outputs, [mine[w] for w, _ in last], [eng._collect(r) for _, r in last])

    audio_local = float(sum(n_samp)) / 16000.0
    audio_all = audio_local
    if world > 1:
        t = torch.tensor([audio_local], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        audio_all = float(t.item())
    audio_s = audio_all * args.steps
    value = audio_s / dt
    e2e = audio_s / dt_e2e
    pk = peaks()
    info = eng.info
    d, Le, Ld, nm = info.n_audio_state, info.n_audio_layer, info.n_text_layer, info.n_mels
    flops_win = (2 * 3000 * nm * 3 * d + 2 * 1500 * d * 3 * d + Le * (24 * 1500 * d * d + 4 * 1500 * 1500 * d)
                 + Ld * 4 * 1500 * d * d)
    lanes = max(1, int(st.get("n_lanes", 1)))
    # device times are SUMS over the context's lanes, which run concurrently: the time the device spent
    # on a stage is the sum divided by the lanes (both lanes enter and leave each stage together here:
    # one sub-batch of `batch` windows per lane)
    for k in ("ms_mel", "ms_encode", "ms_decode"):
        st[k + "_sum"] = st[k]
        st[k] = st[k] / lanes
    xa_ms = st["ms_xattn"] / max(1, st["n_xattn"])
    xa_bytes = st["xattn_bytes"] / max(1, st["n_xattn"])
    xa_gbs = xa_bytes / (xa_ms * 1e-3) / 1e9 if xa_ms > 0 else 0.0
    enc_tf = flops_win * st["n_windows"] / (st["ms_encode"] * 1e-3) / 1e12 if st["ms_encode"] > 0 else 0.0
    dec_gbs = st["decode_bytes"] / (st["ms_decode"] * 1e-3) / 1e9 if st["ms_decode"] > 0 else 0.0
    pcm_bytes = float(sum(n_samp)) * 2

    line = dict(
        metric="audio-sec/sec (RTFx)", value=value, unit="audio-sec/sec", n_gpus=world,
        steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * dt / args.steps,
        host_ms_per_step=1e3 * wall / args.steps,
        timing="CUDA events around the K steps, max over ranks (host clock of the same region: host_ms_per_step)",
        higher_is_better=True, scaling=scaling, vs_baseline=None, dtype="bf16 (f32 accumulate)",
        data="synthetic",
        config=dict(workload=cfg["what"], baseline_config=args.config, model=args.model,
                    windows_per_gpu=W, batch=args.batch, beam=beam, script_tokens=args.script_len,
                    audio_seconds_per_step=audio_all,
                    params="SttEngine defaults: %s, token_timestamps, suppress_nst, temperature_inc 0.2" %
                           ("beam search (5 beams)" if beam > 1 else "greedy (best_of 5)"),
                    lanes="%d lanes (batches in flight) x batch %d" % (lanes, args.batch),
                    host_threads=int(n_threads),
                    l2="per-step working set (cross-KV %.1f GB) exceeds the 126 MB L2" %
                       (Ld * 2 * 1500 * d * 2 * min(args.batch, W) / 1e9)),
        e2e=dict(value=e2e, unit="audio-sec/sec",
                 h2d_bytes_per_step=int(st_e2e["h2d_bytes"] / args.steps),
                 d2h_bytes_per_step=int(st_e2e["d2h_bytes"] / args.steps)),
        gpu_launches=int(st["n_launches"]),
        parity_check=dict(parity, distinct_transcripts=len(seen),
                          note="token ids of every window of one pass vs the transcript its own clip spells "
                               "(keyed model: most tokens of a window are chosen by the audio; clips shorter than 30 s "
                               "are compared up to the first timestamp past their end)"),
        clocks=clk,
        roofline=dict(bound="hbm", kernel="cross_attention_kernel", achieved=xa_gbs, peak=pk["hbm"],
                      unit="GB/s", frac=xa_gbs / pk["hbm"],
                      # dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full
                      # (profiles/r2_ncu_xattn_v2.txt: 491.76 MB read = the algorithmic bytes, 5.1 MB of partials
                      # written; large-v3, 64 windows, one lane)
                      traffic=496.9e6 if (args.model == "large-v3" and args.batch == 64) else None,
                      traffic_source="constant: dram bytes of one launch from the committed ncu --set full capture "
                                     "(profiles/r2_ncu_xattn_v2.txt), not re-measured by this run",
                      avg_launch_ms=xa_ms, algorithmic_bytes_per_launch=xa_bytes, peak_source=pk["src"],
                      note=("timed with CUDA events on the lanes' streams inside the timed region. Under lanes the two "
                            "lanes' cache streams alternate and, with programmatic dependent launch, overlap: a launch (96 "
                            "CTAs) spends part of its elapsed time waiting for the SMs the other lane's stream still holds, so "
                            "the per-launch durations of the two lanes add up to MORE than the wall time (profiles/"
                            "r2_xattn_timeline.txt) and this fraction understates the kernel. `alone` is the same kernel timed "
                            "the same way in a one-lane pass after the timed region (148 CTAs, nothing else on the GPU); "
                            "stages.decode_frac_of_hbm is the aggregate of both lanes (all decode bytes / decode time).")
                      if lanes > 1 else None),
        stages=dict(
            lanes=lanes,
            lanes_note="device_ms_per_step = per-lane device time summed over lanes / lanes (lanes overlap in time)",
            tokens_per_window=n_tok / max(1, W * args.steps),
            decode_steps=int(st["n_steps"] / args.steps),
            device_ms_per_step=dict(mel=st["ms_mel"] / args.steps, encode=st["ms_encode"] / args.steps,
                                    decode=st["ms_decode"] / args.steps),
            frontend_gbs=(pcm_bytes + nm * 3000 * 4 * W) * args.steps / max(1e-9, st["ms_mel"] * 1e-3) / 1e9,
            frontend_note="(int16 PCM in + f32 log-mel out) / device time of the front end (mel + token-timestamp energy kernels, uploads)",
            encoder_ms_per_window=st["ms_encode"] / max(1, st["n_windows"]),
            encoder_tflops=enc_tf, encoder_frac_of_sustained_peak=enc_tf / pk["tf_sust"],
            decode_gbs=dec_gbs, decode_frac_of_hbm=dec_gbs / pk["hbm"]))

    def clip_i16(w):
        return host_np[offs[w]:offs[w + 1]]

    # ---- prosody row (SURVEY.md §8(f) rank 3): every window cut into six 5 s segments, through the C ABI
    # with host int16 buffers (upload inside the timed region), next to the reference's own host code
    if rank == 0 and args.config == 5:
        segs = [(k * 80000, (k + 1) * 80000) for k in range(6)]
        eng.prosody_segments(clip_i16(0), segs)
        t0 = time.perf_counter()
        for i in range(W):
            eng.prosody_segments(clip_i16(i), segs)
        dtp = time.perf_counter() - t0
        line["stages"]["prosody"] = dict(
            gpu_audio_s_per_s=30.0 * W / dtp, ms_per_window=1e3 * dtp / W, segments_per_window=6,
            pcm_gbs=W * 480000 * 2 / dtp / 1e9,
            note="sw_prosody_segments_pcm16 per 30 s window, host int16 in, upload + 2 kernels + read-back")
        if world == 1 and not args.no_cpu_baseline:
            from oracle import prosody as pro
            impl = pro.reference()
            kind = "reference" if impl is not None else "port"
            impl = impl or pro.oracle()
            f32 = synth_audio.to_f32(clip_i16(0))
            t0 = time.perf_counter()
            for a, b in segs:
                impl.extract(f32[a:b])
            dtc = time.perf_counter() - t0
            line["stages"]["prosody"]["cpu_baseline"] = dict(
                value=30.0 / dtc, unit="audio-sec/sec", cores=1, kind=kind,
                sample="extract_prosody over the 6 segments of one window (%s)" %
                       ("oracle/_ref: the reference's own prosody_extractor.cpp" if kind == "reference"
                        else "oracle/prosody_oracle.cpp"))

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # CPU arm beside the GPU number (oracle = "CPU restatement of whisper.cpp v1.8.2, not ggml"), outside
        # every timed region: the reference's default n_threads = 4 (config.h:40) and all host cores; the same
        # windows are also the oracle leg of the parity check (token ids vs the engine's, window by window)
        from oracle import ora
        cores = os.cpu_count() or 1
        o = ora.Oracle(path, weight_round=False, act_round=ora.ACT_F16, threads=cores)
        n_ora = max(1, min(W, args.oracle_windows))
        t_all, same, a_all = 0.0, 0, 0.0
        same_whole, mism = 0, []
        for w in range(n_ora):
            lg = langs[mine[w] % len(langs)]
            kw = dict(SERVICE_PARAMS, language=lg)
            po = o.default_params(1, beam_size=beam, **kw) if beam > 1 else o.default_params(0, **kw)
            pcm = synth_audio.to_f32(clip_i16(w))
            t0 = time.perf_counter()
            r = o.full(pcm, po)
            t_all += time.perf_counter() - t0
            a_all += len(pcm) / 16000.0
            ids = [t["id"] for sg in r["segments"] for t in sg["tokens"]]
            got = got_ids.get(w) or []
            # same rule as against the expected transcript: a clip shorter than 30 s is compared on the prefix its
            # audio decides (behind it the keyed model's alternatives are near-ties); whole-sequence equality and the
            # first differing position are reported next to it
            k = n_sure[w]
            ok = ids[:k] == got[:k] and (k < len(want_ids[w]) or ids == got)
            same += int(ok)
            same_whole += int(ids == got)
            if ids != got:
                first = next((j for j in range(min(len(ids), len(got))) if ids[j] != got[j]), min(len(ids), len(got)))
                mism.append(dict(window=w, first_difference=first, decided_prefix=k, tokens=len(got), oracle_tokens=len(ids),
                                 audio_s=n_samp[w] / 16000.0))
        line["parity_check"]["oracle_windows"] = n_ora
        line["parity_check"]["token_identical_to_oracle"] = same
        line["parity_check"]["whole_sequence_identical_to_oracle"] = same_whole
        if mism:
            line["parity_check"]["oracle_differences"] = mism
        line["cpu_baseline"] = dict(
            value=a_all / t_all, unit="audio-sec/sec", cores=cores, kind="port",
            sample="%d of the %d windows (%.0f s of audio), %.1f s of CPU; CPU restatement of whisper.cpp "
                   "v1.8.2, not ggml" % (n_ora, W, a_all, t_all))
        if cores > 4:
            o.set_threads(4)
            po = o.default_params(1, beam_size=beam, **dict(SERVICE_PARAMS, language=langs[mine[0] % len(langs)])) \
                if beam > 1 else o.default_params(0, **dict(SERVICE_PARAMS, language=langs[mine[0] % len(langs)]))
            t0 = time.perf_counter()
            o.full(synth_audio.to_f32(clip_i16(0)), po)
            dt4 = time.perf_counter() - t0
            line["cpu_baseline"]["n_threads_4"] = dict(
                value=n_samp[0] / 16000.0 / dt4, cores=4,
                sample="1 window with the reference's default n_threads = 4 (config.h:40), %.1f s" % dt4)
        o.close()
    eng.close()
    if rank == 0 and world == 1 and lanes > 1 and xa_ms > 0:
        # the dominant kernel with the GPU to itself: one lane (uncapped persistent grid), one pass of `batch`
        # windows from pinned host buffers, outside every timed region
        n1 = min(W, args.batch)
        eng1 = swb.Engine(path, device=local_rank, max_batch=args.batch, max_beams=5, n_lanes=1)
        eng1.set_kernel_timing(True)
        p1 = eng1.default_params(1, beam_size=beam, **dict(SERVICE_PARAMS, language=langs[0])) if beam > 1 else \
            eng1.default_params(0, **dict(SERVICE_PARAMS, language=langs[0]))
        p1.n_threads = n_threads
        for rep in range(2):
            if rep == 1:
                eng1.stats(reset=True)
            for r in eng1.full_batch_ptrs(groups[0]["host"], groups[0]["lens"], n1, p1,
                                          languages=groups[0]["langs"]):
                L.sw_result_free(r)
        s1 = eng1.stats(reset=True)
        eng1.close()
        if s1["n_xattn"] > 0 and s1["ms_xattn"] > 0:
            ms1 = s1["ms_xattn"] / s1["n_xattn"]
            b1 = s1["xattn_bytes"] / s1["n_xattn"]
            line["roofline"]["alone"] = dict(
                achieved=b1 / (ms1 * 1e-3) / 1e9, frac=b1 / (ms1 * 1e-3) / 1e9 / pk["hbm"], avg_launch_ms=ms1,
                algorithmic_bytes_per_launch=b1, windows=n1,
                decode_frac_of_hbm=s1["decode_bytes"] / (s1["ms_decode"] * 1e-3) / 1e9 / pk["hbm"],
                note="one lane, %d windows, persistent grid on every SM; CUDA events on the lane's stream" % n1)
    if rank == 0 and world == 1 and args.facade:
        line["e2e_facade"] = run_facade(args, path, host_np, offs, n_samp, beam, langs[0])
    if rank == 0:
        print(json.dumps(line), flush=True)
    L.sw_host_free(host)
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_inproc(args, cfg):
    """One process, N GPUs: a host dispatcher deals the utterances to per-GPU worker threads, each with its own
    sw_ctx (weights replicated), streams and lanes; results come back to the caller through the threads' result
    lists (SURVEY.md §8(e) "host dispatcher ... host-side result gather"). No collective, no torch.distributed.
    Timed per device with CUDA events (max over devices) and with the host clock around all threads."""
    import torch
    N = args.inproc
    if torch.cuda.device_count() < N:
        raise SystemExit("bench.py --inproc %d: only %d CUDA devices" % (N, torch.cuda.device_count()))
    from tools import synth_audio
    disp = importlib.util.spec_from_file_location("dispatch", os.path.join(PKG, "dispatch.py"))
    dispatch = importlib.util.module_from_spec(disp)
    disp.loader.exec_module(dispatch)
    path = ensure_model(args.model, args.script_len)
    minfo = model_info(path)
    swb = load_binding()
    L = swb.lib()
    L.sw_result_token_data.restype = swb.TokenData
    W0 = int(cfg.get("windows", 128))
    total = W0 * N
    n_s = 480000
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 4)
    ptr16 = C.POINTER(C.c_int16)
    workers = []
    for dev in range(N):
        eng = swb.Engine(path, device=dev, max_batch=args.batch, max_beams=5)
        p = eng.default_params(0, **SERVICE_PARAMS)
        p.n_threads = max(2, min(16, cores // N))
        mine = dispatch.shard_utterances(total, N, dev)
        host = L.sw_host_alloc(len(mine) * n_s * 2)
        host_np = np.ctypeslib.as_array(C.cast(host, C.POINTER(C.c_int16)), shape=(len(mine), n_s))
        want = []
        for j, i in enumerate(mine):
            host_np[j], ids = window_clip(minfo, i)
            want.append(ids)
        workers.append(dict(dev=dev, eng=eng, params=p, n=len(mine), host=host, want=want,
                            lens=(C.c_int * len(mine))(*([n_s] * len(mine))),
                            ptrs=(ptr16 * len(mine))(*[C.cast(host + j * n_s * 2, ptr16) for j in range(len(mine))]),
                            ok=0, dt=0.0))

    def one_pass(w, check):
        res = w["eng"].full_batch_ptrs(w["ptrs"], w["lens"], w["n"], w["params"])
        for j, r in enumerate(res):
            if check:
                ids = [L.sw_result_token_data(r, s, q).id for s in range(L.sw_result_n_segments(r))
                       for q in range(L.sw_result_n_tokens(r, s))]
                w["ok"] += int(ids == w["want"][j])
            L.sw_result_free(r)

    start = threading.Barrier(N + 1)

    def worker(w, k, check):
        torch.cuda.set_device(w["dev"])
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        start.wait()
        ev0.record()
        for _ in range(k):
            one_pass(w, check)
        ev1.record()
        torch.cuda.synchronize()
        w["dt"] = ev0.elapsed_time(ev1) * 1e-3

    def run(k, check=False):
        th = [threading.Thread(target=worker, args=(w, k, check)) for w in workers]
        for t in th:
            t.start()
        start.wait()
        t0 = time.perf_counter()
        for t in th:
            t.join()
        return time.perf_counter() - t0, max(w["dt"] for w in workers)

    run(1, check=True)
    if args.warmup > 1:
        run(args.warmup - 1)
    clocks = ClockSampler(0)
    clocks.start()
    wall, dt = run(args.steps)
    clk = clocks.stop()
    h2d = sum(w["eng"].stats(reset=True)["h2d_bytes"] for w in workers)
    audio_s = 30.0 * total * args.steps
    line = dict(metric="audio-sec/sec (RTFx)", mode="inproc", value=audio_s / dt, unit="audio-sec/sec", n_gpus=N,
                steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * dt / args.steps,
                host_ms_per_step=1e3 * wall / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="bf16 (f32 accumulate)", data="synthetic",
                timing="CUDA events per device around its K passes, max over devices (host clock: host_ms_per_step)",
                config=dict(workload=cfg["what"] + "; ONE process, %d contexts / host threads (in-process dispatcher), "
                                     "host PCM in pinned memory" % N, model=args.model, windows_per_gpu=W0, batch=args.batch),
                e2e=dict(value=audio_s / dt, unit="audio-sec/sec", h2d_bytes_per_step=int(h2d / (args.steps + args.warmup)),
                         note="inputs are host buffers in this mode: value is end to end"),
                parity_check=dict(windows=total, token_identical_to_expected=sum(w["ok"] for w in workers)),
                clocks=clk)
    print(json.dumps(line), flush=True)
    for w in workers:
        w["eng"].close()
        L.sw_host_free(w["host"])
    return 0


def run_facade(args, path, host_np, offs, n_samp, beam, lang):
    """The reference-facing front door under load (VERDICT r1 weak #8): W caller threads, each handing its own
    clip to SttEngine::transcribe_pcm16 as a pageable std::vector (what the HTTP / gRPC handlers do,
    http_server.cpp:165, grpc_server.cpp:58), parallel_requests = W, batched by the facade's dispatcher.
    Runs host/build/stt_cli in its `bench` mode (separate process: the engine above is closed first)."""
    W = len(n_samp)
    clip = max(n_samp)
    raw = "/tmp/sw_bench_facade_%d.raw" % os.getpid()
    buf = np.zeros((W, clip), np.int16)
    for w in range(W):
        buf[w, : n_samp[w]] = host_np[offs[w]:offs[w + 1]]
    buf.tofile(raw)
    cli = os.path.join(PKG, "host", "build", "stt_cli")
    cmd = [cli, os.path.dirname(path), os.path.basename(path), raw, str(W), str(beam), "bench", "16000",
           "max_batch=%d" % args.batch, "steps=%d" % args.steps, "warmup=1", "clip=%d" % clip,
           "language=%s" % lang, "batch_window_us=20000", "admission=%d" % W]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
        os.unlink(raw)
        if r.returncode != 0:
            return dict(error=(r.stderr or r.stdout)[-300:])
        o = json.loads(r.stdout.strip().splitlines()[-1])
        return dict(value=o["audio_s_per_s"], unit="audio-sec/sec", callers=o["callers"], ms_per_step=o["ms_per_step"],
                    device_passes=o["device_passes"], failures=o["failures"], tokens=o["tokens"],
                    note="SttEngine::transcribe_pcm16 from %d caller threads, pageable std::vector<int16_t> input, "
                         "results as TranscriptionResult vectors incl. prosody + speaker ids; host clock" % W)
    except Exception as ex:  # the facade leg must not take the bench line down
        return dict(error=str(ex)[-300:])


if __name__ == "__main__":
    sys.exit(main())
