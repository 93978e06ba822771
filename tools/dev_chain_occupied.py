"""Development timing (GPU box): what a decoder layer's latency chain (the eleven kernels around the cross
attention) costs when it does NOT have the GPU to itself - which is how it runs under lanes, where the other
lane's cross attention holds 96 SMs and saturates HBM. An occupier kernel (sw_dev_occupy) holds N SMs (shared
memory and register file full, so nothing co-resides) and optionally streams HBM; the step of a large-v3-width
model (64 rows, graph replay, teacher-forced) is timed beside it with SW_SKIP=64 (chain only) and complete.
Per-layer cost = (t_8_layers - t_2_layers) / 6, as in tools/dev_step_time.py."""
import importlib.util, json, os, subprocess, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CASES = [  # (name, n_ctas, smem, stream_bytes)
    ("alone", 0, 0, 0),
    ("96 SMs held", 96, 200 * 1024, 0),
    ("96 SMs held + HBM stream", 96, 200 * 1024, 4 << 30),
    ("74 SMs held", 74, 200 * 1024, 0),
    ("120 SMs held", 120, 200 * 1024, 0),
    ("48 SMs held + HBM stream", 48, 200 * 1024, 4 << 30),
]


def run(swb, size, occ, n=64, n_tok=40):
    from tools import gen_model
    path = "/tmp/sw_%s_s0.bin" % size
    if not os.path.exists(path):
        gen_model.generate(path, size, seed=7)
    eng = swb.Engine(path, max_batch=n, max_beams=1)
    tok = np.random.default_rng(0).integers(0, 50000, size=(n, n_tok)).astype(np.int32)
    eng.decode_logits(tok)
    L = swb.lib()
    name, n_ctas, smem, sbytes = occ
    if n_ctas:
        assert L.sw_dev_occupy(n_ctas, smem, 1.0, sbytes) == 0
        assert L.sw_dev_occupy(0, 0, 0.0, 0) == 0
    eng.stats(reset=True)
    if n_ctas:
        assert L.sw_dev_occupy(n_ctas, smem, 600.0, sbytes) == 0
    eng.decode_logits(tok)
    st = eng.stats(reset=True)
    if n_ctas:
        assert L.sw_dev_occupy(0, 0, 0.0, 0) == 0
    eng.close()
    return st["ms_decode"] / max(1, st["n_steps"])


def one(case_idx):
    import ctypes as C
    spec = importlib.util.spec_from_file_location("sw_binding", os.path.join(ROOT, "sentiric-stt-whisper-service_b200", "sw_binding.py"))
    swb = importlib.util.module_from_spec(spec); spec.loader.exec_module(swb)
    swb.lib().sw_dev_occupy.argtypes = [C.c_int, C.c_int, C.c_float, C.c_size_t]
    occ = CASES[case_idx]
    t8, t2 = run(swb, "large-v3-8l", occ), run(swb, "large-v3-2l", occ)
    per_layer = (t8 - t2) / 6.0
    return dict(case=occ[0], skip=int(os.environ.get("SW_SKIP", "0")), us_per_layer=round(per_layer * 1e3, 2),
                us_fixed=round((t2 - 2 * per_layer) * 1e3, 2))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "--case":
        print(json.dumps(one(int(sys.argv[2]))), flush=True)
    elif len(sys.argv) > 1 and sys.argv[1] == "--kernels":
        # in-chain cost of every kernel beside an occupier that holds 96 SMs
        names = {0: "chain", 1: "layer_norm x3", 2: "qkv gemm", 4: "self attention", 8: "wo gemm", 16: "wxq gemm",
                 32: "reduce q", 256: "wxo gemm", 512: "fc1 gemm", 1024: "fc2 gemm"}
        base = None
        for bit, name in names.items():
            env = dict(os.environ, SW_SKIP=str(64 | bit))
            out = subprocess.run([sys.executable, __file__, "--case", "1"], env=env, capture_output=True, text=True)
            try:
                r = json.loads(out.stdout.strip().splitlines()[-1])
            except Exception:
                print("skip", bit, "FAILED", out.stdout[-300:], out.stderr[-500:], flush=True)
                continue
            if bit == 0:
                base = r["us_per_layer"]
            r.update(kernel=name, in_chain_cost_us=None if base is None else round(base - r["us_per_layer"], 2))
            print(json.dumps(r), flush=True)
    else:
        for ci in range(len(CASES)):
            for skip in ((64, 0, 2047 - 64) if ci == 0 else (64,)):
                env = dict(os.environ, SW_SKIP=str(skip))
                out = subprocess.run([sys.executable, __file__, "--case", str(ci)], env=env, capture_output=True, text=True)
                try:
                    r = json.loads(out.stdout.strip().splitlines()[-1])
                except Exception:
                    print("case", ci, "skip", skip, "FAILED", out.stdout[-300:], out.stderr[-500:], flush=True)
                    continue
                r["what"] = {64: "chain only", 0: "whole layer", 2047 - 64: "cross attention only"}[skip]
                print(json.dumps(r), flush=True)
