"""Kernel-level tests of the attention kernels and the fused LayerNorm of the hot path, each against a float64
reference of the same operation computed from the same bf16 (or f32) inputs, through the C ABI's device-pointer hooks:
encoder self attention (attn_enc_tc.cu: sw_dev_encoder_attention), decoder cross attention + combine (xattn.cu:
sw_dev_cross_attention), paged causal self attention + self-KV append (decode.cu: sw_dev_self_attention) and the
split-K reduce + LayerNorm (elementwise.cu: sw_dev_layer_norm).

The inputs make a wrong key, head, row, page or mask an O(1) error, not a 1e-3 one:
- needles: key entries are +-1 in head dims 0..61 and the query is 8 * K[k*] for a key k* of its own, so k* leads
  every other key by >= 256 in the raw score (> 32 in the exponent) and the output is V[k*]. Every test asserts on
  its own reference that >= 1 - 1e-6 of each such row's mass sits on its needle (or on the keys equal to it).
- pairs: two identical keys in different 128-key tiles, tile halves or cross-attention chunks; the output is the
  mean of their two V rows.
- profiles: a score channel (dim 0) whose per-128-key-tile maxima rise, fall or peak in the middle tile, with scores
  spread over +-60 in log2 units; the rescale of the running maximum carries the result.
- poison: memory a correct kernel loads (or could reach) but must not use holds keys that win the softmax by >= 1000
  raw score, with V = 4: the keys after a window's end, windows no group uses, pool pages of other slots, other
  layers, positions after `pos` and the stale cache copies of positions >= pos0. The offsets sit in the reserved
  head dims 62 and 63 (queries +-32, keys +-64: +-2048 raw score). Where the hardware zero-fills instead (the last
  window of a buffer), every valid key of that window carries a -2048 offset, so a zero key that escaped the mask
  would win.

Tolerances. Encoder and cross attention round P to bf16 before P V (relative error <= 2^-8 per weight, so
<= 2^-8 * sum p|V| / l <= 2 * 2^-9 * Vmax) and round the output to bf16 (half an ulp of |out| <= Vmax: <= 2^-9 Vmax),
where Vmax is the power of two at or above max|V| of the (window, head). The f32 scores, ex2.approx and f32
accumulation add < 1e-4 relative. Bound: 3 * 2^-9 * Vmax per element, and 2^-9 * Vmax on the mean absolute error
(a key leaking with weight 1/1500 on every row, or a biased rescale, moves the mean; rounding does not). The self
attention keeps P in f32: only the output rounding counts, 2^-9 * Vmax (+ 1/16 of that for the f32 sums).
LayerNorm: the updated x is an f32 sum of <= 14 terms (<= n * 2^-24 * sum|terms|); the bf16 output is within one
bf16 rounding (2^-8 |y|) plus the f32 statistics' error, dominated by the mean: 64 * 2^-24 * mean|x| * scale * |g|.
A one-pass variance (E[x^2] - E[x]^2) misses rows of mean 1e3 and standard deviation 1 by percent.
"""
import ctypes
import math

import pytest

pytestmark = pytest.mark.gpu

NEEDLE = 8.0          # query = NEEDLE * K[k*]
TAG_Q, TAG_K = 32.0, 64.0
V_POISON = 4.0
MODES = ["needle", "pair_half", "pair_far", "rise", "fall", "peak", "spread"]
WIDTHS = [(2, 128), (6, 384), (8, 512), (12, 768), (16, 1024), (20, 1280)]  # (n_head, d) of every Whisper size


@pytest.fixture(scope="module")
def lib(swb):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    L = swb.lib()
    vp, ci = ctypes.c_void_p, ctypes.c_int
    L.sw_dev_encoder_attention.argtypes = [vp, vp, ci, ci, ci, ci, vp]
    L.sw_dev_cross_attention_ws_floats.restype = ctypes.c_size_t
    L.sw_dev_cross_attention_ws_floats.argtypes = [ci, ci, ci]
    L.sw_dev_cross_attention.argtypes = [vp, vp, ctypes.c_int64, vp, vp, vp, ci, ci, ci, ci, ci, ci, vp, vp, ci, vp]
    L.sw_dev_self_attention.argtypes = [vp, vp, ci, ci, ci, vp, ci, ci, vp, vp]
    L.sw_dev_layer_norm.argtypes = [vp, ci, ci, vp, vp, vp, vp, ci, vp, vp]
    return L


def pow2_at_least(x):
    return 2.0 ** math.ceil(math.log2(x)) if x > 0 else 1.0


def bf(x):
    return x.bfloat16().float()


def head_content(mode, T, targets, gen, dev):
    """K, V [T][64] and Q [len(targets)][64] of one (window, head), f32 holding bf16 values; dims 62 / 63 are left
    zero for the offsets. targets: each query's needle key (needle and pair modes)."""
    import torch
    n_q = len(targets)
    K = torch.zeros(T, 64, device=dev)
    Q = torch.zeros(n_q, 64, device=dev)
    V = bf(torch.rand(T, 64, generator=gen, device=dev) * 2 - 1)
    if mode in ("needle", "pair_half", "pair_far"):
        K[:, :62] = torch.randint(0, 2, (T, 62), generator=gen, device=dev).float() * 2 - 1
        a = torch.arange(T, device=dev)
        if mode == "pair_half":    # same 128-key tile, other half
            src = a[(a & 64) == 0]
            dst = src | 64
        elif mode == "pair_far":   # different tiles / chunks
            src = a[: T // 2]
            dst = src + T // 2
        if mode != "needle":
            keep = dst < T
            K[dst[keep]] = K[src[keep]]
        Q[:, :62] = NEEDLE * K[targets, :62]
    else:
        tile = torch.arange(T, device=dev) // 128
        nt = int(tile[-1]) + 1
        u = torch.rand(T, generator=gen, device=dev)
        if mode == "rise":
            prof = (tile + u) / nt
        elif mode == "fall":
            prof = (nt - 1 - tile + u) / nt
        elif mode == "peak":
            prof = (nt / 2 - (tile - (nt - 1) / 2).abs() + u) / (nt / 2 + 1)
        else:
            prof = u
        K[:, 0] = 2 * prof - 1
        K[:, 1:62] = torch.randn(T, 61, generator=gen, device=dev) * 0.5
        Q[:, 0] = 200 + 130 * torch.rand(n_q, generator=gen, device=dev)  # x 1/8 x log2(e): up to +-60 in log2 units
        Q[:, 1:62] = torch.randn(n_q, 61, generator=gen, device=dev) * 0.5
    return bf(K), V, bf(Q)


def needle_mass(P, K, targets):
    """Per query: softmax mass on the keys equal to its needle key (dims 0..61). P [n][T] f64, K [T][64]."""
    import torch
    code = K[:, :62].double() @ torch.rand(62, dtype=torch.float64, device=K.device, generator=None)
    eq = code[None, :] == code[targets][:, None]
    return (P * eq).sum(-1)


def check_close(got, ref, V, what):
    """got / ref [n][64] for one head; V: that head's values (its Vmax)."""
    vmax = pow2_at_least(float(V.abs().max()))
    err = (got.double() - ref).abs()
    assert err.max().item() <= 3 * 2 ** -9 * vmax, "%s: max error %.3g (Vmax %g)" % (what, err.max().item(), vmax)
    assert err.mean().item() <= 2 ** -9 * vmax, "%s: mean error %.3g (Vmax %g)" % (what, err.mean().item(), vmax)


def spread_targets(allowed, n, gen):
    """n needle keys covering every allowed key (n >= len(allowed)), in random row order."""
    import torch
    dev = allowed.device
    t = allowed[torch.randperm(len(allowed), generator=gen, device=dev)]
    if n > len(t):
        t = torch.cat([t, allowed[torch.randint(0, len(allowed), (n - len(t),), generator=gen, device=dev)]])
    return t[:n][torch.randperm(n, generator=gen, device=dev)]


# ------------------------------------------------------------------------------------------ encoder attention
ENC_CASES = [(n_win, H, d, 1500) for H, d in WIDTHS for n_win in (1, 3)] + [(2, 6, 384, 1430), (1, 20, 1280, 1430)]


@pytest.mark.parametrize("case", ENC_CASES, ids=lambda c: "win%d_h%d_d%d_T%d" % c)
def test_encoder_attention_matches_float64_reference(lib, case):
    """Window w's last key tile reads n_spill = 128 * ceil(T / 128) - T keys of window w + 1 (poison for w: offset
    +-2048 through dim 63, sign alternating with w, V = 4); the last window's are zero-filled (every valid score of
    that window is offset by -2048 instead). T = 1430 leaves the upper half of the last tile fully masked. Rows after
    n_win * T stay untouched, and a second run gives the same bits."""
    import torch
    n_win, H, d, T = case
    dev = "cuda"
    seed = 1000 * n_win + d + T
    gen = torch.Generator(device=dev).manual_seed(seed)
    n_spill = (T + 127) // 128 * 128 - T
    qkv = torch.zeros(n_win * T, 3 * d, device=dev)
    plan = {}
    for w in range(n_win):
        sigma = 1.0 if w % 2 == 0 else -1.0
        last = w == n_win - 1
        # keys 0..n_spill-1 of a window after the first are the previous window's poison: for this window's own
        # queries they sit 2048 lower (except in the last window, where every key carries the same offset)
        lo = n_spill if (w > 0 and not last) else 0
        allowed = torch.arange(lo, T, device=dev)
        for h in range(H):
            mode = MODES[(w * H + h + seed) % len(MODES)]
            targets = spread_targets(allowed, T, gen)
            K, V, Q = head_content(mode, T, targets, gen, dev)
            Q[:, 63] = sigma * TAG_Q
            if last:
                K[:, 63] = -sigma * TAG_K
            if w > 0:
                K[:n_spill, 63] = -sigma * TAG_K  # attracts window w-1's queries (whose sign is -sigma)
                V[:n_spill] = V_POISON
            rows = slice(w * T, (w + 1) * T)
            qkv[rows, h * 64:(h + 1) * 64] = Q
            qkv[rows, d + h * 64:d + (h + 1) * 64] = K
            qkv[rows, 2 * d + h * 64:2 * d + (h + 1) * 64] = V
            plan[w, h] = (mode, targets)
    qkv = qkv.bfloat16()
    outs = []
    for _ in range(2):
        out = torch.full((n_win * T + 4, d), 1234.0, device=dev, dtype=torch.bfloat16)
        rc = lib.sw_dev_encoder_attention(qkv.data_ptr(), out.data_ptr(), n_win, T, d, H, None)
        assert rc == 0, lib.sw_last_error()
        torch.cuda.synchronize()
        outs.append(out)
    assert torch.equal(outs[0].view(torch.int16), outs[1].view(torch.int16)), "not bit-reproducible"
    out = outs[0]
    assert (out[n_win * T:].float() == 1232.0).all(), "rows after n_win * T were written"  # bf16(1234) = 1232
    for w in range(n_win):
        rows = slice(w * T, (w + 1) * T)
        Qw = qkv[rows, :d].double().view(T, H, 64).transpose(0, 1)
        Kw = qkv[rows, d:2 * d].double().view(T, H, 64).transpose(0, 1)
        Vw = qkv[rows, 2 * d:].double().view(T, H, 64).transpose(0, 1)
        P = torch.softmax(Qw @ Kw.transpose(1, 2) / 8.0, dim=-1)
        ref = P @ Vw
        got = out[rows].view(T, H, 64).transpose(0, 1)
        for h in range(H):
            mode, targets = plan[w, h]
            if mode in ("needle", "pair_half", "pair_far"):
                mass = needle_mass(P[h], Kw[h], targets)
                assert mass.min().item() >= 1 - 1e-6, (w, h, mode, mass.min().item())
            check_close(got[h], ref[h], Vw[h], "window %d head %d (%s)" % (w, h, mode))


# ------------------------------------------------------------------------------------------ cross attention
# name, T, max_batch (windows in the buffer), rows per group, max_ctas
XA_CONFIGS = [
    ("b8", 1500, 8, [3, 1, 8, 5, 2, 7], 0),
    ("b8_ctas1", 1500, 8, [8, 2, 5, 1], 1),
    ("b8_ctas7", 1500, 8, [4, 8, 1, 6, 3], 7),
    ("b8_ctas37", 1500, 8, [2, 7, 8, 1, 5, 3, 6], 37),
    ("T45", 45, 6, [2, 8, 1, 4], 0),
    ("b64x5", 1500, 64, [5] * 64, 0),
]


@pytest.mark.parametrize("cfg", XA_CONFIGS, ids=lambda c: c[0])
@pytest.mark.parametrize("width", WIDTHS, ids=lambda w: "h%d_d%d" % w)
def test_cross_attention_matches_float64_reference(lib, width, cfg):
    """Groups of 1..8 decoder rows, each row and head with its own needle; grp_win permuted over a buffer of
    max_batch windows whose last window is in use. Windows no group uses hold poison (offset +2048 through dim 62
    for every query). The 16-key stage after key T - 1 reads n_spill keys of the next window: poison through dim 63
    (sign alternating with the window) or zero-filled past the buffer's end (every valid score of the last window
    offset by -2048). max_ctas 1 / 7 / 37 make CTAs walk many items (ring phase wrap, next item's Q prefetched).
    The widths cover 1 and 2 heads per warp, the half-head split of d = 1280 and ring depths 3 to 8."""
    import torch
    H, d = width
    name, T, max_batch, counts, max_ctas = cfg
    dev = "cuda"
    seed = d + 7 * T + 131 * len(counts) + max_ctas
    gen = torch.Generator(device=dev).manual_seed(seed)
    G, R = len(counts), sum(counts)
    starts = [sum(counts[:g]) for g in range(G)]
    n_spill = (T + 15) // 16 * 16 - T
    used = sorted(torch.randperm(max_batch - 1, generator=gen, device=dev)[:G - 1].tolist() + [max_batch - 1])
    wins = [used[i] for i in torch.randperm(G, generator=gen, device=dev).tolist()]
    used = set(used)
    # needle keys: the first, middle and last key of every 16-key stage (so of every chunk of any plan), and 0 / T-1
    stage_keys = sorted(set(k for s in range(0, T, 16) for k in (s, s + 8, min(s + 15, T - 1)) if k < T))
    kv = torch.zeros(max_batch * T, 2 * d, device=dev)
    q = torch.zeros(R, d, device=dev)
    for w in range(max_batch):
        if w in used:
            continue
        rows = slice(w * T, (w + 1) * T)
        kv[rows, :d] = (torch.randint(0, 2, (T, d), generator=gen, device=dev).float() * 2 - 1)
        kv[rows, :d].view(T, H, 64)[:, :, 62:] = 0
        kv[rows, :d].view(T, H, 64)[:, :, 62] = TAG_K
        kv[rows, d:] = V_POISON
    plan = {}
    for g in range(G):
        w, cnt, r0 = wins[g], counts[g], starts[g]
        sigma = 1.0 if w % 2 == 0 else -1.0
        last = w == max_batch - 1
        prev_used = w > 0 and (w - 1) in used
        lo = n_spill if (prev_used and not last) else 0
        cover = torch.tensor([k for k in stage_keys if k >= lo], device=dev)
        rows = slice(w * T, (w + 1) * T)
        for h in range(H):
            mode = MODES[(g * H + h + seed) % len(MODES)]
            first = ((g * H + h) * 8) % len(cover)
            targets = cover[(first + torch.arange(cnt, device=dev)) % len(cover)]  # distinct within the group
            K, V, Q = head_content(mode, T, targets, gen, dev)
            Q[:, 62] = TAG_Q
            Q[:, 63] = sigma * TAG_Q
            if last:
                K[:, 63] = -sigma * TAG_K
            if prev_used:
                K[:n_spill, 63] = -sigma * TAG_K  # attracts window w-1's queries
                V[:n_spill] = V_POISON
            kv[rows, h * 64:(h + 1) * 64] = K
            kv[rows, d + h * 64:d + (h + 1) * 64] = V
            q[r0:r0 + cnt, h * 64:(h + 1) * 64] = Q
            plan[g, h] = (mode, targets)
    kv, q = kv.bfloat16(), q.bfloat16()
    grp_win = torch.tensor(wins, dtype=torch.int32, device=dev)
    grp_start = torch.tensor(starts, dtype=torch.int32, device=dev)
    grp_count = torch.tensor(counts, dtype=torch.int32, device=dev)
    ws = torch.empty(lib.sw_dev_cross_attention_ws_floats(R, d, H), device=dev)
    outs = []
    for _ in range(2):
        out = torch.full((R + 2, d), 1234.0, device=dev, dtype=torch.bfloat16)
        ws.fill_(float("nan"))
        rc = lib.sw_dev_cross_attention(q.data_ptr(), kv.data_ptr(), max_batch * T, grp_win.data_ptr(),
                                        grp_start.data_ptr(), grp_count.data_ptr(), G, max(counts), R, T, d, H,
                                        ws.data_ptr(), out.data_ptr(), max_ctas, None)
        assert rc == 0, lib.sw_last_error()
        torch.cuda.synchronize()
        outs.append(out)
    assert torch.equal(outs[0].view(torch.int16), outs[1].view(torch.int16)), "not bit-reproducible"
    out = outs[0]
    assert (out[R:].float() == 1232.0).all(), "rows after R were written"
    for g in range(G):
        w, cnt, r0 = wins[g], counts[g], starts[g]
        Kg = kv[w * T:(w + 1) * T, :d].double().view(T, H, 64).transpose(0, 1)
        Vg = kv[w * T:(w + 1) * T, d:].double().view(T, H, 64).transpose(0, 1)
        Qg = q[r0:r0 + cnt].double().view(cnt, H, 64).transpose(0, 1)
        P = torch.softmax(Qg @ Kg.transpose(1, 2) / 8.0, dim=-1)
        ref = P @ Vg
        got = out[r0:r0 + cnt].view(cnt, H, 64).transpose(0, 1)
        for h in range(H):
            mode, targets = plan[g, h]
            if mode in ("needle", "pair_half", "pair_far"):
                mass = needle_mass(P[h], Kg[h], targets)
                assert mass.min().item() >= 1 - 1e-6, (g, h, mode, mass.min().item())
            check_close(got[h], ref[h], Vg[h], "group %d (window %d) head %d (%s)" % (g, w, h, mode))


# ------------------------------------------------------------------------------------------ self attention
KV_PAGE, KV_MAX_PAGES = 32, 14
# per slot: (pos0, pos, flat). Rows pos0..pos of the slot are consecutive rows of the step.
SA_SLOTS = [(p, p, False) for p in (0, 31, 32, 63, 64, 127, 128, 447)] + [
    (29, 34, False),     # several rows of one slot across a page boundary
    (120, 130, False),   # ... across the 128 keys of the first load
    (440, 447, False),
    (0, 4, False),       # a whole prompt in the step
    (0, 40, False),
    (3, 3, True),        # Q = 0: the output is the mean of exactly pos + 1 values
    (0, 6, True),
    (30, 33, True),
]


@pytest.mark.parametrize("layer", [0, 3])
@pytest.mark.parametrize("width", [(6, 384), (20, 1280)], ids=lambda w: "h%d_d%d" % w)
def test_self_attention_matches_float64_reference(lib, width, layer):
    """Causal self attention over the paged self-KV (pool [page][n_layer = 4][2][32][d]) with pages scattered and
    permuted. Cache positions < pos0 of the slot hold its keys in `layer`; everything else in the pool is poison
    (offset +2048 through dim 62, V = 4): other layers of the same pages, positions >= pos0 (which must come from
    qkv rows r - (pos - k)), other slots' pages. After the call the pool equals its previous contents except the
    appended K / V slices, which equal the qkv K / V bit for bit."""
    import torch
    H, d = width
    n_layer = 4
    dev = "cuda"
    gen = torch.Generator(device=dev).manual_seed(17 * d + layer)
    n_slots = len(SA_SLOTS)
    n_pages = n_slots * KV_MAX_PAGES + 9
    page_of = torch.randperm(n_pages, generator=gen, device=dev)[:n_slots * KV_MAX_PAGES].view(n_slots, KV_MAX_PAGES)
    pool = torch.zeros(n_pages, n_layer, 2, KV_PAGE, d, device=dev)
    pk = pool[:, :, 0].view(n_pages, n_layer, KV_PAGE, H, 64)
    pk[..., :62] = torch.randint(0, 2, pk[..., :62].shape, generator=gen, device=dev).float() * 2 - 1
    pk[..., 62] = TAG_K
    pool[:, :, 1] = V_POISON
    R = sum(p - p0 + 1 for p0, p, _ in SA_SLOTS)
    qkv = torch.zeros(R, 3 * d, device=dev)
    rows = torch.zeros(R, 20, dtype=torch.int32)
    keys, vals, plan = {}, {}, []
    r = 0
    for s, (pos0, pos, flat) in enumerate(SA_SLOTS):
        Ks = torch.randint(0, 2, (pos + 1, H, 64), generator=gen, device=dev).float() * 2 - 1
        Ks[..., 62:] = 0
        Vs = bf(torch.rand(pos + 1, H, 64, generator=gen, device=dev) * 2 - 1)
        keys[s], vals[s] = Ks, Vs
        for k in range(pos0):  # the cache of this slot, in `layer`
            pool[page_of[s, k // KV_PAGE], layer, 0, k % KV_PAGE] = Ks[k].reshape(d)
            pool[page_of[s, k // KV_PAGE], layer, 1, k % KV_PAGE] = Vs[k].reshape(d)
        for p in range(pos0, pos + 1):
            qkv[r, d:2 * d] = Ks[p].reshape(d)
            qkv[r, 2 * d:] = Vs[p].reshape(d)
            cand = sorted(set(k for k in (0, 31, 32, 63, 64, 127, 128, 447, p, p - 1, pos0, pos0 - 1, p // 2)
                              if 0 <= k <= p))
            tg = []
            for h in range(H):
                if flat:
                    continue  # Q = 0
                if h % 4 == 3:  # spread scores
                    qkv[r, h * 64:h * 64 + 62] = torch.randn(62, generator=gen, device=dev) * 3
                else:
                    k = cand[(h + r) % len(cand)]
                    tg.append((h, k))
                    qkv[r, h * 64:h * 64 + 62] = NEEDLE * Ks[k, h, :62]
                qkv[r, h * 64 + 62] = TAG_Q
            rows[r, :4] = torch.tensor([s, p, 0, pos0], dtype=torch.int32)
            rows[r, 4:4 + KV_MAX_PAGES] = page_of[s].int().cpu()
            plan.append((s, p, flat, tg))
            r += 1
    qkv, pool = qkv.bfloat16(), pool.bfloat16()
    d_rows = rows.to(dev)
    before = pool.clone()
    out = torch.full((R + 1, d), 1234.0, device=dev, dtype=torch.bfloat16)
    rc = lib.sw_dev_self_attention(qkv.data_ptr(), d_rows.data_ptr(), R, d, H, pool.data_ptr(), layer, n_layer,
                                   out.data_ptr(), None)
    assert rc == 0, lib.sw_last_error()
    torch.cuda.synchronize()
    assert (out[R].float() == 1232.0).all(), "row R was written"
    want = before.clone()
    for r, (s, p, _, _) in enumerate(plan):
        want[page_of[s, p // KV_PAGE], layer, 0, p % KV_PAGE] = qkv[r, d:2 * d]
        want[page_of[s, p // KV_PAGE], layer, 1, p % KV_PAGE] = qkv[r, 2 * d:]
    assert torch.equal(pool.view(torch.int16), want.view(torch.int16)), "the pool changed beyond the appended slices"
    qd = qkv.double()
    for r, (s, p, flat, tg) in enumerate(plan):
        Kr = bf(keys[s][:p + 1]).double().transpose(0, 1)  # [H][p + 1][64]
        Vr = vals[s][:p + 1].double().transpose(0, 1)
        Qr = qd[r, :d].view(H, 1, 64)
        P = torch.softmax(Qr @ Kr.transpose(1, 2) / 8.0, dim=-1)  # [H][1][p + 1]
        ref = (P @ Vr)[:, 0]
        if flat:
            assert torch.allclose(ref, Vr.mean(1), rtol=0, atol=1e-12)
        for h, k in tg:
            assert P[h, 0, k].item() >= 1 - 1e-6, (r, h, k, P[h, 0, k].item())
        got = out[r].view(H, 64).double()
        for h in range(H):
            vmax = pow2_at_least(float(Vr[h].abs().max()))
            err = (got[h] - ref[h]).abs().max().item()
            assert err <= 2 ** -9 * vmax * (1 + 1 / 16), "slot %d pos %d head %d: error %.3g" % (s, p, h, err)


# ------------------------------------------------------------------------------------------ LayerNorm
LN_SPLITS = [(0, False)] + [(s, b) for s in (1, 5, 8, 9, 12) for b in (False, True)]


@pytest.mark.parametrize("rows", [1, 7, 64, 320, 2048, 2049, 3001])
@pytest.mark.parametrize("d", [128, 384, 512, 768, 1024, 1280, 1536])
def test_layer_norm_matches_float64_reference(lib, d, rows):
    """rows <= 2048: one CTA per row (n_split > 8 takes the row kernel's tail loop); rows > 2048: a warp per row,
    with a rows % 4 tail. Rows of three kinds: N(0, 2), mean 1e3 with standard deviation 1, and constant (output
    exactly b). n_split = 0 passes no partials: x must not change at all."""
    import torch
    dev = "cuda"
    gen = torch.Generator(device=dev).manual_seed(d * 7 + rows)
    kind = torch.arange(rows, device=dev) % 5
    base = torch.randn(rows, d, generator=gen, device=dev) * 2
    base[kind == 1] = 1e3 + torch.randn(int((kind == 1).sum()), d, generator=gen, device=dev)
    base[kind == 3] = 3.0
    g = 1 + 0.2 * torch.randn(d, generator=gen, device=dev)
    b = 0.5 * torch.randn(d, generator=gen, device=dev)
    for n_split, with_bias in LN_SPLITS:
        x = torch.full((rows + 1, d), 77.0, device=dev)
        x[:rows] = base
        part = torch.randn(max(n_split, 1), rows, d, generator=gen, device=dev) * 0.3
        part[:, kind == 3] = 0.0
        bias = 0.3 * torch.randn(d, generator=gen, device=dev) if with_bias else None
        x0 = x.clone()
        out = torch.full((rows + 1, d), 1234.0, device=dev, dtype=torch.bfloat16)
        rc = lib.sw_dev_layer_norm(x.data_ptr(), rows, d, g.data_ptr(), b.data_ptr(), out.data_ptr(),
                                   part.data_ptr() if n_split else None, n_split,
                                   bias.data_ptr() if bias is not None else None, None)
        assert rc == 0, lib.sw_last_error()
        torch.cuda.synchronize()
        what = "n_split %d bias %d" % (n_split, with_bias)
        assert torch.equal(x[rows], x0[rows]) and (out[rows].float() == 1232.0).all(), what + ": row `rows` written"
        if n_split == 0:
            assert torch.equal(x.view(torch.int32), x0.view(torch.int32)), what + ": x changed without partials"
            xr = x0[:rows].double()
        else:
            terms = [x0[:rows].double()] + ([bias.double().expand(rows, d)] if with_bias else []) + \
                [part[s].double() for s in range(n_split)]
            xr = sum(terms)
            bound = len(terms) * 2 ** -24 * sum(t.abs() for t in terms)
            err = (x[:rows].double() - xr).abs()
            assert (err <= bound).all(), what + ": x + partials off by %.3g" % err.max().item()
        xk = x[:rows].double()  # what the kernel normalised
        mean = xk.mean(1, keepdim=True)
        scale = 1.0 / torch.sqrt(((xk - mean) ** 2).mean(1, keepdim=True) + 1e-5)
        y = (xk - mean) * scale * g.double() + b.double()
        tol = (2 ** -8 * y.abs() + 64 * 2 ** -24 * xk.abs().mean(1, keepdim=True) * scale * g.double().abs()
               + 2 ** -16 * (y - b.double()).abs() + 1e-6)
        err = (out[:rows].double() - y).abs()
        assert (err <= tol).all(), what + ": LayerNorm off by %.3g (row %d)" % (
            err.max().item(), int((err - tol).max(1).values.argmax()))
        if not with_bias and rows > 3:
            assert torch.equal(out[3].float(), bf(b)), what + ": constant row is not b"
