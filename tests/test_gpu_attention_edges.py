"""The flash-attention kernels of KD on the paths that random activations never reach: late row maxima, peaky and
one-hot rows, logits far below or far above zero, tile and key-range edges, every head_dim.

Probes.  `ops.cross_attention` with w_q = I_C, w_kv = I_2C (ctx = [K | V]), w_o = I_C and no bias feeds the flash
kernel chosen q, k, v exactly: every projection output is one product per fp32 accumulator, so the fp16 result IS the
attention output o.  `ops.attention` (the self-attention entry, L queries = L keys, the fused QKV epilogue, PnP's
shared_qk) is probed with block-permutation weights: head h takes q from x's head-block h, k from block (h+1) mod H and
v from block (h+2) mod H, so that head 0 sees a designed (q, k, v) and the other heads see the same blocks in other
roles.

Model.  The kernels work in log2 units with c32 = fp32(fp32(scale) * fp32(log2 e)).  On the embedded-reference path
(head_dim % 16 == 8, VTM_FA_EMBED not 0, grouped kernel off) the projection epilogue stores q' = fp16(fp32(q) * c32)
and the logits are t = q' . k; on every other path t = (q . k) * c32.  The reference is o = sum_j softmax2(t)_j v_j in
float64 on the device.

Bound.  o is a convex combination of the v rows, so every error source that is relative to the weights is bounded by
the same fraction of max_j |v_j|:  P is stored as fp16 for the numerator while the denominator is either the same fp16
P (head_dim % 16 == 8) or the fp32 P (2 x 2^-11);  the polynomial exp2 has a relative error of 7.5e-5;  o is rounded
to fp16 (2^-11).  That is 1.54e-3; fp32 accumulation of logits up to |t| = 4096 adds < 2e-4.  So each row must satisfy
    max_e |o_ie - ref_ie|  <=  2e-3 * max_j |v_j|_inf      (over the head's keys; no absolute term).

Envelope.  |q'| < 6e4 (fp16 range after the scale is folded in) and |t| <= 4096 log2 units (the reference maximum stays
an fp16 number and fp32 keeps 12 fractional bits of it).  Every scenario asserts it.

Scenarios (each asserts its own precondition on the fp64 model logits first, so that it cannot degrade into the
benign case):
  S1 benign      std(t) ~ 1.5: what random activations give
  S2 peaky       std(t) ~ 8: the reference moves in early tiles
  S3 ramp        t_j ~ 0.19 j (+ noise 0.3): the row maximum rises by > 9 on every 64- and 96-key tile, so the
                 reference moves, O is rescaled and (embedded path) the reference is republished on every tile
  S4 late spike  the row maximum is one key (by default the last), above everything else by 8 - 2^-6, 8 or 8 + 2^-6:
                 both sides of the 2^8 rescale threshold, in the masked last tile
  S5 one-hot     per row one target key (key 0, the last key, both sides of tile boundaries, random ones) at least 40
                 above every other key, |t| <= 2048: o must be v_target bit for bit
  S6 deep        6 of 7 keys 150 - 220 below the other keys, at least 130 below the row maximum: the polynomial's clamp and ex2's flush to zero
  S7 offset      all logits shifted by +100 or +1000 through a shared component: a large fp16 reference and
                 cancellation in the QK accumulator
  S8 uniform     identical keys: o = mean(v)
With a single key (Lk = 1) o must be v bit for bit in every scenario.
"""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

LOG2E = 1.4426950408889634
TOL = 2e-3
Q_MAX = 6e4
T_MAX = 4096.0
RAMP = 0.19                    # log2 units per key: 12.2 per 64-key tile, 18.2 per 96-key tile
GAP = 8.0                      # the kernels' RESCALE_LOG2
HEAD_DIMS = tuple(range(8, 129, 8))
S4_GAPS = (GAP - 2.0 ** -6, GAP, GAP + 2.0 ** -6)
VARIANTS = {"S1": ({},), "S2": ({},), "S3": ({},), "S4": tuple({"gap": g} for g in S4_GAPS), "S5": ({},),
            "S6": ({},), "S7": ({"offset": 100.0}, {"offset": 1000.0}), "S8": ({},)}
LK_EDGES = (1, 2, 63, 64, 65, 77, 95, 96, 97, 129, 191, 193, 1000)
LQ_EDGES = (1, 127, 128, 129, 300)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def c32(scale):
    return float(np.float32(np.float32(scale) * np.float32(LOG2E)))


def embedded(d, env=None):
    """Whether the flash kernel runs the embedded-reference path for head_dim d in a process with environment `env`."""
    env = os.environ if env is None else env
    return d % 16 == 8 and env.get("VTM_FA_EMBED", "1")[:1] != "0" and env.get("VTM_FA_GROUPS", "")[:1] != "1"


def q_eff(q, scale, emb):
    if not emb:
        return q.double()
    return (q.float() * torch.tensor(c32(scale), dtype=torch.float32, device=q.device)).half().double()


def model_logits(q, k, scale, emb):
    """fp64 logits (log2 units) that the kernel is specified to exponentiate: [..., Lq, Lk]."""
    t = q_eff(q, scale, emb) @ k.double().transpose(-1, -2)
    return t if emb else t * c32(scale)


def softmax2_apply(t, v):
    p = torch.exp2(t - t.amax(-1, keepdim=True))
    return (p @ v.double()) / p.sum(-1, keepdim=True)


def m_eff(a, scale, emb):
    """Logit contribution per unit of k of a q column that holds the constant a."""
    if emb:
        return float(np.float16(np.float32(a) * np.float32(c32(scale))))
    return float(np.float16(a)) * c32(scale)


# ------------------------------------------------------------------------------------------------ scenario builders
def make_scenario(name, G, Lq, Lk, d, scale, emb, seed, gap=GAP, offset=0.0, spike=None):
    """fp16 q [G, Lq, d], k [G, Lk, d], v [G, Lk, d] on the CPU, and a dict with what the scenario promises."""
    g = torch.Generator().manual_seed(seed)
    rn = lambda *s: torch.randn(s, generator=g, dtype=torch.float64)
    c = c32(scale)
    q = torch.zeros(G, Lq, d, dtype=torch.float64)
    k = torch.zeros(G, Lk, d, dtype=torch.float64)
    v = rn(G, Lk, d)
    info = {}

    def noise(sigma, c0):       # q, k columns c0.. with a logit contribution of std ~ sigma
        n = d - c0
        q[..., c0:] = rn(G, Lq, n) * (sigma / (c * math.sqrt(n)))
        k[..., c0:] = rn(G, Lk, n)

    if name in ("S1", "S2", "S8"):
        noise(8.0 if name == "S2" else 1.5, 0)
        if name == "S8":
            k[:] = k[:, :1]
    elif name == "S7":
        noise(1.5, 1)
        q[..., 0] = 1.0
        k[..., 0] = offset / m_eff(1.0, scale, emb)
    elif name == "S3":
        noise(0.3, 1)
        q[..., 0] = 16.0
        k[..., 0] = (RAMP * torch.arange(Lk, dtype=torch.float64) / m_eff(16.0, scale, emb))
    elif name == "S4":
        # background in column 0 (its maximum bmax sits at key `bm`; a power of two, so the fp16 reference the embedded
        # path keeps is exact), the spike in columns 1 + 2 (hi + lo fp16 parts: ~22 bits for the gap)
        me = m_eff(1.0, scale, emb)
        spike = Lk - 1 if spike is None else spike
        bm = 0 if spike != 0 else Lk - 1
        bmax = 2.0 ** math.ceil(math.log2(4.5 / me))
        b = (rn(G, Lk) * (1.5 / me)).clamp(-3 * bmax, 0.9 * bmax)
        b[:, bm] = bmax
        b[:, spike] = 0.0
        q[..., 0:3] = 1.0
        k[..., 0] = b
        amp = bmax + gap / me
        hi = float(np.float16(amp))
        lo = float(np.float16(amp - hi))
        k[:, spike, 1] = hi
        k[:, spike, 2] = lo
        info.update(spike=spike, gap=gap)
    elif name == "S5":
        # distinct +-1 codes on dc = min(d, 16) columns for the target keys, zero elsewhere; q = alpha * its target's
        # code: t = 24 dc at the target, <= 24 (dc - 2) at any other target, 0 at the rest
        dc = min(d, 16)
        alpha = 24.0 / c
        nt = max(1, min(Lk, Lq, 2 ** dc))
        special = []
        for p in (0, Lk - 1, 63, 64, 95, 96, 127, 128, 191, 192):
            if p < Lk and p not in special:
                special.append(p)
        tgt = torch.empty(G, Lq, dtype=torch.long)
        for gi in range(G):
            rest = [int(p) for p in torch.randperm(Lk, generator=g) if int(p) not in special]
            pos = (special + rest)[:nt]
            codes = torch.randperm(2 ** dc, generator=g)[:nt]
            bits = ((codes[:, None] >> torch.arange(dc)) & 1).double() * 2 - 1
            k[gi, pos, :dc] = bits
            which = torch.arange(Lq) % nt
            which = which[torch.randperm(Lq, generator=g)] if Lq > nt else which
            q[gi, :, :dc] = alpha * bits[which]
            tgt[gi] = torch.tensor(pos)[which]
        v = torch.sign(rn(G, Lk, d)) * torch.exp2(4 * torch.rand((G, Lk, d), generator=g, dtype=torch.float64) - 2)
        info.update(target=tgt)
    elif name == "S6":
        noise(1.5, 1)
        me = m_eff(1.0, scale, emb)
        q[..., 0] = 1.0
        deep = torch.arange(Lk) % 7 != 0
        depth = 150 + 70 * torch.rand((G, Lk), generator=g, dtype=torch.float64)
        k[..., 0] = torch.where(deep, -depth / me, torch.zeros_like(depth))
    else:
        raise ValueError(name)
    q, k, v = q.half(), k.half(), v.half()
    assert torch.isfinite(q).all() and torch.isfinite(k).all() and torch.isfinite(v).all()
    return q, k, v, info


def check_scenario(name, q, k, scale, emb, info, gap=GAP, offset=0.0, spike=None):
    """Assert the scenario's precondition and the envelope on the fp64 model logits; returns them."""
    assert q_eff(q, scale, emb).abs().max().item() < Q_MAX
    t = model_logits(q, k, scale, emb)
    assert t.abs().max().item() <= T_MAX, t.abs().max().item()
    Lk = t.shape[-1]
    big = t.numel() >= 512 and Lk >= 32      # enough keys for a standard deviation to mean something
    if name in ("S1", "S2", "S7") and big:
        lo, hi = (6.0, 10.0) if name == "S2" else (1.0, 2.2)
        tt = t - offset if name == "S7" else t
        assert lo <= tt.std().item() <= hi, (name, tt.std().item())
        if name == "S7":
            assert abs(tt.mean().item()) < 1.0, tt.mean().item()     # k's fp16 rounding of the offset
    if name == "S3":
        for bkv in (64, 96):
            for j in range(1, Lk // bkv):
                rise = t[..., j * bkv:(j + 1) * bkv].amax(-1) - t[..., :j * bkv].amax(-1)
                assert rise.min().item() > 9.0 and rise.max().item() < 24.0, (bkv, j, rise.min().item())
    if name == "S4" and Lk >= 2:
        top2 = t.topk(2, dim=-1)
        assert (top2.indices[..., 0] == info["spike"]).all()
        assert (top2.values[..., 0] - top2.values[..., 1] - gap).abs().max().item() <= 2.0 ** -10
    if name == "S5":
        top2 = t.topk(min(2, Lk), dim=-1)
        assert (top2.indices[..., 0] == info["target"].to(t.device)).all()
        if Lk >= 2:
            assert (top2.values[..., 0] - top2.values[..., 1]).min().item() >= 40.0
        assert t.abs().max().item() <= 2048.0
    if name == "S6" and Lk >= 7:
        deep = (t <= t.amax(-1, keepdim=True) - 130.0).double().mean(-1)
        assert deep.min().item() >= 0.75, deep.min().item()
    if name == "S8":
        assert (t.amax(-1) == t.amin(-1)).all()
    return t


# ------------------------------------------------------------------------------------------------ probes
def cross_probe(q, k, v, scale):
    """o [B, H, Lq, d] of the flash kernel for q [B, H, Lq, d], k / v [B, H, Lk, d] (fp16, CUDA)."""
    from vidtome_b200 import ops
    B, H, Lq, d = q.shape
    Lk, C = k.shape[2], H * d
    x = q.transpose(1, 2).reshape(B, Lq, C).contiguous()
    ctx = torch.cat([k.transpose(1, 2).reshape(B, Lk, C), v.transpose(1, 2).reshape(B, Lk, C)], -1).contiguous()
    eye = torch.eye(C, device=q.device, dtype=torch.float16)
    eye2 = torch.eye(2 * C, device=q.device, dtype=torch.float16)
    y = ops.cross_attention(x, ctx, eye, eye2, eye, None, H, scale)
    return y.view(B, Lq, H, d).transpose(1, 2)


def self_probe_qkv(x, H):
    """The per-head q, k, v [B, H, L, d] that the block-permutation weights make of x [B, L, H*d]."""
    B, L, C = x.shape
    blocks = x.view(B, L, H, C // H).transpose(1, 2)
    return blocks, blocks.roll(-1, 1), blocks.roll(-2, 1)


def self_probe(x, H, scale, shared_qk=False):
    from vidtome_b200 import ops
    C = x.shape[-1]
    d = C // H
    eye = torch.eye(C, device=x.device, dtype=torch.float16)
    w_qkv = torch.cat([eye, eye.roll(d, 1), eye.roll(2 * d, 1)], 0).contiguous()
    y = ops.attention(x, w_qkv, eye, None, H, scale, shared_qk=shared_qk)
    return y.view(x.shape[0], x.shape[1], H, d).transpose(1, 2)


def row_ratio(o, ref, v):
    """max_e |o - ref| per row over max_j |v_j|_inf of the row's head: [..., Lq]."""
    vmax = v.abs().amax(dim=(-2, -1)).double()
    return (o.double() - ref).abs().amax(-1) / vmax[..., None]


def run_cross_case(name, B, H, Lq, Lk, d, seed, kw, env=None):
    """One cross-probe case; returns (max error ratio, list of failures)."""
    scale = d ** -0.5
    emb = embedded(d, env)
    q, k, v, info = make_scenario(name, B * H, Lq, Lk, d, scale, emb, seed, **kw)
    q, k, v = [t.view(B, H, *t.shape[1:]).cuda() for t in (q, k, v)]
    if "target" in info:
        info["target"] = info["target"].view(B, H, Lq)
    t = check_scenario(name, q, k, scale, emb, info, **kw)
    o = cross_probe(q, k, v, scale)
    torch.cuda.synchronize()
    ref = softmax2_apply(t, v)
    ratio = row_ratio(o, ref, v)
    tag = f"{name}{kw} d={d} Lq={Lq} Lk={Lk}"
    bad = []
    if not torch.isfinite(o).all():
        bad.append(f"{tag}: non-finite output")
    r = ratio.max().item()
    if not r <= TOL:
        bad.append(f"{tag}: error {r:.3e} x max|v| > {TOL}")
    if name == "S5":
        want = torch.gather(v, 2, info["target"].cuda()[..., None].expand(-1, -1, -1, d))
        n = (o != want).any(-1).sum().item()
        if n:
            bad.append(f"{tag}: {n} one-hot rows are not v_target bit for bit")
    if Lk == 1 and not torch.equal(o, v.expand_as(o)):
        bad.append(f"{tag}: a single key does not give o == v")
    return r, bad


def run_cross_cases(cases, env=None):
    worst, bad = {}, []
    for name, B, H, Lq, Lk, d, seed, kw in cases:
        r, b = run_cross_case(name, B, H, Lq, Lk, d, seed, kw, env)
        key = name + ("" if not kw else "/" + ",".join(f"{a}={kw[a]:g}" for a in kw))
        worst[key] = max(worst.get(key, 0.0), r)
        bad += b
    return worst, bad


def _report(label, worst):
    print(f"\nEDGES {label} " + json.dumps({k: float(f"{w:.3e}") for k, w in worst.items()}))


# ------------------------------------------------------------------------------------------------ CPU: the builders
def _cpu_cases():
    for name, kws in VARIANTS.items():
        for kw in kws:
            for d in (8, 40, 64, 80, 128):
                for Lq, Lk in ((129, 1000), (1, 1), (127, 2), (128, 97), (300, 193)):
                    yield name, kw, d, Lq, Lk


@pytest.mark.parametrize("name", list(VARIANTS))
@pytest.mark.parametrize("emb", [False, True])
def test_scenario_builders_meet_their_preconditions(name, emb):
    """Every generator meets its precondition (and the envelope) for every parametrisation the GPU cases use, on both
    logit models: a failure on the GPU then means the kernel, not the test data."""
    for _, kw, d, Lq, Lk in (c for c in _cpu_cases() if c[0] == name):
        scale = d ** -0.5
        q, k, v, info = make_scenario(name, 2, Lq, Lk, d, scale, emb, seed=Lk * 131 + d, **kw)
        check_scenario(name, q, k, scale, emb, info, **kw)


def test_ramp_moves_the_maximum_on_every_tile():
    q, k, _, _ = make_scenario("S3", 2, 64, 10241, 40, 40 ** -0.5, True, seed=1)
    t = model_logits(q, k, 40 ** -0.5, True)
    for bkv in (64, 96):
        tiles = t[..., :(t.shape[-1] // bkv) * bkv].unflatten(-1, (-1, bkv)).amax(-1)
        assert (tiles.diff(dim=-1) > 9.0).all()
    assert t.abs().max().item() <= T_MAX


def test_one_hot_gaps_and_positions():
    for d in (8, 16, 40):
        q, k, _, info = make_scenario("S5", 3, 300, 193, d, d ** -0.5, False, seed=d)
        t = model_logits(q, k, d ** -0.5, False)
        top2 = t.topk(2, dim=-1)
        assert (top2.indices[..., 0] == info["target"]).all()
        assert (top2.values[..., 0] - top2.values[..., 1]).min().item() >= 40.0
        used = set(info["target"].flatten().tolist())
        assert {0, 63, 64, 95, 96, 127, 128, 191, 192} <= used


def test_offsets_and_spike_gaps_are_what_they_claim():
    for emb in (False, True):
        for off in (100.0, 1000.0):
            q, k, _, _ = make_scenario("S7", 2, 128, 500, 40, 40 ** -0.5, emb, seed=3, offset=off)
            t = model_logits(q, k, 40 ** -0.5, emb)
            assert abs(t.mean().item() - off) < 1.0
        for gap in S4_GAPS:
            q, k, _, _ = make_scenario("S4", 2, 16, 193, 40, 40 ** -0.5, emb, seed=4, gap=gap)
            top2 = model_logits(q, k, 40 ** -0.5, emb).topk(2, dim=-1).values
            assert ((top2[..., 0] - top2[..., 1]) - gap).abs().max().item() <= 2.0 ** -10


def test_embedded_model_rounds_q_like_the_projection_epilogue():
    """q' = fp16(fp32(q) * c32): one fp32 product, then one rounding to fp16 (round to nearest even)."""
    q = torch.tensor([[1.0, -3.0, 65504.0 / 8, 0.0, 1e-3]], dtype=torch.float16)
    scale = 40 ** -0.5
    want = [float(np.float16(np.float32(float(x)) * np.float32(c32(scale)))) for x in q[0]]
    assert q_eff(q, scale, True)[0].tolist() == want
    assert q_eff(q, scale, False)[0].tolist() == [float(x) for x in q[0]]


# ------------------------------------------------------------------------------------------------ GPU: cross probe
@pytest.mark.gpu
def test_every_head_dim_benign_ramp_one_hot():
    """All 16 head_dims (every k-step instantiation, ONES / embedded reference, the second 64-column block) through
    S1, S3 and S5 at one mid length."""
    cases = [(name, 1, 8, 129, 1000, d, 17 * d + i, {}) for d in HEAD_DIMS for i, name in enumerate(("S1", "S3", "S5"))]
    worst, bad = run_cross_cases(cases)
    _report("head_dims", worst)
    assert not bad, "\n".join(bad[:40])


@pytest.mark.gpu
@pytest.mark.parametrize("d", [40, 64, 80, 128])
@pytest.mark.parametrize("name", list(VARIANTS))
def test_key_and_query_lengths(name, d):
    """Every scenario at key lengths around the 64- and 96-key tiles (one key, two keys, no steady state, a last tile
    of one key) and query lengths around the 128-row tile.  Two samples where a length is 1 or 2: the projection
    epilogue's 32-row warps then span several samples."""
    cases = [(name, 2 if min(Lq, Lk) <= 2 else 1, 8, Lq, Lk, d, 7 * Lk + Lq + vi, kw)
             for vi, kw in enumerate(VARIANTS[name]) for Lk in LK_EDGES for Lq in LQ_EDGES]
    worst, bad = run_cross_cases(cases)
    _report(f"lengths d={d}", worst)
    assert not bad, "\n".join(bad[:40])


def _child(env, cases, label):
    """Run cross-probe cases in a child process: the kernel-selection variables are read once per process."""
    code = (
        "import json, sys\n"
        f"sys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, 'tests')!r}]\n"
        "import test_gpu_attention_edges as T\n"
        "cases = [tuple(c) for c in json.loads(sys.stdin.read())]\n"
        "worst, bad = T.run_cross_cases(cases)\n"
        "print('RESULT ' + json.dumps({'worst': worst, 'bad': bad}))\n")
    r = subprocess.run([sys.executable, "-c", code], input=json.dumps(cases), env=dict(os.environ, **env),
                       capture_output=True, text=True, timeout=600)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")]
    assert r.returncode == 0 and lines, r.stdout[-3000:] + r.stderr[-3000:]
    res = json.loads(lines[-1][7:])
    _report(label, res["worst"])
    assert not res["bad"], "\n".join(res["bad"][:40])


@pytest.mark.gpu
@pytest.mark.parametrize("splits", [2, 3, 8])
def test_forced_key_range_splits(splits):
    """Every tile cut into 2, 3 or 8 key ranges and merged by the combine kernel (8 x 3 = 24 tiles, fewer than the
    SMs, so all of them are split), with the maximum in different key ranges: the ramp (last range), the late spike at
    the start, the middle and the end, one-hot targets everywhere."""
    cases = []
    for d in (40, 64, 80, 128):
        for Lk in (769, 1000, 2000):
            cases.append(("S3", 1, 8, 300, Lk, d, Lk + d, {}))
            cases.append(("S5", 1, 8, 300, Lk, d, Lk + d + 1, {}))
            for sp in (0, Lk // 2, Lk - 1):
                for gap in S4_GAPS:
                    cases.append(("S4", 1, 8, 300, Lk, d, Lk + d + sp, {"gap": gap, "spike": sp}))
    _child({"VTM_FA_SPLITS": str(splits)}, cases, f"splits={splits}")


@pytest.mark.gpu
@pytest.mark.parametrize("env,dims", [({"VTM_FA_PAIRS": "1"}, (8, 24, 40)), ({"VTM_FA_GROUPS": "1"}, (40, 64, 80, 128)),
                                      ({"VTM_FA_EMBED": "0"}, (8, 40, 72, 120))])
def test_opt_in_flash_kernels_on_edge_scenarios(env, dims):
    """The alternative kernels kept for A/B runs (eight softmax warps, the grouped kernel, the non-embedded softmax)
    through the peaky, ramp, one-hot and deep scenarios."""
    cases = [(name, 1, 8, Lq, Lk, d, Lk * 3 + d + i, {})
             for d in dims for i, name in enumerate(("S2", "S3", "S5", "S6"))
             for Lq, Lk in ((128, 1), (129, 97), (300, 1000), (127, 193))]
    _child(env, cases, "opt-in " + ",".join(f"{a}={b}" for a, b in env.items()))


# ------------------------------------------------------------------------------------------------ GPU: self probe
def _self_case(name, B, H, L, d, seed, rows=None, shared_qk=False, kw=None):
    """Head 0 of every sample gets the designed (q, k, v); the other heads see the same blocks in other roles (plus
    benign blocks when H > 3).  Returns the worst error ratio over all heads and the checked rows."""
    kw = kw or {}
    scale = d ** -0.5
    emb = embedded(d)
    q0, k0, v0, info = make_scenario(name, B, L, L, d, scale, emb, seed, **kw)
    g = torch.Generator().manual_seed(seed + 1)
    rest = [torch.randn((B, L, d), generator=g).half() for _ in range(H - 3)]
    x = torch.stack([q0, k0, v0] + rest, 2).reshape(B, L, H * d).cuda()
    q, k, v = self_probe_qkv(x, H)
    sel = torch.arange(L, device="cuda") if rows is None else rows
    check_scenario(name, q0[:, sel.cpu()].cuda(), k0.cuda(), scale, emb, info, **kw)
    o = self_probe(x, H, scale, shared_qk)
    torch.cuda.synchronize()
    if L == 1:
        assert torch.equal(o, v), "a single key does not give o == v"
    if shared_qk:
        q, k = q[:1].expand_as(q), k[:1].expand_as(k)
    worst = 0.0
    for h in range(H):
        t = model_logits(q[:, h, sel], k[:, h], scale, emb)
        assert t.abs().max().item() <= T_MAX
        ref = softmax2_apply(t, v[:, h])
        worst = max(worst, row_ratio(o[:, h, sel], ref, v[:, h]).max().item())
    assert torch.isfinite(o).all()
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["S2", "S3"])
@pytest.mark.parametrize("B,L,H,d", [(1, 10241, 8, 40), (2, 2561, 8, 80)])
def test_self_attention_full_size(name, B, L, H, d):
    """The full-size merged lengths of BASELINE config 2 (ds1: L = 10241, head_dim 40; ds2: L = 2561, head_dim 80 at
    B = 2, H = 8, whose last wave is partial so the default key-range split applies) through the self-attention entry.
    The fp64 reference is evaluated on 640 rows (the last query tile included)."""
    g = torch.Generator().manual_seed(L)
    rows = torch.cat([torch.randperm(L - 128, generator=g)[:512], torch.arange(L - 128, L)]).sort().values.cuda()
    worst = _self_case(name, B, H, L, d, seed=L + d, rows=rows)
    _report(f"self {name} L={L} d={d}", {name: worst})
    assert worst <= TOL, worst


@pytest.mark.gpu
@pytest.mark.parametrize("L", [1, 2, 3, 63, 97, 300, 1000])
@pytest.mark.parametrize("d", [40, 80])
def test_self_attention_short_and_ragged(L, d):
    """Self-attention with fewer keys than one tile, ragged tiles and the fused QKV epilogue, S1 / S3 / S5.  L = 1 and 2
    with two samples: a 32-row warp of the projection epilogue spans up to 32 samples (L = 1 used to write rows 2 and 3
    of every four to the wrong place)."""
    worst = {}
    for i, name in enumerate(("S1", "S3", "S5")):
        worst[name] = _self_case(name, 2, 4, L, d, seed=L * 5 + d + i)
    _report(f"self short L={L} d={d}", worst)
    assert max(worst.values()) <= TOL, worst


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["S1", "S3"])
@pytest.mark.parametrize("d", [40, 80])
def test_pnp_shared_qk(name, d):
    """PnP's injection (shared_qk): the attention map of sample 0 applied to every sample's v."""
    worst = _self_case(name, 3, 4, 777, d, seed=d + 5, shared_qk=True)
    _report(f"pnp {name} d={d}", {name: worst})
    assert worst <= TOL, worst


# ------------------------------------------------------------------------------------------------ GPU: model-free
@pytest.mark.gpu
@pytest.mark.parametrize("d", [40, 64, 80, 128])
@pytest.mark.parametrize("name", ["S1", "S2"])
def test_no_worse_than_the_fp16_reference_formulation(name, d):
    """Against float64 of the UNROUNDED logits (q k^T * scale * log2 e, no fp32 scale, no fp16 q'): folding the scale
    into q costs nothing measurable against the reference's own fp16 formulation (einsum -> * scale -> softmax ->
    einsum, utils/pnp_utils.py:72-90)."""
    B, H, Lq, Lk = 2, 8, 300, 1000
    scale = d ** -0.5
    q, k, v, _ = make_scenario(name, B * H, Lq, Lk, d, scale, embedded(d), seed=d + len(name))
    q, k, v = [t.view(B * H, *t.shape[1:]).cuda() for t in (q, k, v)]
    t = (q.double() @ k.double().transpose(-1, -2)) * (scale * LOG2E)
    exact = softmax2_apply(t, v)
    sim = torch.einsum("b i d, b j d -> b i j", q, k) * scale
    ref16 = torch.einsum("b i j, b j d -> b i d", sim.softmax(dim=-1), v)
    o = cross_probe(q.view(B, H, Lq, d), k.view(B, H, Lk, d), v.view(B, H, Lk, d), scale).reshape(B * H, Lq, d)
    err_kd = (o.double() - exact).abs().max().item()
    err_16 = (ref16.double() - exact).abs().max().item()
    vmax = v.abs().max().item()
    print(f"\nEDGES model-free {name} d={d} kd={err_kd:.3e} fp16-reference={err_16:.3e} max|v|={vmax:.3g}")
    assert err_kd <= 2 * err_16 + 1e-3 * vmax, (err_kd, err_16)


# ------------------------------------------------------------------------------------------------ GPU: reference fixture
@pytest.mark.gpu
@pytest.mark.parametrize("fixture", ["pnp_attention_d40", "pnp_attention_d80"])
def test_reference_fixture_wide_heads(fixture):
    """The reference's replaced attn1.forward (utils/pnp_utils.py:39-106) at head_dim 40 and 80 with peaky logits,
    injection off and on (tests/make_golden_r02.py --pnp-wide).  KD must be no worse against float64 of the same module
    than 2 x the fixture's own error, + 1e-3 max|fixture|."""
    from vidtome_b200 import attention as A, pnp
    from vidtome_b200.skeleton import Attention
    g = np.load(os.path.join(ROOT, "tests", "golden", fixture + ".npz"))
    dim, heads = int(g["dim"]), int(g["heads"])
    attn = Attention(dim, heads, dim // heads).half()
    attn.load_state_dict({k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd_")})
    attn = attn.cuda().eval()
    pnp.register_attention_control(None, [int(t) for t in g["schedule"]], int(g["num_inputs"]), modules=[attn])
    x = torch.from_numpy(g["x"]).cuda()
    rows = torch.from_numpy(g["rows"]).long().cuda()
    B, L, _ = x.shape
    sd = {k: w.double() for k, w in attn.state_dict().items()}
    d, scale = dim // heads, float((dim // heads) ** -0.5)
    split = lambda t: t.view(B, L, heads, d).transpose(1, 2)
    xq = x.double()
    q, k, v = [split(xq @ sd[f"to_{n}.weight"].t()) for n in "qkv"]
    for t_step, key, inject in ((981, "out_inject", True), (500, "out_plain", False)):
        pnp.register_time(None, t_step, modules=[attn])
        qq, kk = (q[:1].expand_as(q), k[:1].expand_as(k)) if inject else (q, k)
        s = (qq[:, :, rows] @ kk.transpose(-1, -2)) * scale
        o = (s.softmax(-1) @ v).transpose(1, 2).reshape(B, len(rows), dim)
        exact = o @ sd["to_out.0.weight"].t() + sd["to_out.0.bias"]
        fix = torch.from_numpy(g[key]).cuda().double()
        with torch.no_grad():
            kd = A.self_attention(attn, x, shared_qk=pnp.injection_active(attn))[:, rows].double()
        err_fix = (fix - exact).abs().max().item()
        err_kd = (kd - exact).abs().max().item()
        print(f"\nEDGES fixture {fixture} {key} kd={err_kd:.3e} fixture={err_fix:.3e} max|fixture|={fix.abs().max().item():.3g}")
        assert err_kd <= 2 * err_fix + 1e-3 * fix.abs().max().item(), (key, err_kd, err_fix)
