"""KD (QKV projection + flash attention + output projection, all tcgen05) against a torch fp32 reference of
the same op (utils/pnp_utils.py:47-95 math) and against the numpy oracle.  Needs a B200."""
import numpy as np
import pytest
import torch

import vidtome_oracle as O

pytestmark = pytest.mark.gpu


def _ref_attention(x, wq, wk, wv, wo, bo, heads, scale):
    B, L, C = x.shape
    xf = x.float()
    q = (xf @ wq.float().t()).half().float().view(B, L, heads, -1).transpose(1, 2)
    k = (xf @ wk.float().t()).half().float().view(B, L, heads, -1).transpose(1, 2)
    v = (xf @ wv.float().t()).half().float().view(B, L, heads, -1).transpose(1, 2)
    s = (q @ k.transpose(-1, -2)) * scale
    o = (s.softmax(-1) @ v).transpose(1, 2).reshape(B, L, C).half().float()
    return o @ wo.float().t() + bo.float()


@pytest.mark.parametrize("B,L,C,heads", [
    (1, 128, 320, 8),       # one tile, head_dim 40
    (2, 333, 320, 8),       # ragged tiles (SURVEY: F=4, T=256 -> 333 merged tokens)
    (2, 641, 640, 8),       # head_dim 80: two 64-wide blocks
    (2, 1332, 320, 5),      # head_dim 64 (SD2.x)
    (2, 2561, 640, 8),      # BASELINE config 2, ds2 merged length
    (1, 700, 1024, 8),      # head_dim 128
    (2, 450, 384, 8),       # head_dim 48 (three k-steps, no spare column)
])
def test_attention_matches_fp32_reference(B, L, C, heads):
    from vidtome_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(L)
    x = torch.randn((B, L, C), generator=g, device="cuda").half()
    ws = [(torch.randn((C, C), generator=g, device="cuda") / C ** 0.5).half() for _ in range(4)]
    bo = (0.1 * torch.randn((C,), generator=g, device="cuda")).half()
    scale = (C // heads) ** -0.5
    y = ops.attention(x, torch.cat(ws[:3], 0).contiguous(), ws[3], bo, heads, scale)
    ref = _ref_attention(x, ws[0], ws[1], ws[2], ws[3], bo, heads, scale)
    err = (y.float() - ref).abs().max().item()
    assert torch.isfinite(y).all()
    assert err <= 1e-3 * ref.abs().max().item(), err      # measured on a B200: at most 4.9e-4 x max|ref| over these shapes


def test_attention_matches_oracle_small():
    from vidtome_b200 import ops
    rng = np.random.default_rng(0)
    B, L, C, heads = 2, 200, 128, 2
    x = rng.standard_normal((B, L, C)).astype(np.float16)
    w = [(rng.standard_normal((C, C)) / np.sqrt(C)).astype(np.float16) for _ in range(4)]
    bo = (0.1 * rng.standard_normal(C)).astype(np.float16)
    want = O.attention(x, w[0], w[1], w[2], w[3], bo, heads).astype(np.float32)
    t = lambda a: torch.from_numpy(a).cuda()
    y = ops.attention(t(x), torch.cat([t(w[0]), t(w[1]), t(w[2])], 0).contiguous(), t(w[3]), t(bo), heads,
                      (C // heads) ** -0.5)
    err = np.abs(y.float().cpu().numpy() - want).max()
    assert err <= 1.5e-3 * np.abs(want).max(), err      # measured on a B200: 4.9e-4 (one fp16 ulp) = 5.7e-4 x max|want|


def test_attention_full_size_c2_ds1_vs_sdpa():
    """BASELINE config 2, ds1 merged length (B=2, L=10241, C=320, 8 heads x 40) against torch SDPA on the
    same projections."""
    from vidtome_b200 import ops
    B, L, C, heads = 2, 10241, 320, 8
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn((B, L, C), generator=g, device="cuda").half()
    ws = [(torch.randn((C, C), generator=g, device="cuda") / C ** 0.5).half() for _ in range(4)]
    bo = torch.zeros((C,), device="cuda").half()
    y = ops.attention(x, torch.cat(ws[:3], 0).contiguous(), ws[3], bo, heads, 40 ** -0.5)
    q, k, v = [(x @ w.t()).view(B, L, heads, 40).transpose(1, 2) for w in ws[:3]]
    o = torch.nn.functional.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(B, L, C)
    ref = (o @ ws[3].t()).float()
    err = (y.float() - ref).abs().max().item()
    assert err <= 2e-3 * ref.abs().max().item(), err      # measured on a B200: 2.4e-4 (one fp16 ulp) = 7.2e-4 x max|ref|


def test_patched_block_uses_cuda_attention(monkeypatch):
    """With the attention kernel enabled the patched block must not call attn1.forward."""
    import vidtome_b200
    from vidtome_b200 import attention
    from vidtome_b200.skeleton import make_skeleton
    if not attention.ENABLED:
        pytest.skip("attention kernel not enabled")
    net = make_skeleton("tiny", device="cuda", max_downsample=1)
    vidtome_b200.apply_patch(net, batch_size=2)
    calls = []
    for blk in net.blocks:
        orig = type(blk.attn1).forward
        monkeypatch.setattr(type(blk.attn1), "forward", lambda self, *a, **k: calls.append(1) or orig(self, *a, **k))
    lat = torch.randn(8, 4, 16, 16, device="cuda", dtype=torch.float16)
    with torch.no_grad():
        out = net(lat, 0).sample
    assert torch.isfinite(out).all() and not calls


def test_pnp_shared_qk_attention_matches_reference_fixture():
    """f2: PnP's source-sample Q/K injection on merged tokens.  The fixture is the REFERENCE's replaced attn1.forward
    (utils/pnp_utils.py:39-106) on 3 samples with and without the injection active; here the same module goes through
    pnp.register_attention_control + KD (vtm_attention_ex, VTM_ATTN_SHARED_QK) and through the torch fallback forward."""
    import os
    import numpy as np
    from vidtome_b200 import attention as A, pnp
    from vidtome_b200.skeleton import Attention
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pnp_attention_b3.npz"))
    attn = Attention(int(g["dim"]), int(g["heads"]), int(g["dim"]) // int(g["heads"])).half()
    attn.load_state_dict({k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd_")})
    attn = attn.cuda().eval()
    pnp.register_attention_control(None, [int(v) for v in g["schedule"]], int(g["num_inputs"]), modules=[attn])
    x = torch.from_numpy(g["x"]).cuda()
    for t, key in ((981, "out_inject"), (500, "out_plain")):
        pnp.register_time(None, t, modules=[attn])
        ref = torch.from_numpy(g[key]).float()
        scale = ref.abs().max().item()
        with torch.no_grad():
            kd = A.self_attention(attn, x, shared_qk=pnp.injection_active(attn)).float().cpu()
            tf = attn(x).float().cpu()                           # the torch forward installed by pnp.py
        assert (kd - ref).abs().max().item() <= 1e-3 * scale + 1e-3, key
        assert (tf - ref).abs().max().item() <= 1e-3 * scale + 1e-3, key
    assert pnp.injection_active(attn) is False


def test_pnp_block_path_uses_kd_with_injection():
    """A patched block whose attn1 carries pnp.py's control runs KD with the shared attention map while the timestep is
    in the schedule: equal to the torch forward of the same module on the block's merged tokens."""
    import vidtome_b200
    from vidtome_b200 import patch, pnp
    from vidtome_b200.skeleton import make_skeleton
    net = make_skeleton("tiny", device="cuda", max_downsample=1, seed=3)
    vidtome_b200.apply_patch(net, batch_size=3, local_merge_ratio=0.9, align_batch=True)
    mods = [b.attn1 for b in net.blocks]
    pnp.register_attention_control(net, [981], 3, modules=mods)
    pnp.register_time(net, 981)
    assert all(patch._plain_attention_module(m) for m in mods)
    torch.manual_seed(1)
    lat = torch.randn(3 * 4, 4, 16, 16, device="cuda", dtype=torch.float16)
    outs = []
    for kd in (True, False):
        from vidtome_b200 import attention as A
        A.ENABLED = kd
        try:
            torch.manual_seed(5); torch.cuda.manual_seed(5)
            for b in net.blocks:
                if hasattr(b, "generator"):
                    del b.generator
            with torch.no_grad():
                outs.append(net(lat, 0).sample.float())
        finally:
            A.ENABLED = True
    err = (outs[0] - outs[1]).abs().max().item()
    assert err <= 2e-3 * outs[1].abs().max().item() + 1e-3


@pytest.mark.parametrize("B,Lq,Lk,C,Cctx,heads", [(6, 500, 77, 320, 768, 8), (4, 1024, 77, 640, 768, 8), (3, 130, 7, 128, 32, 2),
                                                    (2, 300, 77, 320, 1024, 5)])
def test_cross_attention_matches_fp32_reference(B, Lq, Lk, C, Cctx, heads):
    """f3: attn2 of the block (77 text tokens as keys/values, vidtome/patch.py:171-185) through vtm_cross_attention,
    with the residual fused, against fp32 torch."""
    from vidtome_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(Lq)
    x = torch.randn((B, Lq, C), generator=g, device="cuda").half()
    ctx = torch.randn((B, Lk, Cctx), generator=g, device="cuda").half()
    wq = (torch.randn((C, C), generator=g, device="cuda") / C ** 0.5).half()
    wk = (torch.randn((C, Cctx), generator=g, device="cuda") / Cctx ** 0.5).half()
    wv = (torch.randn((C, Cctx), generator=g, device="cuda") / Cctx ** 0.5).half()
    wo = (torch.randn((C, C), generator=g, device="cuda") / C ** 0.5).half()
    bo = (0.1 * torch.randn((C,), generator=g, device="cuda")).half()
    resid = torch.randn((B, Lq, C), generator=g, device="cuda").half()
    d = C // heads
    y = ops.cross_attention(x, ctx, wq, torch.cat([wk, wv], 0).contiguous(), wo, bo, heads, d ** -0.5, resid=resid)
    q = (x.float() @ wq.float().t()).view(B, Lq, heads, d).transpose(1, 2)
    k = (ctx.float() @ wk.float().t()).view(B, Lk, heads, d).transpose(1, 2)
    v = (ctx.float() @ wv.float().t()).view(B, Lk, heads, d).transpose(1, 2)
    o = torch.nn.functional.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(B, Lq, C)
    ref = o @ wo.float().t() + bo.float() + resid.float()
    err = (y.float() - ref).abs().max().item()
    assert err <= 1e-3 * ref.abs().max().item()      # measured on a B200: at most 4.4e-4 x max|ref| over these shapes
    y2 = ops.cross_attention(x, ctx, wq, torch.cat([wk, wv], 0).contiguous(), wo, bo, heads, d ** -0.5)
    # measured on a B200: at most 2.6e-4 x max|ref|
    assert (y2.float() - (ref - resid.float())).abs().max().item() <= 1e-3 * ref.abs().max().item()


def test_full_block_fast_paths_match_module_paths():
    """Full blocks (self-attention + cross-attention + GEGLU feed-forward) with the attn2 / ff fast paths on equal the
    same blocks with attn2 / ff running through their torch modules (FUSE_* switches off).  max_downsample=0 keeps the
    merge out of the comparison: through several blocks a 1e-3 difference would otherwise flip last-bit ties of LATER
    blocks' matches and turn a numerics check into a decision check (those are covered by the parity tests)."""
    import vidtome_b200
    from vidtome_b200 import patch
    from vidtome_b200.skeleton import make_skeleton
    outs = []
    for fast in (True, False):
        patch.FUSE_CROSS_ATTENTION = patch.FUSE_FEED_FORWARD = fast
        try:
            net = make_skeleton("tiny", device="cuda", hot_path_only=False, seed=11)
            vidtome_b200.apply_patch(net, batch_size=2, max_downsample=0)
            torch.manual_seed(2); torch.cuda.manual_seed(2)
            lat = torch.randn(2 * 4, 4, 16, 16, device="cuda", dtype=torch.float16)
            ctx = torch.randn(2 * 4, 77, 768, device="cuda", dtype=torch.float16)
            with torch.no_grad():
                outs.append(net(lat, 0, encoder_hidden_states=ctx).sample.float())
        finally:
            patch.FUSE_CROSS_ATTENTION = patch.FUSE_FEED_FORWARD = True
    err = (outs[0] - outs[1]).abs().max().item()
    assert err <= 3e-3 * outs[1].abs().max().item()


@pytest.mark.parametrize("env", [{"VTM_FA_PAIRS": "1"}, {"VTM_FA_GROUPS": "1"}, {"VTM_FA_EMBED": "0"}])
def test_opt_in_flash_kernels_match_fp32_reference(env):
    """The alternative flash kernels kept for A/B runs (eight softmax warps per CTA, the grouped kernel, the
    non-embedded softmax) are selected by environment variables read once per process: each runs in a child process on
    shapes that reach the steady-state loop, a masked last tile and the key-range split."""
    import os
    import subprocess
    import sys
    code = r'''
import sys, torch
sys.path.insert(0, %r)
from vidtome_b200 import ops
for (B, L, C, H) in [(2, 1000, 320, 8), (3, 1500, 320, 8), (1, 128, 320, 8)]:
    g = torch.Generator(device="cuda").manual_seed(L)
    x = torch.randn((B, L, C), generator=g, device="cuda").half()
    ws = [(torch.randn((C, C), generator=g, device="cuda") / C ** 0.5).half() for _ in range(4)]
    d = C // H
    y = ops.attention(x, torch.cat(ws[:3], 0).contiguous(), ws[3], None, H, d ** -0.5)
    q, k, v = [(x.float() @ w.float().t()).half().float().view(B, L, H, d).transpose(1, 2) for w in ws[:3]]
    o = ((q @ k.transpose(-1, -2)) * d ** -0.5).softmax(-1) @ v
    ref = o.transpose(1, 2).reshape(B, L, C).half().float() @ ws[3].float().t()
    err = (y.float() - ref).abs().max().item()
    # measured on a B200: at most 7.4e-4 x max|ref| (about one fp16 ulp of y) over the three kernels and shapes
    assert torch.isfinite(y).all() and err <= 1.5e-3 * ref.abs().max().item(), (L, err)
print("ok")
''' % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
