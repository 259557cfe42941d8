"""GPU: every kernel writes only its declared outputs and reads only its declared inputs (tests/footprint.py), op by op over
the tiny step plans, the full-size cfg2 and default128 engines and the opt-in engines; and the conv / GroupNorm / elementwise
kernels on channel slices of wider tensors (eoff > 0, ld > C) against fp32 torch, with the neighbouring channels and a guard
region after the buffer holding a sentinel that must come back bit for bit."""
import os
import subprocess
import sys
import time

import pytest
import torch as th
import torch.nn.functional as F

from clip_guided_diffusion_b200.plan import Act, Plan, pack_conv
from tests.footprint import CODE, Guard, execution_order, format_failures
from tests.test_footprint_cpu import IDS, VARIANTS, staged_tiny

pytestmark = pytest.mark.gpu

# ops that accumulate with float atomics: not bitwise reproducible, compared at a tolerance
ATOMIC_OPS = ("GUIDE_GRAD", "CUTOUTS_AUG_BWD", "LPIPS_TAP")


def _guard_plan(plan, label):
    def run(k):
        plan.run(k, 1)
        th.cuda.synchronize()

    order = execution_order(plan)
    t0 = time.time()
    fails = Guard(plan, run, atomic_ops=ATOMIC_OPS).check(order)
    print(f"{label}: {len(order)} ops, arena {plan.arena.numel() / 1e9:.2f} GB, {time.time() - t0:.1f} s")
    assert not fails, f"{label}: {len(fails)} footprint violations:\n{format_failures(fails, 60)}"


@pytest.mark.parametrize("kw", VARIANTS, ids=IDS)
def test_tiny_step_footprint(kw):
    eng = staged_tiny("cuda", **kw)
    th.cuda.synchronize()
    _guard_plan(eng.plan, "tiny " + str(kw))


def test_epilogue_stats_footprint():
    """CONV flags 2 (epilogue statistics) -> GN_APPLY_EPI and their backward: the pair only large activations reach"""
    th.manual_seed(0)
    N, H, W, Cin, C = 1, 128, 128, 256, 256
    plan = Plan()
    plan.gn_epi_stats, plan.fused_gn, plan.grid_gn = True, False, True
    cw = pack_conv(plan, th.randn(C, Cin, 3, 3) * (9 * Cin) ** -0.5, th.randn(C) * 0.1, name="w")
    x = plan.act(N, H, W, Cin, "x")
    h = plan.conv(x, cw, name="c")
    y = plan.group_norm(h, plan.const(1 + 0.1 * th.randn(C), "f", "g"), plan.const(0.1 * th.randn(C), "f", "b"),
                        emb=(plan.const(0.2 * th.randn(N * 2 * C), "f", "e"), 0), name="gn")
    dy = plan.act(N, H, W, C, "dy")
    plan._grads[y.key()] = dy
    plan.backward()
    plan.finalize("cuda")
    assert any(CODE[o.code] == "GN_APPLY_EPI" for o in plan.ops)
    plan.view(x.buf).normal_()
    plan.view(dy.buf).normal_()
    _guard_plan(plan, "epilogue stats")


FULL = {"cfg2": dict(size=256, respacing="ddim250", cutn=16, clip="ViT-B/32", t_index=180),
        "default128": dict(size=128, respacing="1000", cutn=16, clip="ViT-B/32", t_index=500)}


@pytest.mark.parametrize("name", list(FULL))
def test_full_size_footprint(name):
    """the benchmarked plan (256x256 UNet, ViT-B/32 over 16 cutouts) and the 128x128 checkpoint (192- / 768-wide concatenations,
    wide-head attention), built as tests/test_gpu_baseline_configs.py builds them"""
    from clip_guided_diffusion_b200 import gaussian_diffusion as pgd
    from clip_guided_diffusion_b200 import guidance as pg
    from clip_guided_diffusion_b200 import unet as pu
    from clip_guided_diffusion_b200 import vit as pv
    from clip_guided_diffusion_b200 import weights as pw
    c = FULL[name]
    ucfg, vcfg = pu.config_for(c["size"], True), pv.VIT_CONFIGS[c["clip"]]
    usd = pw.seeded_state_dict(pw.unet_param_shapes(ucfg), 1234)
    vsd = pw.seeded_state_dict(pw.vit_param_shapes(vcfg), 1235)
    g = th.Generator().manual_seed(17)
    eng = pg.GuidedStepB200(ucfg, usd, vcfg, vsd, batch=1, num_cutouts=c["cutn"], device="cuda:0")
    del usd, vsd
    eng.set_targets(th.randn(1, vcfg.output_dim, generator=g), th.ones(1))
    pdiff = pgd.create_gaussian_diffusion(1000, "linear", c["respacing"], rescale_timesteps=ucfg.rescale_timesteps)
    th.manual_seed(23)
    coords = pg.MakeCutouts(vcfg.input_resolution, c["cutn"])._generate_coords(c["size"], c["size"], c["cutn"])
    eng.stage_step(pdiff.scalar_table(c["t_index"], c["t_index"], 0.0), coords, pdiff.model_timestep(c["t_index"]), th.tensor([417]))
    eng.img(eng.unet.x_in).copy_(th.randn(1, 3, c["size"], c["size"], generator=g))
    eng.img(eng.noise).copy_(th.randn(1, 3, c["size"], c["size"], generator=g))
    th.cuda.synchronize()
    try:
        _guard_plan(eng.plan, name)
    finally:
        del eng
        th.cuda.empty_cache()


@pytest.mark.parametrize("env", [dict(CGD_CONV_SMALL="1"), dict(CGD_GN_GRID_ENGINE="stream"), dict(CGD_GN_GRID_ENGINE="ring"),
                                 dict(CGD_GN_EPI_STATS="1")], ids=["conv_small", "gn_stream", "gn_ring", "gn_epi_stats"])
def test_opt_in_engines_footprint(env):
    """engines the default plans never reach are chosen once per process: the tiny plans (the RN tower has 8 x 8 convs) and the
    epilogue-statistics plan are re-run in a child process with each switch on"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_footprint.py", "-q", "-x", "-m", "gpu", "-k",
                        "tiny_step_footprint and (b2_32px or rn80) or epilogue_stats_footprint", "-p", "no:cacheprovider"],
                       cwd=root, env=dict(os.environ, **env), capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]


# ---------------------------------------------------------------------- slice layouts against fp32 torch
def _slice(plan, N, H, W, C, name, lead=8, tail=24, guard=64):
    """channel slice [lead, lead + C) of a [N, H, W, lead + C + tail] tensor whose buffer ends with `guard` more elements"""
    ld = lead + C + tail
    return Act(plan.new(N * H * W * ld + guard, "h", name), lead, N, H, W, C, ld)


def _sentinel_fill(plan, a: Act, gen, data=None):
    """fill a's whole buffer with a seeded non-zero sentinel, then the slice with `data` (or N(0, 1)); returns the buffer's
    snapshot and the mask of its sentinel elements"""
    buf = plan.view(a.buf)
    buf.copy_((th.rand(buf.numel(), generator=gen) * 900 + 100).half().to(buf.device))
    sl = _sl(plan, a)
    sl.copy_(data if data is not None else th.randn(sl.shape, generator=gen).to(sl.device))
    mask = th.ones(buf.numel(), dtype=th.bool, device=buf.device)
    _sl(plan, a, mask).fill_(False)
    return buf.clone(), mask


def _sl(plan, a: Act, t=None):
    t = plan.view(a.buf) if t is None else t  # as_strided offsets count from the storage, not from the view
    v = t.as_strided((a.N, a.H, a.W, a.C), (a.H * a.W * a.ld, a.W * a.ld, a.ld, 1), t.storage_offset() + a.eoff)
    assert v.data_ptr() == t.data_ptr() + a.eoff * t.element_size()
    return v


def _assert_sentinel(plan, a: Act, snap, mask, what):
    now = plan.view(a.buf)
    bad = (now.view(th.int16) != snap.view(th.int16)) & mask
    n = int(bad.sum())
    if n:
        e = int(th.nonzero(bad)[0])
        px, ch = divmod(e, a.ld) if e < a.N * a.H * a.W * a.ld else (None, e - a.N * a.H * a.W * a.ld)
        raise AssertionError(f"{what}: {n} sentinel elements overwritten, first at element {e} "
                             + (f"(pixel {px}, channel {ch} of ld {a.ld}; slice is [{a.eoff}, {a.eoff + a.C}))" if px is not None else f"(guard element {ch})"))


CONV_CASES = [
    # name, NB, H, W, Cin, Cout, taps, bias, res, existing dx
    ("tma_epi_1x1_64x64", 1, 64, 64, 256, 192, 1, True, True, False),        # pair kernel, TMA-store epilogue
    ("scalar_epi_cout96", 1, 32, 32, 128, 96, 1, True, True, False),         # Cout % 64 != 0: scalar / vector epilogue (no dgrad:
                                                                             # its K = Cout would not be a multiple of 64)
    ("ws_splitk_16x16_c512", 1, 16, 16, 512, 512, 9, True, True, False),     # workspace split-K (12 splits)
    ("cluster_splitk_32x32_c256", 1, 32, 32, 256, 256, 9, False, False, True),  # in-cluster split-K; dgrad accumulates into a strided gradient
    ("img8x8_c256_b2", 2, 8, 8, 256, 256, 9, True, True, True),              # 8 x 8 images
]


@pytest.mark.parametrize("impl", [0, 1, 2, 3, 13], ids=["auto", "simt", "tc1", "tc2pair", "tc2pair_ws_splitk"])
@pytest.mark.parametrize("case", CONV_CASES, ids=[c[0] for c in CONV_CASES])
def test_conv_on_channel_slices(case, impl):
    name, NB, H, W, Cin, Cout, taps, has_b, has_r, acc = case
    cluster = impl != 13
    impl = 3 if impl == 13 else impl
    th.manual_seed(0)
    gen = th.Generator().manual_seed(5)
    k = 3 if taps == 9 else 1
    w = th.randn(Cout, Cin, k, k) * (taps * Cin) ** -0.5
    b = th.randn(Cout) * 0.1 if has_b else None
    plan = Plan(conv_impl=impl)
    plan.cluster_splitk = cluster
    bwd = Cout % 64 == 0
    cw = pack_conv(plan, w, b, need_bwd=bwd, name=name)
    x = _slice(plan, NB, H, W, Cin, "x", lead=64, tail=64)
    res = _slice(plan, NB, H, W, Cout, "res", lead=16, tail=40) if has_r else None
    y = _slice(plan, NB, H, W, Cout, "y", lead=24, tail=8)
    plan.conv(x, cw, res=res, out=y, name=name)
    dy = _slice(plan, NB, H, W, Cout, "dy", lead=8, tail=56)
    plan._grads[y.key()] = dy
    gx = _slice(plan, NB, H, W, Cin, "gx", lead=128, tail=8) if acc else None
    if acc:
        plan._grads[x.key()] = gx
    plan.mark("bwd")
    plan.backward()
    plan.mark("end")
    plan.finalize("cuda")
    snaps = {nm: _sentinel_fill(plan, a, gen) for nm, a in (("x", x), ("res", res), ("y", y), ("dy", dy), ("gx", gx)) if a is not None}
    g0 = _sl(plan, gx).float().clone() if acc else 0.0
    plan.run(0, plan.marks["bwd"])
    th.cuda.synchronize()
    xv = _sl(plan, x).float()
    ref = F.conv2d(xv.permute(0, 3, 1, 2), w.cuda(), b.cuda() if has_b else None, padding=k // 2).permute(0, 2, 3, 1)
    if has_r:
        ref = ref + _sl(plan, res).float()
    got = _sl(plan, y).float()
    err = float((got - ref).abs().max() / ref.abs().max())
    assert th.isfinite(got).all() and err < 3e-3, f"{name} fwd impl={impl}: rel-to-max err {err:.3e}"
    if bwd:
        _check_dgrad(plan, x, dy, gx, w, k, xv, g0, acc, f"{name} impl={impl}")
    for nm, a in (("x", x), ("res", res), ("y", y), ("dy", dy), ("gx", gx)):
        if a is not None:
            _assert_sentinel(plan, a, *snaps[nm], f"{name} impl={impl} {nm}")


def _check_dgrad(plan, x, dy, gx, w, k, xv, g0, acc, what):
    plan.run(plan.marks["bwd"], plan.marks["end"] - plan.marks["bwd"])
    th.cuda.synchronize()
    xg = xv.clone().requires_grad_()
    yr = F.conv2d(xg.permute(0, 3, 1, 2), w.cuda(), None, padding=k // 2).permute(0, 2, 3, 1)
    (gref,) = th.autograd.grad((yr * _sl(plan, dy).float()).sum(), xg)
    gref = gref + g0
    dx = plan.grad_of(x)
    assert (dx is gx) == acc
    gg = _sl(plan, dx).float()
    err = float((gg - gref).abs().max() / gref.abs().max())
    assert th.isfinite(gg).all() and err < 3e-3, f"{what} dgrad: rel-to-max err {err:.3e}"


GN_CASES = [(1, 1024, 512), (1, 16384, 256), (2, 4096, 192)]


@pytest.mark.parametrize("acc", [False, True], ids=["dx", "dx_acc"])
@pytest.mark.parametrize("fused", ["auto", "grid", "twopass"])
@pytest.mark.parametrize("case", GN_CASES, ids=[f"n{c[0]}_hw{c[1]}_c{c[2]}" for c in GN_CASES])
def test_group_norm_on_channel_slices(case, fused, acc):
    N, HW, C = case
    th.manual_seed(0)
    gen = th.Generator().manual_seed(6)
    plan = Plan()
    plan.fused_gn = fused == "auto"
    plan.grid_gn = fused != "twopass"
    gamma, beta, emb = 1 + 0.2 * th.randn(C), 0.1 * th.randn(C), 0.3 * th.randn(N, 2 * C)
    x = _slice(plan, N, 1, HW, C, "x", lead=40, tail=24)
    y = plan.group_norm(x, plan.const(gamma, "f", "g"), plan.const(beta, "f", "b"), emb=(plan.const(emb, "f", "e"), 0), silu=True, name="gn")
    dy = _slice(plan, N, 1, HW, C, "dy", lead=8, tail=64)
    plan._grads[y.key()] = dy
    gx = _slice(plan, N, 1, HW, C, "gx", lead=64, tail=8) if acc else None
    if acc:
        plan._grads[x.key()] = gx
    plan.backward()
    plan.finalize("cuda")
    bwd = [o for o in plan.ops if CODE[o.code] in ("GN_BWD_APPLY", "GN_BWD_FUSED", "GN_BWD_GRID")]
    assert bwd and all(bool(o.flags & 2) == acc for o in bwd)
    xd = th.randn(N, 1, HW, C, generator=gen) * 1.5 + 0.3 * th.randn(N, 1, 1, C, generator=gen)
    snaps = {nm: _sentinel_fill(plan, a, gen, xd if nm == "x" else None) for nm, a in (("x", x), ("dy", dy), ("gx", gx)) if a is not None}
    g0 = _sl(plan, gx).float().clone() if acc else 0.0
    plan.run()
    th.cuda.synchronize()
    xg = _sl(plan, x).float().view(N, HW, C).clone().requires_grad_()
    e = emb.cuda()
    h = F.group_norm(xg.permute(0, 2, 1), 32, gamma.cuda(), beta.cuda(), 1e-5).permute(0, 2, 1)
    ref = F.silu(h * (1 + e[:, None, :C]) + e[:, None, C:])
    got = plan.view(y.buf, (N, HW, C)).float()
    err = float((got - ref.detach()).abs().max() / ref.detach().abs().max())
    assert th.isfinite(got).all() and err < 2e-3, f"y {fused}: rel-to-max {err:.3e}"
    (gref,) = th.autograd.grad((ref * _sl(plan, dy).float().view(N, HW, C)).sum(), xg)
    gref = gref.view(N, 1, HW, C) + g0
    gg = _sl(plan, plan.grad_of(x)).float()
    err = float((gg - gref).abs().max() / gref.abs().max())
    assert th.isfinite(gg).all() and err < 3e-3, f"dx {fused} acc={acc}: rel-to-max {err:.3e}"
    for nm, a in (("x", x), ("dy", dy), ("gx", gx)):
        if a is not None:
            _assert_sentinel(plan, a, *snaps[nm], f"gn {fused} acc={acc} {nm}")


@pytest.mark.parametrize("code", ["ADD", "COPY", "POOL2", "UP2"])
def test_elementwise_on_channel_slices(code):
    """ADD / COPY / POOL2 / UP2 with three different leading dimensions and element offsets"""
    gen = th.Generator().manual_seed(7)
    N, H, W, C = 2, 16, 12, 200
    plan = Plan()
    a = _slice(plan, N, H, W, C, "a", lead=8, tail=16)
    b = _slice(plan, N, H, W, C, "b", lead=32, tail=48)
    Ho, Wo = {"POOL2": (H // 2, W // 2), "UP2": (2 * H, 2 * W)}.get(code, (H, W))
    c = _slice(plan, N, Ho, Wo, C, "c", lead=64, tail=8)
    if code == "ADD":
        plan.emit("ADD", i=[a.rows, C, a.ld, b.ld, c.ld], p=[plan._ap(a), plan._ap(b), plan._ap(c)])
    elif code == "COPY":
        plan.emit("COPY", i=[a.rows, C, a.ld, c.ld], p=[plan._ap(a), plan._ap(c)])
    else:
        plan.emit(code, i=[N, H, W, C, a.ld, c.ld], f=[0.25 if code == "POOL2" else 1.5], p=[plan._ap(a), plan._ap(c)])
    plan.finalize("cuda")
    snaps = {nm: _sentinel_fill(plan, t, gen) for nm, t in (("a", a), ("b", b), ("c", c))}
    plan.run()
    th.cuda.synchronize()
    av, bv = _sl(plan, a).float(), _sl(plan, b).float()
    ref = {"ADD": lambda: av + bv, "COPY": lambda: av,
           "POOL2": lambda: F.avg_pool2d(av.permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1),
           "UP2": lambda: 1.5 * av.repeat_interleave(2, 1).repeat_interleave(2, 2)}[code]()
    got = _sl(plan, c).float()
    assert float((got - ref).abs().max()) <= 2e-3 * float(ref.abs().max()), code
    for nm, t in (("a", a), ("b", b), ("c", c)):
        _assert_sentinel(plan, t, *snaps[nm], f"{code} {nm}")
