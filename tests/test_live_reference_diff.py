"""CPU: differential tests against the reference on many random inputs -- its importable modules (`cgd.modules`, `cgd.losses`), the
function bodies of `cgd/script_util.py` and the `cond_fn` closure of `cgd/cgd.py`.  The inputs are drawn below from fixed seeds;
`tests/golden/live_diff_golden.npz` holds what the reference returned for exactly these inputs (tests/golden/make_golden_live_diff.py
runs it on them).  The committed goldens of the other tests pin a handful of seeds; these widen the same comparisons.

Where the reference and ours agree bit for bit, the golden keeps the SHA-256 of the tensor's bytes, so the comparison stays exact; the
`cond_fn` gradients, compared to 1e-5 of their largest element, keep a fixed sample of 256 elements with their max and norm."""
import hashlib
import json
import os
import random

import numpy as np
import pytest
import torch as th

from tests.test_cond_fn_reference import StubClip, stub_pred_xstart

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "live_diff_golden.npz")
SAMPLE = 256


@pytest.fixture(scope="module")
def gold():
    d = np.load(GOLDEN)
    return dict(json.loads(bytes(d["json"]).decode()), cond_fn_samples=d["cond_fn_samples"], cond_fn_stats=d["cond_fn_stats"])


def digest(t: th.Tensor):
    """shape and SHA-256 of the float32 bytes: equal digests <=> bit-identical tensors"""
    t = t.detach().float().contiguous()
    return [list(t.shape), hashlib.sha256(t.numpy().tobytes()).hexdigest()]


def text_digest(s: str) -> str:
    return hashlib.sha256(s.encode()).hexdigest()[:16]


def sample_index(n: int) -> th.Tensor:
    return th.randperm(n, generator=th.Generator().manual_seed(0))[:SAMPLE].sort().values


# ------------------------------------------------------------------------------------------------ inputs (shared with the golden script)
def prompt_cases():
    """2000 (texts, batch index) pairs for alphanumeric_filter / clean_and_combine_prompts, then 2000 prompts for parse_prompt"""
    rng = random.Random(7)
    alphabet = "abc XYZ019_-.,:;!?/\\'\"()[]{}<>@#$%^&*+=~`|\t\néü中\U0001f600"
    combine, prompts = [], []
    for _ in range(2000):
        texts = ["".join(rng.choice(alphabet) for _ in range(rng.randint(0, n))) for n in (40, 300)]
        combine.append((texts, rng.randint(0, 99)))
    for _ in range(2000):
        body = "".join(rng.choice("ab :/.-") for _ in range(rng.randint(0, 12)))
        prompts.append(rng.choice(["", "http://", "https://"]) + body + rng.choice(["", ":1", ":-0.5", ":2e-1", ":3", ":", ":x"]))
    return combine, prompts


def window_cases():
    """300 random (cut size, image size, cutout count, power) geometries"""
    rng = random.Random(11)
    for trial in range(300):
        cs = rng.choice([32, 224, 288, 336, 384])
        side_x, side_y = rng.choice([64, 128, 256, 320, 512]), rng.choice([64, 128, 256, 320, 512])
        cutn, power = rng.randint(1, 40), rng.choice([1.0, 0.5, 2.0, 0.25])
        yield trial, cs, side_x, side_y, cutn, power


def window_outputs(make_cutouts):
    """the windows `make_cutouts(cut_size, cutn, power)` draws for every geometry: fresh, cached, and the default generator's state after
    the fresh draw; then the coords_for() prefix rule's inputs (cgd/modules.py:50-58) on 256x256"""
    rows = []
    for trial, cs, side_x, side_y, cutn, power in window_cases():
        mk = make_cutouts(cs, cutn, power)
        th.manual_seed(trial)
        fresh = mk._generate_coords(side_x, side_y, cutn)
        state = hashlib.sha256(th.get_rng_state().numpy().tobytes()).hexdigest()
        th.manual_seed(trial + 1)
        mk.cache_coordinates(side_x, side_y)
        rows.append(dict(fresh=[list(c) for c in fresh], cached=[list(c) for c in mk.cached_coords], rng_state=state))
    mk = make_cutouts(224, 16, 1.0)
    th.manual_seed(3)
    mk.cache_coordinates(256, 256)
    cached = [list(c) for c in mk.cached_coords]
    th.manual_seed(4)
    fresh = [list(c) for c in mk._generate_coords(256, 256, 8)]
    return dict(trials=rows, cached_256=cached, fresh_256=fresh)


def loss_outputs(range_loss, tv_loss, spherical_dist_loss, make_cutouts):
    """values and input gradients of the three losses and of MakeCutouts on 12 random batches, as digests"""
    g = th.Generator().manual_seed(5)
    out = []
    for trial in range(12):
        B, H, W = [1, 2, 3][trial % 3], [48, 64, 40][trial % 3], [48, 40, 64][(trial // 3) % 3]
        x = (th.randn(B, 3, H, W, generator=g) * 1.5).requires_grad_()
        seed = th.randn(B, generator=g)
        row = {}
        for name, fn in (("range", range_loss), ("tv", tv_loss)):
            a = fn(x)
            row[name] = digest(a)
            row[name + "_grad"] = digest(th.autograd.grad((a * seed).sum(), x)[0])
        e, t = th.randn(1, 5, B, 16, generator=g).requires_grad_(), th.randn(1, 1, 16, generator=g)
        a = spherical_dist_loss(e, t)
        row["spherical"], row["spherical_grad"] = digest(a), digest(th.autograd.grad(a.sum(), e)[0])
        if H >= W:  # wide images make the reference's swapped axes produce empty crops (RuntimeError in adaptive_avg_pool2d)
            th.manual_seed(trial)
            cut = make_cutouts(32, 4)(x)
            w = th.randn(cut.shape, generator=g)
            row["cutouts"], row["cutouts_grad"] = digest(cut), digest(th.autograd.grad((cut * w).sum(), x)[0])
        out.append(row)
    return out


def cond_fn_cases():
    """40 random (batch, prompts, image size, cutouts, power, chain length, timestep, scales, saturation, magnitude) configurations"""
    rng = random.Random(3)
    for trial in range(40):
        B = rng.choice([1, 1, 2, 3])
        P = 1 if B > 1 else rng.choice([1, 2, 4])  # quirk B1: the broadcast is only defined for B == 1 or P == 1
        H = rng.choice([32, 40, 48, 64])
        W = rng.choice([w for w in (32, 40, 48, 64) if w <= H])
        cutn, power, T = rng.randint(1, 7), rng.choice([1.0, 0.5, 2.0]), rng.choice([25, 50, 100])
        t, sat, mag = rng.randrange(T), rng.choice([0.0, 0.0, 12.5]), rng.random() < 0.5
        scales = dict(clip_guidance_scale=rng.choice([1000, 250.0]), tv_scale=rng.choice([150, 0.0, 20.0]), range_scale=rng.choice([50, 5.0]))
        g = th.Generator().manual_seed(1000 + trial)
        x = th.randn(B, 3, H, W, generator=g) * rng.choice([0.5, 1.0, 1.6])
        target = th.randn(P, 16, generator=g)
        w = th.randn(P, generator=g).abs() + 0.1
        w = w / w.sum().abs()
        yield dict(trial=trial, B=B, P=P, H=H, W=W, cutn=cutn, power=power, T=T, t=t, sat=sat, mag=mag, scales=scales, x=x, target=target, w=w)


# ------------------------------------------------------------------------------------------------ tests
def test_prompt_helpers_on_random_strings(gold):
    from clip_guided_diffusion_b200 import cgd
    want = gold["prompts"]
    combine, prompts = prompt_cases()
    for k, (texts, b) in enumerate(combine):
        assert cgd.alphanumeric_filter(texts[0]) == want["alphanumeric_filter"][k], k
        assert text_digest(cgd.clean_and_combine_prompts("base", texts, b)) == want["clean_and_combine_prompts"][k], k
    for prompt, w in zip(prompts, want["parse_prompt"]):
        if w is None:  # "text:" / "text:x": float('') raises in the reference, so it must here
            with pytest.raises(ValueError):
                cgd.parse_prompt(prompt)
        else:
            assert cgd.parse_prompt(prompt) == tuple(w), prompt


def test_cutout_windows_follow_the_reference_generator_for_random_geometries(gold):
    """same CPU-generator consumption and the same windows as cgd/modules.py:26-48 for random image sizes, cut sizes, counts, powers --
    fresh draws, cached draws and the `num_cutouts_override` prefix rule; product class and oracle class"""
    from clip_guided_diffusion_b200 import guidance as pg
    from oracle import guidance as og
    want = gold["windows"]
    for make in (lambda cs, n, p: pg.MakeCutouts(cs, n, cutout_size_power=p), og.MakeCutouts):
        got = window_outputs(make)
        for k, (g, w) in enumerate(zip(got["trials"], want["trials"])):
            assert g["fresh"] == w["fresh"] and g["cached"] == w["cached"], k
            assert g["rng_state"] == w["rng_state"], f"{k}: different consumption of the default generator"
        assert got["cached_256"] == want["cached_256"] and got["fresh_256"] == want["fresh_256"]
    # the product's coords_for() mirrors forward()'s choice between the cache and fresh draws (cgd/modules.py:50-58)
    mk = pg.MakeCutouts(224, 16)
    th.manual_seed(3)
    mk.cache_coordinates(256, 256)
    assert [list(c) for c in mk.coords_for(256, 256, use_cache=True, num_cutouts_override=4)] == want["cached_256"][:4]
    th.manual_seed(4)
    assert [list(c) for c in mk.coords_for(256, 256, use_cache=False, num_cutouts_override=8)] == want["fresh_256"]


def test_oracle_cutouts_and_losses_equal_the_reference_modules_on_random_inputs(gold):
    from oracle import guidance as og
    got = loss_outputs(og.range_loss, og.tv_loss, og.spherical_dist_loss, og.MakeCutouts)
    assert len(got) == len(gold["losses"])
    for trial, (g, w) in enumerate(zip(got, gold["losses"])):
        assert g == w, (trial, sorted(k for k in w if g.get(k) != w[k]))


def test_oracle_cond_fn_equals_the_live_reference_closure_on_random_configurations(gold):
    """the committed cond_fn goldens widened: the reference closure (cgd/cgd.py:151-239, compiled from its source) vs `OracleCondFn`
    on 40 random configurations"""
    from oracle import diffusion as od
    from oracle import guidance as og
    samples, stats = gold["cond_fn_samples"], gold["cond_fn_stats"]
    for c in cond_fn_cases():
        trial = c["trial"]
        diff = od.create_gaussian_diffusion(1000, "linear", str(c["T"]))
        cond = og.OracleCondFn(diff, StubClip(32, 16), c["target"], c["w"], cut_size=32, num_cutouts=c["cutn"], cutout_power=c["power"],
                               sat_scale=c["sat"], use_magnitude=c["mag"], **c["scales"])
        cond.current_timestep = c["t"]
        th.manual_seed(trial)
        xr = c["x"].clone().requires_grad_()
        got = cond(xr, th.full((c["B"],), c["t"]), {"pred_xstart": stub_pred_xstart(xr)}).detach().double().flatten()
        n, want_max, want_norm = int(stats[trial, 0]), float(stats[trial, 1]), float(stats[trial, 2])
        assert got.numel() == n, trial
        tol = 1e-5 * want_max + 1e-12
        idx = sample_index(n)
        err = float((got[idx] - th.from_numpy(samples[trial, :len(idx)]).double()).abs().max())
        assert err <= tol, (trial, c["B"], c["P"], c["H"], c["W"], c["cutn"], c["T"], c["t"], c["sat"], c["mag"])
        # what the elementwise bound implies for the elements outside the sample
        assert abs(float(got.abs().max()) - want_max) <= tol, trial
        assert abs(float(got.norm()) - want_norm) <= tol * n ** 0.5, trial
