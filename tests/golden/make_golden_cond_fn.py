"""Golden vectors of the reference's OWN `cond_fn` (cgd/cgd.py:151-239), executed here.

`cgd/cgd.py` does not import (clip / guided_diffusion / lpips are absent), but the guidance closure only needs its free variables: the
nested `def cond_fn` is cut out of the module source with `ast` and compiled UNMODIFIED into a namespace that supplies them --
the reference's real `cgd.modules.MakeCutouts` and `cgd.losses` (both import), `CLIP_NORMALIZE` evaluated from its own source line
(cgd/clip_util.py:45), a schedule table from the DDPM formulas, and two stand-ins whose definition is repeated in the test: a
deterministic "CLIP" (`StubClip`) and a deterministic `pred_xstart = f(x)` in place of the UNet.  What is pinned is everything the
closure itself does: the x_in blend with the float64 `fac`, normalisation, the view / broadcast of the spherical loss, the weighting and
reduction of every term, the saturation term, the sign, the whole-batch RMS clamp, the reduce_clip / progressive_cutout schedules.

    CGD_REFERENCE=<reference checkout> python tests/golden/make_golden_cond_fn.py      # writes tests/golden/cond_fn_golden.npz (committed)
"""
import ast
import json
import os
import sys
import types

import numpy as np
import torch as th
import torch.nn.functional as F
import torchvision.transforms as tvt

REF = os.environ["CGD_REFERENCE"]  # a checkout of the reference repository
sys.path.insert(0, REF)
from cgd import losses  # noqa: E402  (the reference's own module)
from cgd.modules import MakeCutouts  # noqa: E402  (the reference's own module)


def reference_cond_fn_code():
    tree = ast.parse(open(os.path.join(REF, "cgd", "cgd.py")).read())
    outer = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "clip_guided_diffusion")
    fn = next(n for n in ast.walk(outer) if isinstance(n, ast.FunctionDef) and n.name == "cond_fn")
    return compile(ast.Module([fn], []), "cgd/cgd.py", "exec")


def reference_clip_normalize():
    tree = ast.parse(open(os.path.join(REF, "cgd", "clip_util.py")).read())
    node = next(n for n in tree.body if isinstance(n, ast.Assign) and getattr(n.targets[0], "id", "") == "CLIP_NORMALIZE")
    return eval(compile(ast.Expression(node.value), "cgd/clip_util.py", "eval"), {"tvt": tvt})


class StubClip:
    """deterministic stand-in for clip_model: 8x8 mean pool -> fixed [3 * (cs / 8)^2, D] matrix of sines -> tanh"""

    def __init__(self, cut_size, dim):
        k = 3 * (cut_size // 8) ** 2
        i, j = th.arange(k, dtype=th.float64).view(-1, 1), th.arange(dim, dtype=th.float64).view(1, -1)
        self.w = th.sin(0.37 * i + 0.11 * j * j + 0.5).float()

    def encode_image(self, img):
        return th.tanh(F.avg_pool2d(img, 8).flatten(1) @ self.w)


def stub_pred_xstart(x):
    """deterministic stand-in for the UNet + p_mean_variance: any differentiable function of x_t"""
    return th.tanh(1.5 * x.roll(1, -1)) * 1.2 + 0.05 * x ** 2


def schedule(T):
    """sqrt(1 - abar) of the linear schedule respaced to T evenly strided steps of 1000 (float64, like guided-diffusion's numpy tables)"""
    abar = np.cumprod(1.0 - np.linspace(1e-4, 2e-2, 1000, dtype=np.float64))
    use = np.round(np.linspace(0, 999, T)).astype(int) if T < 1000 else np.arange(1000)
    return np.sqrt(1.0 - abar[use])


def make_closure(code, **free):
    ns = dict(th=th, losses=losses, tqdm=types.SimpleNamespace(write=lambda *a, **k: None), wandb_project=None, progress=False,
              clip_util=types.SimpleNamespace(CLIP_NORMALIZE=reference_clip_normalize()), lpips_vgg=None, init_tensor=None, init_scale=0,
              reduce_clip=False, progressive_cutout=False, cached_cutouts=False, timestep_respacing="25")
    ns.update(free)
    exec(code, ns)
    return ns


CASES = {
    # name: B, P, (H, W), cutn, cut_pow, T, current_timestep, sat_scale, use_magnitude, seed
    "plain": dict(B=1, P=1, hw=(48, 48), cutn=5, pow=1.0, T=25, t=10, sat=0.0, mag=False, seed=1),
    "late_step": dict(B=1, P=1, hw=(48, 48), cutn=3, pow=1.0, T=25, t=1, sat=0.0, mag=False, seed=2),
    "batch2_sat_magnitude": dict(B=2, P=1, hw=(48, 48), cutn=4, pow=1.0, T=25, t=20, sat=30.0, mag=True, seed=3),
    "three_prompts": dict(B=1, P=3, hw=(48, 48), cutn=4, pow=1.0, T=50, t=31, sat=0.0, mag=False, seed=4),
    "tall_image_cut_power": dict(B=1, P=1, hw=(48, 40), cutn=6, pow=0.5, T=25, t=15, sat=5.0, mag=True, seed=5),
}


def main():
    code = reference_cond_fn_code()
    out = {}
    cs, D = 32, 16
    for name, c in CASES.items():
        g = th.Generator().manual_seed(100 + c["seed"])
        x = th.randn(c["B"], 3, *c["hw"], generator=g) * 1.3
        target = th.randn(c["P"], D, generator=g)
        w = th.tensor([1.0, 0.6, -0.3][:c["P"]])
        w = w / w.sum().abs()  # cgd/cgd.py:102-105
        sq = schedule(c["T"])
        ns = make_closure(code, diffusion=types.SimpleNamespace(num_timesteps=c["T"], sqrt_one_minus_alphas_cumprod=sq), current_timestep=c["t"],
                          num_cutouts=c["cutn"], make_cutouts=MakeCutouts(cs, c["cutn"], cutout_size_power=c["pow"]), clip_model=StubClip(cs, D),
                          target_embeds=target, weights=w, clip_guidance_scale=1000, tv_scale=150, range_scale=50, sat_scale=c["sat"],
                          use_saturation=c["sat"] != 0, use_magnitude=c["mag"])
        th.manual_seed(c["seed"])  # the cutout windows come from the default CPU generator (cgd/modules.py:38-48)
        xr = x.clone().requires_grad_()
        grad = ns["cond_fn"](xr, th.full((c["B"],), c["t"]), {"pred_xstart": stub_pred_xstart(xr)})
        out[name + "_x"], out[name + "_target"], out[name + "_weights"] = x.numpy(), target.numpy(), w.numpy()
        out[name + "_grad"], out[name + "_fac"] = grad.detach().numpy(), np.array([sq[c["t"]]])
    # the two schedules, as the closure itself decides them for every value of current_timestep
    sched = {}

    class _Stop(Exception):
        pass

    def spy(x, use_cache=False, num_cutouts_override=None):
        raise _Stop(num_cutouts_override, use_cache)

    for T in (25, 50, 250, 1000):
        for n in (16, 8, 6, 32):
            rows = []
            for reduce_clip, progressive, cached in ((True, False, False), (False, True, True), (True, True, False)):
                ns = make_closure(code, diffusion=types.SimpleNamespace(num_timesteps=T, sqrt_one_minus_alphas_cumprod=schedule(min(T, 1000))), num_cutouts=n,
                                  make_cutouts=spy, reduce_clip=reduce_clip, progressive_cutout=progressive, cached_cutouts=cached, clip_model=None,
                                  target_embeds=None, weights=None, clip_guidance_scale=0, tv_scale=0, range_scale=0, sat_scale=0, use_saturation=False,
                                  use_magnitude=False, current_timestep=0)
                per_t = []
                for t in range(T - 1, -1, -1):
                    ns["current_timestep"] = t
                    x = th.zeros(1, 3, 8, 8, requires_grad=True)
                    try:
                        r = ns["cond_fn"](x, None, {"pred_xstart": x * 1.0})
                        assert th.equal(r, th.zeros_like(x))
                        per_t.append([t, 1, 0, 0])  # guidance skipped: zeros returned before make_cutouts is reached
                    except _Stop as s:
                        per_t.append([t, 0, int(s.args[0]), int(bool(s.args[1]))])
                rows.append(per_t)
            sched[f"{T}/{n}"] = rows
    out["schedules_json"] = np.frombuffer(json.dumps(sched).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(os.path.dirname(os.path.abspath(__file__)), "cond_fn_golden.npz"), **out)
    print({k: v.shape for k, v in out.items() if k.endswith("_grad")}, len(sched))


if __name__ == "__main__":
    main()
