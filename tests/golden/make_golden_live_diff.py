"""Golden vectors of tests/test_live_reference_diff.py: the reference's own prompt helpers (function bodies of cgd/script_util.py cut
out with `ast`; the module does not import), `cgd.modules.MakeCutouts`, `cgd.losses` and the `cond_fn` closure of cgd/cgd.py (compiled
from its source as in make_golden_cond_fn.py), run on the inputs the test draws.

    CGD_REFERENCE=<reference checkout> python tests/golden/make_golden_live_diff.py    # writes tests/golden/live_diff_golden.npz
"""
import ast
import json
import os
import re
import sys
import types

import numpy as np
import torch as th

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REF = os.environ["CGD_REFERENCE"]  # a checkout of the reference repository
sys.path.insert(0, ROOT)
sys.path.append(REF)  # appended: nothing of this repository may be shadowed
sys.path.append(os.path.dirname(os.path.abspath(__file__)))

import make_golden_cond_fn as mg  # noqa: E402
from cgd import losses, modules  # noqa: E402  (the reference's own modules)
from oracle import diffusion as od  # noqa: E402
from tests import test_live_reference_diff as lt  # noqa: E402  (the inputs)


def script_util():
    ns = {"os": os, "re": re}
    src = open(os.path.join(REF, "cgd", "script_util.py")).read()
    for node in ast.parse(src).body:
        if isinstance(node, ast.FunctionDef) and node.name in ("parse_prompt", "alphanumeric_filter", "clean_and_combine_prompts"):
            exec(compile(ast.Module([node], []), "cgd/script_util.py", "exec"), ns)
    return ns


def prompts():
    ref = script_util()
    combine, prompt_list = lt.prompt_cases()
    parsed = []
    for p in prompt_list:
        try:
            parsed.append(list(ref["parse_prompt"](p)))
        except ValueError:
            parsed.append(None)
    return dict(alphanumeric_filter=[ref["alphanumeric_filter"](texts[0]) for texts, _ in combine],
                clean_and_combine_prompts=[lt.text_digest(ref["clean_and_combine_prompts"]("base", texts, b)) for texts, b in combine],
                parse_prompt=parsed)


def cond_fn():
    code = mg.reference_cond_fn_code()
    samples, stats = np.zeros((40, lt.SAMPLE), np.float32), np.zeros((40, 3), np.float64)
    for c in lt.cond_fn_cases():
        diff = od.create_gaussian_diffusion(1000, "linear", str(c["T"]))
        ns = mg.make_closure(code, diffusion=types.SimpleNamespace(num_timesteps=c["T"], sqrt_one_minus_alphas_cumprod=diff.sqrt_one_minus_alphas_cumprod),
                             current_timestep=c["t"], num_cutouts=c["cutn"], make_cutouts=modules.MakeCutouts(32, c["cutn"], cutout_size_power=c["power"]),
                             clip_model=mg.StubClip(32, 16), target_embeds=c["target"], weights=c["w"], sat_scale=c["sat"], use_saturation=c["sat"] != 0,
                             use_magnitude=c["mag"], **c["scales"])
        th.manual_seed(c["trial"])
        xr = c["x"].clone().requires_grad_()
        want = ns["cond_fn"](xr, th.full((c["B"],), c["t"]), {"pred_xstart": mg.stub_pred_xstart(xr)}).detach().flatten()
        idx = lt.sample_index(want.numel())
        samples[c["trial"], :len(idx)] = want[idx].numpy()
        stats[c["trial"]] = [want.numel(), float(want.double().abs().max()), float(want.double().norm())]
    return samples, stats


def main():
    gold = dict(prompts=prompts(),
                windows=lt.window_outputs(lambda cs, n, p: modules.MakeCutouts(cs, n, cutout_size_power=p)),
                losses=lt.loss_outputs(losses.range_loss, losses.tv_loss, losses.spherical_dist_loss, modules.MakeCutouts))
    samples, stats = cond_fn()
    blob = np.frombuffer(json.dumps(gold).encode(), dtype=np.uint8)
    np.savez_compressed(lt.GOLDEN, json=blob, cond_fn_samples=samples, cond_fn_stats=stats)
    print(lt.GOLDEN, os.path.getsize(lt.GOLDEN), "bytes")


if __name__ == "__main__":
    main()
