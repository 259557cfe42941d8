"""CPU: the op footprint model of tests/footprint.py, proven on the interpreter before the GPU tests trust it.

The write guard and the read poison run over the tiny guided-step plans with tests/plan_interp.Interp as the executor: a stray
write or a NaN there is a bug in the model or in the interpreter.  A self-test then shrinks one CONV op's write set and one
GroupNorm op's read set by a single channel and checks that the guard and the poison each report that op."""
import pytest
import torch as th

from tests.footprint import CODE, Guard, execution_order, footprint, format_failures
from tests.plan_interp import Interp
from tests.step_parity import build_tiny, make_inputs

VARIANTS = [dict(image=32), dict(image=64, B=1, cutn=2, use_magnitude=True, sat_scale=20.0, new_order=True),
            dict(image=64, B=2, cutn=3, cutout_resize="lanczos3"), dict(image=64, B=2, cutn=4, use_augs=True),
            dict(image=32, B=1, cutn=2, tower="rn", rn_width=80)]
IDS = ["b2_32px", "b1_64px_mag_sat_neworder", "b2_64px_resize_right", "b2_64px_use_augs", "rn80"]


def staged_tiny(device, **kw):
    """a tiny engine with one step's inputs staged, as tests/test_gpu_ops.py stages them"""
    ctx = build_tiny(device, **kw)
    eng = ctx["eng"]
    x, y, noise, _, coords = make_inputs(ctx)
    sc = ctx["pdiff"].scalar_table(14, 14, 0.0)
    th.manual_seed(77)  # use_augs: the aug parameters / noise fields are drawn while staging
    eng.stage_step(sc, coords, ctx["pdiff"].model_timestep(14), y)
    eng.img(eng.unet.x_in).copy_(x)
    eng.img(eng.noise).copy_(noise)
    return eng


@pytest.mark.parametrize("kw", VARIANTS, ids=IDS)
def test_interpreter_keeps_to_footprint(kw):
    plan = staged_tiny("cpu", **kw).plan
    it = Interp(plan)
    order = execution_order(plan)
    assert sorted(order) == list(range(len(plan.ops)))
    fails = Guard(plan, lambda k: it.run(k, 1)).check(order)
    assert not fails, f"{len(fails)} footprint violations on the interpreter:\n{format_failures(fails)}"


def _shrunk(target, slot, which):
    """footprint() with region `slot` of op `target` one channel narrower (its last dimension minus one)"""
    def fn(op, arena=None):
        fp = footprint(op, arena)
        if op is target:
            regions = fp.writes if which == "writes" else fp.reads
            for j, x in enumerate(regions):
                if x.slot == slot:
                    x.shape = x.shape[:-1] + (x.shape[-1] - 1,)
        return fp
    return fn


def test_guard_and_poison_can_fail():
    plan = staged_tiny("cpu", image=32).plan
    it = Interp(plan)
    order = execution_order(plan)
    conv = next(k for k in order if CODE[plan.ops[k].code] == "CONV" and not plan.ops[k].flags & 1 and plan.ops[k].i[4] > 8)
    gn = next(k for k in order if CODE[plan.ops[k].code].startswith("GN_FWD"))
    run = lambda k: it.run(k, 1)  # noqa: E731
    for k in order[:max(order.index(conv), order.index(gn)) + 1]:  # each target sees the real activations of its step
        if k == conv:
            # a write set one output channel short: the guard must see the op store the missing channel
            fails = Guard(plan, run, footprint_fn=_shrunk(plan.ops[conv], 4, "writes")).check([conv])
            assert any(f["kind"] == "stray write" and f["op"] == conv for f in fails), fails
            assert all(f["op"] == conv for f in fails)
        elif k == gn:
            # a read set one input channel short: that channel is poisoned, the statistics turn NaN, the outputs differ
            fails = Guard(plan, run, footprint_fn=_shrunk(plan.ops[gn], 0, "reads")).check([gn])
            assert any(f["kind"] == "stray read" and f["op"] == gn and f["nan_in_first"] for f in fails), fails
        else:
            run(k)
    # and the unmodified model passes both ops
    assert not Guard(plan, run).check([conv, gn])
