"""Memory footprint of plan ops, and the write guard / read poison that hold every kernel to it.

Every activation lives at a fixed offset in one arena, and the UNet's skip concatenations are written in place by two producers
at different times (channel slices with ld > C).  A kernel that stores one channel too many, or reads past its slice, corrupts
a neighbour that a later op may or may not overwrite.  `footprint(op)` states, from the slot tables of include/cgd_b200.h
alone, which arena bytes an op may write and which it may read; `Guard` runs ops one at a time and checks both:

  write guard  every 2-byte word an op changed lies in its write set (alignment gaps between buffers included);
  read poison  every floating-point buffer region outside the op's read and write sets (and every gap) is set to NaN, the op
               runs, the arena is restored, the op runs again: the outputs of the two runs must be bitwise equal.  Integer
               buffers (coordinates, labels, counters, barriers) are never poisoned, so no poisoned value becomes an address or
               a loop bound.

A clean-twice mismatch (an op that is not bitwise reproducible on identical inputs) is reported as a race unless the op code
is on the caller's allow-list of float-atomic ops, which are compared at a tolerance instead.

The guard works on any arena: the device plan with `plan.run(k, 1)`, or its CPU twin with the interpreter.
"""
from __future__ import annotations

import bisect
from dataclasses import dataclass, field
from typing import Callable, Optional

import torch as th

from clip_guided_diffusion_b200._lib import OP
from clip_guided_diffusion_b200.plan import _DT, Buf

CODE = {v: k for k, v in OP.items()}
ESIZE = {"h": 2, "f": 4, "i32": 4, "u32": 4, "i64": 8}
FLOAT_DT = ("h", "f")
NAN_H = 0x7E00             # fp16 quiet NaN
NAN_F_HI = 0x7FC0          # high word of the fp32 quiet NaN 0x7FC00000 (low word 0)

# op codes whose footprint is stated exactly; every other code falls back to the whole buffers of its pointer slots
EXACT = ("CONV", "GN_STATS", "GN_APPLY", "GN_BWD_STATS", "GN_BWD_APPLY", "GN_FWD_FUSED", "GN_BWD_FUSED", "GN_FWD_GRID", "GN_BWD_GRID",
         "GN_APPLY_EPI", "ADD", "COPY", "POOL2", "UP2", "LN_FWD", "LN_BWD", "ATTN_FWD", "ATTN_BWD", "NCHW_TO_PM", "PM_TO_NCHW",
         "ATTNPOOL_EMBED_FWD", "ATTNPOOL_EMBED_BWD", "LINEAR_SMALL")


@dataclass
class Region:
    """Elements of type `dt` at buffer `buf`, element offset `eoff` (in units of buf.dt, like a plan pointer), laid out as
    `shape` / `strides` (elements of dt) -- or, with `idx`, the listed element offsets."""
    buf: Buf
    eoff: int
    dt: str
    shape: tuple
    strides: tuple
    slot: int
    idx: Optional[th.Tensor] = None

    @property
    def empty(self):
        return (self.idx is not None and self.idx.numel() == 0) or any(int(s) == 0 for s in self.shape)

    @property
    def base_byte(self):
        return self.buf.off + self.eoff * _DT[self.buf.dt][0]

    def _k(self):
        return ESIZE[self.dt] // 2

    def extent(self):
        """(first, last) byte the region touches"""
        k = ESIZE[self.dt]
        if self.idx is not None:
            return self.base_byte + int(self.idx.min()) * k, self.base_byte + int(self.idx.max()) * k + k - 1
        last = sum((int(n) - 1) * int(s) for n, s in zip(self.shape, self.strides))
        return self.base_byte, self.base_byte + last * k + k - 1

    def _widx(self, device):
        k = self._k()
        return (self.base_byte // 2 + self.idx.to(device)[:, None] * k + th.arange(k, device=device)).reshape(-1)

    def words(self, t):
        """view (strided) of a word-granular arena tensor t covering this region"""
        k = self._k()
        return t.as_strided(tuple(int(n) for n in self.shape) + (k,), tuple(int(s) * k for s in self.strides) + (1,), self.base_byte // 2)

    def get(self, t):
        return t[self._widx(t.device)] if self.idx is not None else self.words(t).clone()

    def put(self, t, src):
        """copy this region from word tensor src into word tensor t"""
        if self.idx is not None:
            w = self._widx(t.device)
            t[w] = src[w]
        else:
            self.words(t).copy_(self.words(src))

    def fill(self, t, v):
        if self.idx is not None:
            t[self._widx(t.device)] = v
        else:
            self.words(t).fill_(v)

    def where(self, elem):
        """coordinates of element `elem` (of buf, in units of dt) in this region, or None"""
        rel = elem - self.eoff
        if self.idx is not None or self.dt != self.buf.dt or rel < 0:
            return None
        coords = []
        for n, s in sorted(zip(self.shape, self.strides), key=lambda a: -a[1]):
            c = rel // s if s else 0
            coords.append(int(c))
            rel -= c * s
        return tuple(coords) if rel == 0 else None


@dataclass
class Footprint:
    reads: list = field(default_factory=list)
    writes: list = field(default_factory=list)


def _whole(buf: Buf, slot: int) -> Region:
    return Region(buf, 0, buf.dt, (buf.numel,), (1,), slot)


def footprint(op, arena: Optional[th.Tensor] = None) -> Footprint:
    """read / write sets of one plan op from its i / p fields (include/cgd_b200.h).  `arena` is needed only by ops whose
    footprint is data in the arena (LINEAR_SMALL's scatter table)."""
    name = CODE[op.code]
    i = list(op.i) + [0] * (24 - len(op.i))
    p = list(op.p) + [None] * (12 - len(op.p))
    fl = op.flags
    fp = Footprint()

    def reg(slot, dt, shape, strides=None):
        if p[slot] is None:
            return None
        if strides is None:  # contiguous
            strides, acc = [], 1
            for n in reversed(shape):
                strides.insert(0, acc)
                acc *= n
        return Region(p[slot][0], p[slot][1], dt, tuple(shape), tuple(strides), slot)

    def r(slot, dt, shape, strides=None):
        x = reg(slot, dt, shape, strides)
        if x is not None:
            fp.reads.append(x)
        return x

    def w(slot, dt, shape, strides=None, acc=False):
        x = reg(slot, dt, shape, strides)
        if x is not None:
            fp.writes.append(x)
            if acc:  # accumulating ops read their output
                fp.reads.append(x)
        return x

    def scratch(*slots):
        for s in slots:
            if p[s] is not None:
                fp.writes.append(_whole(p[s][0], s))

    def rows(slot, dt, n, C, ld, write=False, acc=False):
        return (w if write else r)(slot, dt, (n, C), (ld, 1), **({"acc": acc} if write else {}))

    if name == "CONV" and not (i[20] or i[21]):
        NB, H, W_, Cin, Cout, Npad, taps = i[:7]
        r(0, "h", (NB, H, W_, Cin), (i[7], i[8], i[9], 1))
        r(1, "h", (Npad, taps * Cin), (i[22] or taps * Cin, 1))
        r(2, "f", (Cout,))
        r(3, "h", (NB, H, W_, Cout), (i[13], i[14], i[15], 1))
        w(4, "f" if fl & 1 else "h", (NB, H, W_, Cout), (i[10], i[11], i[12], i[19] if i[19] > 1 else 1))
        scratch(5, 6, 7)  # split-K workspace, split-K barriers, epilogue statistics
    elif name.startswith("GN_") and name in EXACT:
        N, HW, C = i[:3]

        def affine(sg, sb, se):
            r(sg, "f", (C,))
            r(sb, "f", (C,))
            r(se, "f", (N * 2 * C,))

        if name == "GN_STATS":
            rows(0, "h", N * HW, C, i[3])
            w(2, "f", (N * 64,))
            scratch(1, 3)
        elif name == "GN_APPLY":
            rows(0, "h", N * HW, C, i[3])
            r(1, "f", (N * 64,))
            affine(2, 3, 4)
            rows(5, "h", N * HW, C, i[5], write=True)
        elif name in ("GN_FWD_FUSED", "GN_FWD_GRID", "GN_APPLY_EPI"):
            rows(0, "h", N * HW, C, i[3])
            affine(1, 2, 3)
            rows(4, "h", N * HW, C, i[4], write=True)
            w(5, "f", (N * 64,))
            if name == "GN_FWD_GRID":
                scratch(6, 7)
            if name == "GN_APPLY_EPI":
                fp.reads.append(_whole(p[6][0], 6))  # the producing conv's epilogue statistics
                scratch(7)
        else:  # backward: p0 dy p1 x p2 stats p3 gamma p4 beta p5 emb
            ld_dy, ldx = i[3], i[4]
            rows(0, "h", N * HW, C, ld_dy)
            rows(1, "h", N * HW, C, ldx)
            r(2, "f", (N * 64,))
            affine(3, 4, 5)
            if name == "GN_BWD_STATS":
                w(7, "f", (N * 64,))
                scratch(6, 8)
            elif name == "GN_BWD_APPLY":
                r(6, "f", (N * 64,))
                rows(7, "h", N * HW, C, i[6], write=True, acc=bool(fl & 2))
            else:  # GN_BWD_FUSED, GN_BWD_GRID
                rows(6, "h", N * HW, C, i[5], write=True, acc=bool(fl & 2))
                if name == "GN_BWD_GRID":
                    scratch(7, 8, 9)  # partials, barrier, the shared d xhat scratch
    elif name in ("POOL2", "UP2"):
        N, H, W_, C, ldx, ldy = i[:6]
        rows(0, "h", N * H * W_, C, ldx)
        rows(1, "h", N * H * W_ // 4 if name == "POOL2" else N * H * W_ * 4, C, ldy, write=True)
    elif name == "ADD":
        n, C, lda, ldb, ldc = i[:5]
        rows(0, "h", n, C, lda)
        rows(1, "h", n, C, ldb)
        rows(2, "h", n, C, ldc, write=True)
    elif name == "COPY":
        n, C, lds, ldd = i[:4]
        rows(0, "h", n, C, lds)
        rows(1, "h", n, C, ldd, write=True)
    elif name in ("ATTN_FWD", "ATTN_BWD"):
        B, heads, T, d = i[:4]
        qkv = (B, heads, T, d), (i[4], i[6], i[5], 1)
        out = (B, heads, T, d), (i[7], i[9], i[8], 1)
        for s in (0, 1, 2):
            r(s, "h", *qkv)
        if name == "ATTN_FWD":
            w(3, "h", *out)
            w(4, "f", (B * heads * T,))
        else:
            r(3, "h", *out)
            r(4, "h", *out)
            r(5, "f", (B * heads * T,))
            for s in (6, 7, 8):
                w(s, "h", *qkv)
            w(9, "f", (B * heads * T,))  # delta workspace
    elif name == "LN_FWD":
        n, wd, ldx, ldy = i[:4]
        rows(0, "h", n, wd, ldx)
        r(1, "f", (wd,))
        r(2, "f", (wd,))
        rows(3, "h", n, wd, ldy, write=True)
        w(4, "f", (n * 2,))
    elif name == "LN_BWD":
        n, wd, ld_dy, ldx, ld_dx = i[:5]
        rows(0, "h", n, wd, ld_dy)
        rows(1, "h", n, wd, ldx)
        r(2, "f", (wd,))
        r(3, "f", (n * 2,))
        rows(4, "h", n, wd, ld_dx, write=True, acc=bool(fl & 2))
    elif name == "NCHW_TO_PM":
        N, C, HW, ld = i[:4]
        r(0, "f", (N * C * HW,))
        w(1, "h", (N * HW * ld,))  # zero-padded to ld channels: the whole row
    elif name == "PM_TO_NCHW":
        N, C, HW, ld = i[:4]
        rows(0, "f" if fl & 1 else "h", N * HW, C, ld)
        w(1, "f", (N * C * HW,), acc=bool(fl & 2))
    elif name == "ATTNPOOL_EMBED_FWD":
        n, HW, C, ldx = i[:4]
        rows(0, "h", n * HW, C, ldx)
        r(1, "f", ((HW + 1) * C,))
        w(2, "h", (n * (HW + 1) * C,))
    elif name == "ATTNPOOL_EMBED_BWD":
        n, HW, C, ld = i[:4]
        r(0, "h", (n * (HW + 1) * C,))
        rows(1, "h", n * HW, C, ld, write=True, acc=bool(fl & 2))
    elif name == "LINEAR_SMALL":
        M, K, N, ldx, ldy = i[:5]
        rows(0, "h" if fl & 4 else "f", M, K, ldx)
        r(1, "h" if fl & 16 else "f", (N, K))
        r(2, "f", (N,))
        ydt = "h" if fl & 8 else "f"
        if p[4] is not None:  # scatter table: column n of row m lands at element tab[n, 0] + m * tab[n, 1] of p3
            if arena is None:
                raise ValueError("LINEAR_SMALL with a scatter table: footprint() needs the arena")
            r(4, "i32", (N * 2,))
            tb, te = p[4]
            o = tb.off + te * _DT[tb.dt][0]
            tab = arena[o:o + N * 8].view(th.int32).view(N, 2).long().cpu()
            idx = (tab[None, :, 0] + th.arange(M)[:, None] * tab[None, :, 1]).reshape(-1)
            x = Region(p[3][0], p[3][1], ydt, (idx.numel(),), (1,), 3, idx=idx)
            fp.writes.append(x)
            if fl & 2:
                fp.reads.append(x)
        else:
            rows(3, ydt, M, N, ldy, write=True, acc=bool(fl & 2))
    else:
        for s, ptr in enumerate(p):
            if ptr is not None:
                fp.reads.append(_whole(ptr[0], s))
                fp.writes.append(_whole(ptr[0], s))
    fp.reads = [x for x in fp.reads if not x.empty]
    fp.writes = [x for x in fp.writes if not x.empty]
    return fp


def execution_order(plan) -> list:
    """op indices in the order one guided step executes them (UNet forward, p_mean_variance, cutouts, CLIP forward / backward,
    losses, UNet dgrad, update), then every op no segment covers"""
    segs = [("unet_emb", "unet_bwd"), ("pmv", "cond"), ("cut_fwd", "sph"), ("vit_fwd", "vit_bwd"), ("sph", "cut_bwd"),
            ("vit_bwd", "vit_end"), ("cut_bwd", "guide"), ("guide", "final"), ("unet_bwd", "unet_end"), ("final", "upd_anc_g"),
            ("upd_anc_g", "upd_anc"), ("upd_anc", "upd_ddim_g"), ("upd_ddim_g", "upd_ddim"), ("upd_ddim", "engine_end")]
    m, order, seen = plan.marks, [], set()
    for a, b in segs:
        if a in m and b in m:
            for k in range(m[a], m[b]):
                if k not in seen:
                    seen.add(k)
                    order.append(k)
    return order + [k for k in range(len(plan.ops)) if k not in seen]


class Guard:
    """Write guard + read poison over one plan's arena.  run_op(k) executes op k on that arena and returns when it is done."""

    def __init__(self, plan, run_op: Callable[[int], None], footprint_fn=footprint, atomic_ops=(), atol_rel=1e-4):
        self.plan, self.run_op, self.footprint_fn = plan, run_op, footprint_fn
        self.atomic_ops, self.atol_rel = set(atomic_ops), atol_rel
        A = plan.arena
        assert A.dtype == th.uint8 and A.numel() % 2 == 0
        self.A = A.view(th.int16)
        self.S = th.empty_like(self.A)   # clean state before the op
        self.Pb = th.empty_like(self.A)  # poisoned state before the op
        dev = A.device
        self.bufs = sorted(plan.bufs, key=lambda b: b.off)
        self.offs = [b.off for b in self.bufs]
        # poison pattern and mask: NaN in every fp16 / fp32 buffer and in every gap between buffers
        self.pat = th.full_like(self.A, NAN_H)
        self.pmask = th.ones(self.A.numel(), dtype=th.bool, device=dev)
        for b in self.bufs:
            a, e = b.off // 2, (b.off + b.nbytes) // 2
            if b.dt == "f":
                self.pat[a:e].view(-1, 2)[:, 0] = 0
                self.pat[a:e].view(-1, 2)[:, 1] = NAN_F_HI
            elif b.dt not in FLOAT_DT:
                self.pmask[a:e] = False

    # ------------------------------------------------------------------ reporting
    def locate(self, word: int, fp: Footprint) -> str:
        byte = 2 * word
        j = bisect.bisect_right(self.offs, byte) - 1
        if j < 0:
            return f"byte {byte}: before the first buffer"
        b = self.bufs[j]
        if byte >= b.off + b.nbytes:
            return f"byte {byte}: alignment gap, {byte - b.off - b.nbytes} B past the end of {b.name!r}"
        elem = (byte - b.off) // _DT[b.dt][0]
        where = [f"p{x.slot}{c}" for x in fp.reads + fp.writes if x.buf is b and (c := x.where(elem)) is not None]
        return f"{b.name!r}[{elem}]" + (f" = {', '.join(dict.fromkeys(where))}" if where else "")

    def _strays(self, after, before, fp, k, run):
        ne = after != before
        for x in fp.writes:
            x.fill(ne, False)
        if not bool(ne.any()):
            return None
        idx = th.nonzero(ne).flatten()
        op = self.plan.ops[k]
        return dict(kind="stray write", op=k, code=CODE[op.code], tag=op.tag, run=run, words=int(idx.numel()),
                    first=[self.locate(int(w), fp) for w in idx[:6].tolist()])

    def _overruns(self, fp, k):
        out = []
        for x in fp.reads + fp.writes:
            op = self.plan.ops[k]
            if x.idx is not None:  # a scatter spans several buffers by design: every element must still lie inside one
                byte = x.base_byte + x.idx * ESIZE[x.dt]
                offs = th.tensor(self.offs)
                ends = th.tensor([b.off + b.nbytes for b in self.bufs])
                j = th.searchsorted(offs, byte, right=True) - 1
                if bool((j < 0).any()) or bool((byte + ESIZE[x.dt] > ends[j.clamp(min=0)]).any()):
                    out.append(dict(kind="scatter outside the buffers", op=k, code=CODE[op.code], tag=op.tag, slot=x.slot))
                continue
            lo, hi = x.extent()
            if lo < x.buf.off or hi >= x.buf.off + x.buf.nbytes:
                out.append(dict(kind="footprint outside its buffer", op=k, code=CODE[op.code], tag=op.tag, slot=x.slot, buf=x.buf.name,
                                bytes=(lo - x.buf.off, hi - x.buf.off), nbytes=x.buf.nbytes))
        return out

    def _outputs(self, fp):
        return [x.get(self.A) for x in fp.writes]

    @staticmethod
    def _as_float(x, words):
        if x.dt == "h":
            return words.view(th.float16).float()
        if x.dt == "f":
            return words.contiguous().view(th.float32).float()
        return None

    def _diff(self, fp, a, b, tolerant):
        """first output region where runs a and b differ: (slot, buffer, words that differ, NaN in a) or None"""
        for x, u, v in zip(fp.writes, a, b):
            if th.equal(u, v):
                continue
            fu, fv = self._as_float(x, u), self._as_float(x, v)
            if tolerant and fu is not None:
                fin = th.isfinite(fv)
                if th.equal(th.isfinite(fu), fin) and bool(((fu - fv).abs()[fin] <= self.atol_rel * (float(fv[fin].abs().max()) if bool(fin.any()) else 0.0) + 1e-6).all()):
                    continue
            nan = bool((~th.isfinite(fu)).any() & th.isfinite(fv).all()) if fu is not None else False
            return dict(slot=x.slot, buf=x.buf.name, words=int((u != v).sum()), nan_in_first=nan)
        return None

    # ------------------------------------------------------------------ one op
    def check_op(self, k: int) -> list:
        A, S, Pb = self.A, self.S, self.Pb
        op = self.plan.ops[k]
        fp = self.footprint_fn(op, self.plan.arena)
        fails = self._overruns(fp, k)
        S.copy_(A)
        # poisoned run
        th.where(self.pmask, self.pat, A, out=A)
        for x in fp.reads + fp.writes:
            x.put(A, S)
        Pb.copy_(A)
        self.run_op(k)
        f = self._strays(A, Pb, fp, k, "poisoned")
        if f:
            fails.append(f)
        out_p = self._outputs(fp)
        # clean run
        A.copy_(S)
        self.run_op(k)
        f = self._strays(A, S, fp, k, "clean")
        if f:
            fails.append(f)
        out_c = self._outputs(fp)
        tolerant = CODE[op.code] in self.atomic_ops
        d = self._diff(fp, out_p, out_c, tolerant)
        if d is not None:
            # stray read or race?  Run clean once more: a clean-twice mismatch is a race
            A.copy_(S)
            self.run_op(k)
            d2 = self._diff(fp, self._outputs(fp), out_c, tolerant)
            kind = "not reproducible (race)" if d2 is not None else "stray read"
            fails.append(dict(kind=kind, op=k, code=CODE[op.code], tag=op.tag, **(d2 or d)))
        return fails

    def check(self, ops) -> list:
        fails = []
        for k in ops:
            fails += self.check_op(k)
        return fails


def format_failures(fails, limit=30) -> str:
    return "\n".join(str(f) for f in fails[:limit]) + (f"\n... {len(fails) - limit} more" if len(fails) > limit else "")
