"""Every instantiation of the tcgen05 convolution kernel (conv_umma.cu) on its own, with several tiles per CTA.

The kernel is persistent: a launch has min(tiles, SMs) CTAs and each CTA walks its tiles round-robin (the arg-max
variants: one contiguous range).  At test sizes that is one tile per CTA, and the code of a CTA's second and later
tiles never runs: the straight-line MMA issue over stationary weights, the second TMEM accumulator stage, ring
wrap-around, the tile-coordinate carries, the arg-max running maximum and its flush when a range crosses into another
image, CTAs left idle.  mvlm_debug_conv_max_ctas caps the grid (the kernels are unchanged), and every case runs
uncapped, on one CTA, and under a cap chosen so that CTAs run >= 3 tiles, the tiles do not divide evenly, ranges
straddle images and M tiles and (arg-max) some CTAs are idle; mvlm_debug_conv_describe confirms each of these.

Every instantiation of the library's table (mvlm_debug_conv_variants) gets a small seeded case that describe
confirms selects it, and:
  * every output, fp32 map and arg-max key is bit-identical across the caps: which CTA computes a tile must not
    change its bits;
  * every element is within plan_ref.bound of an fp64 reference computed from the same bf16 operands:
    2^-8 |ref| (bf16 output rounding; none for fp32 maps) + 2^-14 A, A = the same computation on absolute values.
    Pooled outputs are compared with the pool of the reference (and of the bound); what the kernel computes from its
    own stored bf16 values is checked against those values: pools bit-exact, activations to one bf16 rounding;
  * fp32 maps of four up=(2, 2, a, b) phases go to one buffer and one set of keys (atomicMax): the keys are those of
    the first maximum of the map in row-major order, and the arg-max-only variants give the keys of the exact search;
  * input channels [cin, in_cs) and residual channels outside the slice read are NaN, and no output is; every output
    buffer starts NaN and stays NaN outside its slice, and outside the pixels of the phases run so far;
  * for the first case of each family the reference perturbed (input shifted by a pixel, a neighbouring channel's
    BatchNorm, a residual dropped, another phase's weights) fails the bound.
All cases run once per module (fixture variant_runs); test_conv_variant[v] reports the cases of instantiation v, and
test_variant_table_covered checks that the cases cover the table and prints, per instantiation, the tiles per CTA
reached and the worst err / bound.

Measured on one NVIDIA B200 at a 1000 W power limit: 4.6 s for the file; worst err / bound 0.98 for the bf16 outputs
(the 2^-8 term is the worst-case rounding, so large tensors sit near 1), 0.006 for the fp32 maps; every perturbed
reference fails by 4.6e3 x its bound or more.
"""
import math

import pytest
import torch

from plan_ref import bf16_rn, bound, conv, maxpool, ordered_keys, up2

pytestmark = pytest.mark.gpu

# feature flags of conv_epilogue.cuh
F_PRE, F_RES1, F_RES2, F_RAW, F_POST, F_F32, F_ARGMAX = 1, 2, 4, 8, 16, 32, 64
F_MID, F_POOL, F_UP, F_M64, F_POST2, F_POOLX, F_STAT = 128, 256, 512, 1024, 2048, 4096, 8192
_NAMES = {F_MID: "MID", F_POOL: "POOL", F_POOLX: "POOLX", F_POST2: "POST2", F_UP: "UP", F_PRE: "PRE", F_RES1: "RES1",
          F_RES2: "RES2", F_RAW: "RAW", F_POST: "POST", F_F32: "F32", F_ARGMAX: "ARGMAX", F_M64: "M64", F_STAT: "STAT"}


def vname(v):
    return "|".join(n for b, n in _NAMES.items() if v & b)


# MVLM_CONV_VARIANTS of conv_umma.cu: combinations instantiated at M = 128, M = 64 (.ws) and M = 64 + STAT ...
ALL_M = [F_PRE | F_RES1 | F_RAW | F_POST, F_PRE | F_RES1 | F_RAW, F_RES1 | F_RAW | F_POST, F_RES1 | F_RAW, F_RAW,
         F_F32, F_F32 | F_ARGMAX, F_MID | F_PRE | F_POST,
         F_POOL | F_PRE | F_RES1 | F_RAW | F_POST, F_POOL | F_RES1 | F_RAW | F_POST, F_POOL | F_RAW,
         F_UP | F_PRE | F_RES1 | F_RAW | F_POST, F_UP | F_PRE | F_RES1 | F_RAW, F_UP | F_RES1 | F_RAW | F_POST,
         F_UP | F_RES1 | F_RAW,
         F_POST2 | F_PRE | F_RES1 | F_RAW | F_POST, F_POST2 | F_RES1 | F_RAW | F_POST,
         F_POOLX | F_PRE | F_RES1 | F_RAW | F_POST, F_POOLX | F_RES1 | F_RAW | F_POST]
# ... and at M = 128 only
M128_ONLY = [F_PRE, F_RES1 | F_RES2 | F_RAW | F_POST, F_ARGMAX, F_ARGMAX | F_STAT, F_PRE | F_RES1 | F_RES2 | F_RAW | F_POST,
             F_POOLX | F_RES1 | F_RES2 | F_RAW | F_POST]
VARIANTS = [f | m for f in ALL_M for m in (0, F_M64, F_M64 | F_STAT)] + M128_ONLY

# (H, W): output tiles of 32, 16, 8 and 4 rows (8 at M <= 64); every one ragged in both directions, all even (pools)
SHAPES = [(68, 36), (26, 36), (14, 36), (6, 86)]
# channel offsets of the slices written and read
CO = {"pre": 8, "raw": 16, "post": 24, "aux1": 8, "aux2": 16, "res1": 8, "res2": 24, "res_up": 16}


def cases(v):
    """(n, h, w, cin, cout_pad, k) of the cases of instantiation v."""
    i = VARIANTS.index(v)
    h, w = SHAPES[i % 4]
    n = 2 + i % 2
    head = v & (F_F32 | F_ARGMAX)
    if v == F_ARGMAX | F_STAT:
        # 2 x 2 taps over stationary weights at M = 128: K steps per chunk 4 + 1 and 4 + 2
        return [(2, 26, 36, 80, 80, 2), (3, 68, 36, 96, 96, 2)]
    if v & F_STAT:
        # .ws, 3 x 3 taps over stationary weights (one chunk): K steps 1, 2, 3 (ring path) and 4
        return [(n, h, w, (16, 32, 48, 64)[i % 4], (64, 32, 48, 16)[(i // 3) % 4], 3)]
    if v & F_M64:
        k = (1, 2, 3)[i % 3]
        cin = (96, 128, 112, 80)[i % 4] if k == 3 else (16, 48, 96, 144)[i % 4]  # 3 x 3: streamed weights
        return [(n, h, w, cin, (32, 64, 48, 16)[(i // 3) % 4], k)]
    k = 3 if v == F_ARGMAX else (3, 1, 2)[i % 3]  # F_ARGMAX with 2 x 2 stationary weights would be F_ARGMAX | F_STAT
    cin = (64, 80, 32, 112, 128, 16, 48, 160)[i % 8]
    cout = (128, 256, 96, 80)[i % 4]
    return [(n, h, w, cin, 128 if head and cout > 128 else cout, k)]


def family(v):
    for bit, fam in ((F_F32 | F_ARGMAX, "head"), (F_MID, "stem"), (F_POOL, "pool"), (F_POOLX, "aux2"), (F_POST2, "aux1"),
                     (F_UP, "up-residual"), (F_RES2, "two residuals"), (F_PRE | F_POST, "rb conv")):
        if v & bit:
            return fam
    return "raw"


def teeth(v):
    """The perturbation the first case of v's family must notice (None: not this case)."""
    fam = family(v)
    if VARIANTS.index(v) != min(VARIANTS.index(u) for u in VARIANTS if family(u) == fam):
        return None
    return {"head": "phase", "stem": ("bn", "mid"), "pool": "shift_in", "aux2": ("bn", "post"), "aux1": ("drop", "res1"),
            "up-residual": ("drop", "res_up"), "two residuals": ("drop", "res2"), "rb conv": ("bn", "post"),
            "raw": "shift_in"}[fam]


def schedule(total, grid, contiguous):
    """The tiles of every CTA: round-robin, or contiguous ranges of ceil(total / grid) (arg-max variants)."""
    if contiguous:
        per = -(-total // grid)
        return [range(b * per, min(total, b * per + per)) for b in range(grid)]
    return [range(b, total, grid) for b in range(grid)]


def tiles_per_cta(total, grid):
    return -(-total // grid)


def schedule_facts(total, grid, n_img, n_nt, contiguous):
    rs = schedule(total, grid, contiguous)
    tpi = total // n_img
    return {"three_tiles": tiles_per_cta(total, grid) >= 3, "uneven": total % grid != 0,
            "straddles_images": any(len({t // tpi for t in r}) > 1 for r in rs),
            "straddles_m_tiles": n_nt == 1 or any(len({t % n_nt for t in r}) > 1 for r in rs),
            "idle_ctas": not contiguous or any(len(r) == 0 for r in rs)}


def pick_cap(total, n_img, n_nt, contiguous):
    """The largest cap under which CTAs run >= 3 tiles, unevenly, across images and M tiles, some idle (arg-max)."""
    for g in range(total // 3, 1, -1):
        if all(schedule_facts(total, g, n_img, n_nt, contiguous).values()):
            return g
    raise AssertionError(f"no cap gives the schedule the test needs for {total} tiles over {n_img} images")


def _ratio(got, want, bnd):
    """max |got - want| / bnd, an exact zero counting 0."""
    err = (got - want).abs()
    return torch.where(err == 0, 0.0, err / bnd).max().item()


def _bits(t):
    return t.view({2: torch.int16, 4: torch.int32, 8: torch.int64}[t.element_size()])


class Case:
    def __init__(self, v, n, h, w, cin, cout, k, seed):
        self.v, self.n, self.h, self.w, self.cin, self.cout, self.k = v, n, h, w, cin, cout, k
        self.head = v & (F_F32 | F_ARGMAX) != 0
        self.cout_real = cout - 7 if self.head else cout
        self.n_nt = 1 if cout <= 64 else -(-cout // 128)
        self.in_cs = cin + 8
        g = torch.Generator(device="cuda").manual_seed(seed)

        def rnd(*shape):
            return torch.randn(shape, generator=g, device="cuda")

        def poisoned(hh, ww, co):
            """bf16 (n, hh, ww, co + cout + 8): NaN except the slice [co, co + cout)."""
            t = torch.full((n, hh, ww, co + cout + 8), float("nan"), device="cuda", dtype=torch.bfloat16)
            t[..., co:co + cout] = rnd(n, hh, ww, cout).to(torch.bfloat16)
            return t

        self.x = torch.full((n, h, w, self.in_cs), float("nan"), device="cuda", dtype=torch.bfloat16)
        self.x[..., :cin] = rnd(n, h, w, cin).to(torch.bfloat16)
        self.res = {}
        if v & F_RES1:
            self.res["res1"] = poisoned(h, w, CO["res1"])
        if v & F_RES2:
            self.res["res2"] = poisoned(h, w, CO["res2"])
        if v & F_UP:
            self.res["res_up"] = poisoned(h // 2, w // 2, CO["res_up"])
        # four phases (one weight set each) for the heads, one weight set otherwise; rows past cout_real are zero
        self.wts = []
        for _ in range(4 if self.head else 1):
            wt = bf16_rn(rnd(cout, cin, k, k) / math.sqrt(cin * k * k))
            wt[self.cout_real:] = 0
            self.wts.append(wt)
        from mvlm_b200 import ops

        self.packed = [ops.pack_conv_weight(wt, cout, cin) for wt in self.wts]
        self.bias = rnd(cout)

        def bn():
            s = (torch.rand((cout,), generator=g, device="cuda") + 0.5) * torch.sign(rnd(cout))
            return s, rnd(cout)

        self.bn = {}
        for bit, term in ((F_MID, "mid"), (F_PRE, "pre"), (F_POST, "post")):
            if v & bit:
                self.bn[term] = bn()
        if v & F_POOLX:
            self.bn["aux"] = bn()
        if v & F_POST2:
            # relu(s * raw + t) with t = -s: the activation nearly cancels where raw is close to 1, so that it shows
            # whether the copy starts from the bf16-rounded raw value
            s, _ = bn()
            self.bn["aux"] = (s, -s)

    # ---- launches ----------------------------------------------------------------------------------------------------
    def phase_offsets(self, p):
        a, b = p // 2, p % 2
        off = {1: (0, 0), 2: (a - 1, b - 1), 3: (a - 2, b - 2)}[self.k]
        return (off[0], off[1]) if self.head else (-(self.k // 2), -(self.k // 2))

    def outputs(self, v):
        """NaN-filled output buffers of instantiation v."""
        n, h, w, c = self.n, self.h, self.w, self.cout

        def buf(hh, ww, co):
            return torch.full((n, hh, ww, co + c + 8), float("nan"), device="cuda", dtype=torch.bfloat16)

        o = {}
        hp, wp = (h // 2, w // 2) if v & F_POOL else (h, w)
        if v & F_PRE:
            o["pre"] = buf(h, w, CO["pre"])
        if v & F_RAW:
            o["raw"] = buf(hp, wp, CO["raw"])
        if v & F_POST:
            o["post"] = buf(hp, wp, CO["post"])
        if v & F_POST2:
            o["aux1"] = buf(h, w, CO["aux1"])
        if v & F_POOLX:
            o["aux1"] = buf(h // 2, w // 2, CO["aux1"])
            o["aux2"] = buf(h // 2, w // 2, CO["aux2"])
        if v & F_F32:
            o["map"] = torch.full((n, self.cout_real, 2 * h, 2 * w), float("nan"), device="cuda")
        if v & F_ARGMAX:
            o["keys"] = torch.zeros((n * self.cout_real,), device="cuda", dtype=torch.int64)
        return o

    def kwargs(self, p, o, v=None):
        v = self.v if v is None else v
        y0, x0 = self.phase_offsets(p)
        kw = dict(cin=self.cin, n_tile=min(self.cout, 128), kh=self.k, kw=self.k, y_off0=y0, x_off0=x0, bias=self.bias)
        if v & F_MID:
            kw["mid"] = self.bn["mid"]
        if v & F_PRE:
            kw["pre"] = (*self.bn["pre"], o["pre"], CO["pre"])
        for r in ("res1", "res2", "res_up"):
            if r in self.res:
                kw[r] = (self.res[r], CO[r])
        if v & F_RAW:
            kw["out_raw"] = (o["raw"], CO["raw"])
        if v & F_POST:
            kw["post"] = (*self.bn["post"], o["post"], CO["post"])
        kw["pool2"] = bool(v & F_POOL)
        if v & F_POST2:
            kw["aux"] = (1, *self.bn["aux"], o["aux1"], CO["aux1"], None, 0)
        if v & F_POOLX:
            kw["aux"] = (2, *self.bn["aux"], o["aux1"], CO["aux1"], o["aux2"], CO["aux2"])
        if v & (F_F32 | F_ARGMAX):
            kw.update(out_f32=o.get("map"), argmax_keys=o.get("keys"), cout_real=self.cout_real,
                      up=(2, 2, p // 2, p % 2))
        return kw

    def describe(self, v=None):
        from mvlm_b200 import ops

        v = self.v if v is None else v
        return ops.conv_describe(self.x, self.packed[0], **self.kwargs(0, self.outputs(v), v))

    def run(self, tag, v=None):
        """All phases of instantiation v (default: the case's own) under the current cap; the outputs."""
        from mvlm_b200 import ops

        v = self.v if v is None else v
        o = self.outputs(v)
        for p in range(len(self.packed)):
            ops.conv2d_bf16(self.x, self.packed[p], **self.kwargs(p, o, v))
            torch.cuda.synchronize()
            if "map" in o:
                # the pixels of the phases not run yet are untouched
                for q in range(p + 1, len(self.packed)):
                    assert torch.isnan(o["map"][:, :, q // 2::2, q % 2::2]).all(), \
                        f"{tag}: phase {p} wrote pixels of phase {q}"
        return o

    # ---- fp64 reference ----------------------------------------------------------------------------------------------
    def reference(self, p=0, perturb=None):
        x = self.x[..., :self.cin].double()
        if perturb == "shift_in":
            x = torch.roll(x, 1, dims=2)
        w = self.wts[(p + 1) % 4 if perturb == "phase" else p].double()
        y0, x0 = self.phase_offsets(p)
        b = self.bias.double()
        v = conv(x, w, y0, x0) + b
        A = conv(x.abs(), w.abs(), y0, x0) + b.abs()
        terms = {t: (s.double(), sh.double()) for t, (s, sh) in self.bn.items()}
        if perturb and perturb[0] == "bn":  # a neighbouring channel's BatchNorm
            terms[perturb[1]] = tuple(u.roll(1) for u in terms[perturb[1]])

        def affine(term, val, a):
            s, t = terms[term]
            return torch.relu(val * s + t), a * s.abs() + t.abs()

        out = {}
        if "mid" in terms:
            v, A = affine("mid", v, A)
        if "pre" in terms:
            out["pre"] = affine("pre", v, A)
        for r, t in self.res.items():
            if perturb == ("drop", r):
                continue
            t = t[..., CO[r]:CO[r] + self.cout].double()
            t = up2(t) if r == "res_up" else t
            v, A = v + t, A + t.abs()
        out["raw"] = (v, A)
        if "post" in terms:
            out["post"] = affine("post", v, A)
        return out

    # ---- checks ------------------------------------------------------------------------------------------------------
    def slices(self, o):
        """{name: the written slice}: bf16 outputs (double), the fp32 map, the keys."""
        s = {}
        for name, t in o.items():
            if name in CO:
                s[name] = t[..., CO[name]:CO[name] + self.cout]
            else:
                s[name] = t
        return s

    def check_sentinels(self, o, tag):
        for name, t in o.items():
            if name in CO:
                co = CO[name]
                assert torch.isnan(t[..., :co].float()).all() and torch.isnan(t[..., co + self.cout:].float()).all(), \
                    f"{tag}: {name} written outside its channel slice"
                assert torch.isfinite(t[..., co:co + self.cout].float()).all(), \
                    f"{tag}: {name} has NaN / inf inside its slice (poisoned channels read, or pixels not written)"
            elif name == "map":
                assert torch.isfinite(t).all(), f"{tag}: fp32 map has NaN / inf after all four phases"

    def check(self, o, refs, tag, perturb=None):
        """Worst err / bound over every output; asserts <= 1 unless perturb is given."""
        s = {k: t.double() if k != "keys" else t for k, t in self.slices(o).items()}
        worst = 0.0

        def cmp(name, got, want, bnd):
            nonlocal worst
            r = _ratio(got, want, bnd)
            worst = max(worst, r)
            assert perturb is not None or r <= 1.0, f"{tag}: {name} off by {r:.3g} x its bound"

        if self.head:
            if "map" in s:
                for p, ref in enumerate(refs):
                    v, A = ref["raw"]
                    want = v[..., :self.cout_real].permute(0, 3, 1, 2)
                    bnd = bound(want, A[..., :self.cout_real].permute(0, 3, 1, 2), bf16_out=False)
                    cmp(f"fp32 map phase {p}", s["map"][:, :, p // 2::2, p % 2::2], want, bnd)
            return worst
        ref = refs[0]
        if "pre" in s:
            cmp("out_pre", s["pre"], ref["pre"][0], bound(*ref["pre"]))
        if self.v & F_POOL:
            v, A = ref["raw"]
            cmp("pooled out_raw", s["raw"], maxpool(v), maxpool(bound(v, A)))
        else:
            if "raw" in s:
                cmp("out_raw", s["raw"], ref["raw"][0], bound(*ref["raw"]))
            if "post" in s:
                cmp("out_post", s["post"], ref["post"][0], bound(*ref["post"]))
        if perturb is not None:
            return worst
        if self.v & F_POOL and "post" in s:
            self.check_act(tag, "pooled out_post", s["post"], s["raw"], self.bn["post"])
        if self.v & F_POST2:
            self.check_act(tag, "out_aux1", s["aux1"], s["raw"], self.bn["aux"])
        if self.v & F_POOLX:
            assert torch.equal(s["aux1"], maxpool(s["raw"])), f"{tag}: pooled copy out_aux1 differs from max-pool(out_raw)"
            self.check_act(tag, "out_aux2", s["aux2"], s["aux1"], self.bn["aux"])
        return worst

    @staticmethod
    def check_act(tag, name, got, x, st):
        """relu(s * x + t) of the kernel's own stored bf16 values, to one bf16 rounding."""
        s, t = (u.double() for u in st)
        ref = torch.relu(x * s + t)
        err = (got - ref).abs()
        bnd = 2.0 ** -8 * ref.abs() + 2.0 ** -20 * ((x * s).abs() + t.abs())
        assert (err <= bnd).all(), f"{tag}: {name} off by {(err / bnd).max().item():.3g} x its bound"

    def check_keys(self, o, exact_keys, tag):
        got = o["keys"].view(self.n, self.cout_real)
        if exact_keys is not None:
            assert torch.equal(got, exact_keys), f"{tag}: arg-max keys differ from those of the exact search"
            return
        m = o["map"].view(self.n, self.cout_real, -1)
        idx = torch.arange(m.shape[-1], device="cuda").expand_as(m)
        want = ordered_keys(m, idx).max(-1).values
        assert torch.equal(got ^ (-(2 ** 63)), want), \
            f"{tag}: arg-max keys differ from the first maximum of the fp32 maps"


def _run_case(v, case, ci, set_cap):
    n, h, w, cin, cout, k = case
    c = Case(v, n, h, w, cin, cout, k, seed=1000 + 10 * VARIANTS.index(v) + ci)
    name = f"{vname(v)} case {ci} {case}"
    set_cap(0)
    d = c.describe()
    assert d.variant == v, f"{name}: selects {vname(d.variant) if d.variant >= 0 else 'nothing'}"
    assert d.tail == (cin % 64 if cin % 64 in (16, 32) else 0), name
    contiguous = bool(v & F_ARGMAX)
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    assert d.total_tiles <= n_sm and d.grid == d.total_tiles, f"{name}: the uncapped grid must run one tile per CTA"
    mid = pick_cap(d.total_tiles, n, c.n_nt, contiguous)
    refs = [c.reference(p) for p in range(len(c.wts))]
    # the exact search's keys for the arg-max-only variants (their fp32-map sibling, uncapped)
    exact_keys = None
    if v & F_ARGMAX and not v & F_F32:
        ev = F_F32 | F_ARGMAX
        assert c.describe(ev).variant == ev
        eo = c.run(f"{name} exact search", ev)
        c.check_keys(eo, None, f"{name} exact search")
        exact_keys = eo["keys"].view(n, c.cout_real)
    first, worst, tiles = None, 0.0, []
    for cap in (0, 1, mid):
        tag = f"{name} cap {cap or 'off'}"
        set_cap(cap)
        dc = c.describe()
        assert dc.variant == v and dc.grid == (cap or d.total_tiles), f"{tag}: grid {dc.grid}"
        tiles.append(tiles_per_cta(d.total_tiles, dc.grid))
        if cap == mid:
            facts = schedule_facts(d.total_tiles, dc.grid, n, c.n_nt, contiguous)
            assert all(facts.values()), f"{tag}: schedule {facts}"
        o = c.run(tag)
        c.check_sentinels(o, tag)
        worst = max(worst, c.check(o, refs, tag))
        if "keys" in o:
            c.check_keys(o, exact_keys, tag)
        if first is None:
            first = o
        else:
            for key, t in o.items():
                assert torch.equal(_bits(t), _bits(first[key])), f"{tag}: {key} not bit-identical to the uncapped run"
    set_cap(0)
    p = teeth(v) if ci == 0 else None
    if p is not None:
        bad = [c.reference(q, perturb=p) for q in range(len(c.wts))]
        r = c.check(first, bad, name, perturb=p)
        print(f"teeth {family(v)} ({vname(v)}): {p} -> {r:.3g} x bound")
        assert r > 1.0, f"{name}: the reference perturbed by {p} still passes ({r:.3g} x bound)"
    return dict(tiles=tiles, worst=worst, tile_h=d.tile_h, tail=cin % 64, n_nt=c.n_nt, k=k, cout=cout,
                ragged_w=w % 8 != 0, ragged_h=h % d.tile_h != 0, caps=(0, 1, mid), total=d.total_tiles)


@pytest.fixture(scope="module")
def variant_runs(lib):
    """Every case of every instantiation, run once for the module: {instantiation: [coverage of each case], or the
    exception its cases raised}.  The coverage test needs all of them, so they are run together here rather than by
    the parametrised tests in turn, whichever of the tests are selected.  The grid cap is reset to 0 afterwards."""
    from mvlm_b200 import ops

    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    runs = {}
    try:
        for v in VARIANTS:
            try:
                runs[v] = [_run_case(v, case, ci, ops.set_conv_max_ctas) for ci, case in enumerate(cases(v))]
            except Exception as e:  # reported by test_conv_variant[v]; the other instantiations still run
                runs[v] = e
        yield runs
    finally:
        ops.set_conv_max_ctas(0)


@pytest.mark.parametrize("v", VARIANTS, ids=vname)
def test_conv_variant(variant_runs, v):
    if isinstance(variant_runs[v], Exception):
        raise variant_runs[v]


def test_variant_table_covered(variant_runs):
    """The cases cover the library's table and the shapes where kernels go wrong; prints the coverage."""
    from mvlm_b200 import ops

    table = ops.conv_variants()
    assert len(table) == len(set(table)) and set(table) == set(VARIANTS), \
        f"table {sorted(map(vname, set(table) ^ set(VARIANTS)))} differs from the test's"
    failed = sorted(vname(v) for v in table if isinstance(variant_runs[v], Exception))
    assert not failed, f"instantiations whose cases failed: {failed}"
    runs = [r for v in table for r in variant_runs[v]]
    for v in table:
        for r in variant_runs[v]:
            keys_only = v & F_ARGMAX and not v & F_F32
            print(f"{vname(v):32s} {r['total']:2d} tiles, per CTA {'/'.join(map(str, r['tiles']))} at caps "
                  f"off/1/{r['caps'][2]:<2d}  " + ("keys = exact search" if keys_only else
                                                   f"worst err/bound {r['worst']:.3g}"))
            assert r["tiles"][2] >= 3, vname(v)
    worst = {}
    for v in table:
        for r in variant_runs[v]:
            worst[family(v)] = max(worst.get(family(v), 0.0), r["worst"])
    for fam, wr in sorted(worst.items()):
        print(f"family {fam}: worst err/bound {wr:.3g}")
    assert {r["tile_h"] for r in runs} >= {32, 16, 8, 4}
    assert {r["tail"] for r in runs} >= {0, 16, 32, 48}
    assert {r["n_nt"] for r in runs} >= {1, 2}
    assert {r["k"] for r in runs} >= {1, 2, 3}
    assert any(r["cout"] <= 32 for r in runs) and any(32 < r["cout"] <= 64 for r in runs)
    assert any(r["ragged_w"] for r in runs) and any(r["ragged_h"] for r in runs)
