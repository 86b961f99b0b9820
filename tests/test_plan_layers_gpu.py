"""The CNN plan launch by launch on the device, each launch against an fp64 reference fed the plan's own inputs.

The real plan (default packed workspace, so that reuse bugs show) runs op by op through mvlm_debug_hourglass_run_op.
For every op:
  * before it runs, every input operand's region equals, bit for bit, the tensor its producer wrote (captured when the
    producer ran): a wrong buffer or a clobbered one fails here, naming the op, the operand and the tensor;
  * after it runs, every output is compared element by element with tests/plan_ref.py's fp64 reference computed from
    the captured inputs (teacher forcing: each launch is judged alone, bf16 chaos does not accumulate).  The bound is
    derived from the arithmetic: |got - ref| <= 2^-8 |ref| (the bf16 output rounding; none for the fp32 heat maps)
    + c * A, A = conv(|x|, |w|) (+ |bias|, + |residuals|, times |s| (+ |t|) for every BatchNorm the output passes
    through), c = 2^-14 for the fp32 tensor-core accumulation, + 2^-16 for the stem's hi / lo image split.  Outputs
    the kernels compute from their own bf16 values (max-pools, pooled and second activations) are checked against the
    plan's own stored values: pools bit-exact, activations to one bf16 rounding;
  * nothing outside its recorded output slices changed in the whole workspace.
The fused arg-max keys equal, after every conv11 phase, the running maximum over the plan's own fp32 maps so far, and
the peaks equal the keys' decoding exactly.  For one op of each family, the same comparison fails when the reference is
perturbed (a neighbouring BatchNorm, a residual slice shifted by 8 channels, the input shifted by a pixel, the bias
dropped, another phase's weights), so the bound is tight enough to see such a mistake.

Measured on one NVIDIA B200 at a 1000 W power limit (see DESIGN.md section 5), all six configurations in 9.5 s: the
worst err / bound ratio of the bf16 outputs is 0.98 (the 2^-8 term is the worst-case bf16 rounding, reached by values
just above a power of two, so this ratio sits near 1 from rounding alone), of the fp32 heat maps 0.0044; the fraction
of bf16 outputs bit-equal to bf16_rn(fp64 reference) is at least 0.9992 in every family (floor asserted: 0.9); every
perturbed reference fails by at least 215 x its bound.
"""
import pytest
import torch

from mvlm_b200.weights import IMAGE_CHANNELS, seeded_state_dict
from plan_ref import (bf16_rn, bn_affine, bound, conv_ref, expected_ops, maxpool, net_ops, ordered_keys,
                      padded_landmarks)
from test_plan_layers_cpu import check_plan

pytestmark = pytest.mark.gpu

EXACT_FLOOR = 0.9
# (landmarks, image channels, H, W, views, image entry point, producer-fused pools)
CONFIGS = [
    (73, "RGB+depth", 64, 64, 2, "u8", True),      # 1 x 1 bottom maps
    (73, "RGB+depth", 64, 64, 2, "u8", False),     # stand-alone pool / bnrelu passes
    (84, "geometry+depth", 128, 64, 3, "f32", True),
    (5, "geometry", 64, 192, 1, "u8", True),       # cin 1, Lp 32 (.ws M = 32, 32-channel tail chunk of conv7)
    (40, "RGB", 192, 64, 2, "u8", True),           # Lp 64, 3 x 1 bottom map
    (128, "RGB+depth", 256, 256, 1, "u8", True),   # Lp 128, 32-row tiles, full-resolution stem block
]


def _family(op):
    if op["kind"] != "conv":
        return op["kind"]
    layer = op["layer"]
    if layer == "conv1":
        return "stem conv"
    if layer == "conv11":
        return "conv11 phase"
    if ".resample." in layer:
        return "resample"
    if op.get("pool2"):
        return "pool2"
    if op.get("aux_mode"):
        return f"aux{op['aux_mode']}"
    if "res_up" in op["reads"]:
        return "up-residual"
    if ".rb" in layer or ".conv" in layer:
        return "rb conv"
    return layer


def _ratio(got, want, bnd):
    """max |got - want| / bnd, an exact zero counting 0 (padded channels have a zero reference and a zero bound)."""
    err = (got - want).abs()
    return torch.where(err == 0, 0.0, err / bnd).max().item()


def _teeth(op):
    """The perturbation the family's first op must notice (None: not this op)."""
    fam, layer = _family(op), op["layer"]
    if fam == "stem conv":
        return ("bn", "post", "conv2.bn1")
    if fam == "resample" or fam == "pool2":
        return "shift_in"
    if fam == "rb conv" and "pre" in op["terms"] and "post" in op["terms"] and layer.endswith("conv1"):
        return ("bn", "post", layer.rsplit(".", 1)[0] + ".bn1")
    if fam == "up-residual" and layer.endswith("conv1"):
        return "shift_res"
    if layer == "conv7":
        return "bias"
    if fam == "conv11 phase":
        return "phase"
    return None


class _Run:
    def __init__(self, lib, n_landmarks, mode, h, w, views, entry, fusion):
        from mvlm_b200 import ops

        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
        self.lib, self.L, self.h, self.w, self.V = lib, n_landmarks, h, w, views
        self.cin = IMAGE_CHANNELS[mode]
        self.lp = padded_landmarks(n_landmarks)
        sd = seeded_state_dict(n_landmarks, mode, seed=1000 + n_landmarks)
        with ops._plan_env(MVLM_HG_ELT_FUSION="1" if fusion else "0"):
            self.net = ops.Hourglass(sd, n_landmarks, self.cin, views, h, w)
        self.sd = self.net._sd
        g = torch.Generator().manual_seed(n_landmarks + h)
        if entry == "u8":
            img = torch.randint(0, 256, (views, h, w, 4), generator=g, dtype=torch.uint8)
            img[..., self.cin:] = 0
            self.u8, self.f32 = img.cuda(), None
            # u8 / 255 in fp32, divided elementwise (torch turns a division by a Python scalar into a product with
            # its reciprocal, which rounds differently)
            x = self.u8[..., :self.cin].float()
            self.image = x / torch.full_like(x, 255.0)
        else:
            self.u8, self.f32 = None, torch.rand((views, h, w, self.cin), generator=g).cuda()
            self.image = self.f32
        self.recs, self.bufs = net_ops(lib, self.net)
        self.exp, self.tensors = expected_ops(n_landmarks, self.cin, h, w, fusion)
        errs = check_plan(self.recs, self.bufs, self.exp, self.tensors, n_landmarks, views)
        assert not errs, "\n".join(errs[:20])
        for i, r in enumerate(self.recs):
            for name, (buf, _cs, _co, ws) in r["operands"].items():
                assert ws == self.bufs[buf][1], f"op {i}: {name} is not at its buffer's packed offset"
        self.ws = self.net.workspace
        self.hm = torch.full((views, n_landmarks, h, w), float("nan"), device="cuda")
        self.peaks = torch.full((n_landmarks, views, 3), float("nan"), device="cuda")
        self.stats = {}

    # the workspace region of a tensor: its whole buffer as (V, h, w, c) bf16, or the keys as (V, L) int64
    def region(self, tensor):
        op_buf = self.where[tensor]
        off = self.bufs[op_buf][1]
        if tensor == "keys":
            return self.ws[off:off + 8 * self.V * self.L].view(torch.int64).view(self.V, self.L)
        h, w, c = self.tensors[tensor]
        return self.ws[off:off + 2 * self.V * h * w * c].view(torch.bfloat16).view(self.V, h, w, c)

    def note(self, fam, ratio=None, exact=None):
        s = self.stats.setdefault(fam, [0.0, 0, 0])
        if ratio is not None:
            s[0] = max(s[0], ratio)
        if exact is not None:
            s[1] += exact[0]
            s[2] += exact[1]

    def run(self):
        from mvlm_b200 import _lib

        self.where = {}
        for r, e in zip(self.recs, self.exp):
            for name, (tensor, _co) in {**e["reads"], **e["writes"]}.items():
                self.where[tensor] = r["operands"][name][0]
        last_read = {}
        for i, e in enumerate(self.exp):
            for tensor, _co in e["reads"].values():
                last_read[tensor] = i
        cap = {}
        stream = torch.cuda.current_stream().cuda_stream
        for i, (r, e) in enumerate(zip(self.recs, self.exp)):
            tag = f"op {i} ({e['kind']} {e['layer']}{' phase %s' % (e['phase'],) if e['phase'][0] >= 0 else ''})"
            for name, (tensor, _co) in e["reads"].items():
                assert torch.equal(self.region(tensor).view(torch.uint8) if tensor != "keys" else self.region(tensor),
                                   cap[tensor].view(torch.uint8) if tensor != "keys" else cap[tensor]), \
                    f"{tag}: {name} ({tensor}) differs from what its producer wrote"
            before = self.ws.clone()
            _lib.check(self.lib.mvlm_debug_hourglass_run_op(
                self.net._h, i, _lib.ptr(self.u8), _lib.ptr(self.f32), self.hm.data_ptr(), self.peaks.data_ptr(),
                stream), tag)
            torch.cuda.synchronize()
            # stray writes: the whole workspace outside the op's output slices is unchanged
            width = e.get("cout_pad") if e["kind"] == "conv" else None
            for name, (tensor, co) in e["writes"].items():
                dst, src = before, self.ws
                off = self.bufs[self.where[tensor]][1]
                n = 8 * self.V * self.L if tensor == "keys" else 2 * self.V * self.tensors[tensor][0] * \
                    self.tensors[tensor][1] * self.tensors[tensor][2]
                if tensor == "keys" or width is None:
                    dst[off:off + n] = src[off:off + n]
                else:
                    h, w, c = self.tensors[tensor]
                    dv = dst[off:off + n].view(torch.bfloat16).view(self.V, h, w, c)
                    dv[..., co:co + width] = self.region(tensor)[..., co:co + width]
            if not torch.equal(before, self.ws):
                bad = int((before != self.ws).nonzero()[0, 0])
                owners = [k for k, (b, o) in enumerate(self.bufs) if o <= bad < o + b]
                raise AssertionError(f"{tag}: wrote workspace byte {bad} (buffers {owners}) outside its outputs")
            self.check(i, e, cap, tag)
            for tensor, _co in e["writes"].values():
                cap[tensor] = self.region(tensor).clone()
            for tensor in [t for t in cap if last_read.get(t, -1) <= i]:
                del cap[tensor]

    def check(self, i, e, cap, tag):
        kind, fam = e["kind"], _family(e)
        out = {name: self.region(t)[..., co:co + (e["cout_pad"] if kind == "conv" else self.tensors[t][2])].double()
               for name, (t, co) in e["writes"].items() if t != "keys"}
        if kind == "stem":
            v = self.image
            hi = bf16_rn(v)
            lo = bf16_rn(v - hi)
            want = torch.zeros((self.V, self.h, self.w, 16), device="cuda")
            want[..., :self.cin], want[..., 4:4 + self.cin] = hi, lo
            got = self.region("img16").float()
            assert torch.equal(got, want), f"{tag}: hi / lo staging differs"
            self.note(fam, exact=(got.numel(), got.numel()))
        elif kind == "memset":
            assert (self.region("keys") == 0).all(), tag
        elif kind == "peaks":
            k = self.region("keys")
            idx = 0xFFFFFFFF - (k & 0xFFFFFFFF)
            o = (k >> 32) & 0xFFFFFFFF
            bits = torch.where(o >= 0x80000000, o & 0x7FFFFFFF, (~o) & 0xFFFFFFFF)
            val = torch.where(bits >= 2 ** 31, bits - 2 ** 32, bits).to(torch.int32).view(torch.float32)
            want = torch.stack([(idx // self.w - 1).float(), (idx % self.w).float() - 0.5, val], -1).transpose(0, 1)
            assert torch.equal(self.peaks, want), f"{tag}: peaks differ from the keys"
        elif kind in ("pool", "bnrelu"):
            x = cap[e["reads"]["in"][0]].double()
            s, t = bn_affine(self.sd, *e["terms"]["scale"], x.shape[-1])
            if kind == "pool":
                assert torch.equal(out["out_raw"], maxpool(x)), f"{tag}: max-pool differs"
                x = out["out_raw"]
            self._act(tag, fam, out["out_post"], x, s, t)
        elif e["layer"] == "conv11":
            self._phase(i, e, cap, tag)
        else:
            self._conv(e, cap, out, tag, fam)

    def _act(self, tag, fam, got, x, s, t):
        ref = torch.relu(x * s + t)
        err = (got - ref).abs()
        bnd = 2.0 ** -8 * ref.abs() + 2.0 ** -20 * ((x * s).abs() + t.abs())
        assert (err <= bnd).all(), f"{tag}: activation off by {(err / bnd).max().item():.3g} x its bound"
        self.note(fam)

    def _inputs(self, e, cap, perturb=None):
        if e["layer"] == "conv1":
            x = self.image.double()
        else:
            t, co = e["reads"]["in"]
            x = cap[t][..., co:co + e["cin"]].double()
        res = {}
        for k in ("res1", "res2", "res_up"):
            if k in e["reads"]:
                t, co = e["reads"][k]
                if perturb == "shift_res" and k == "res_up":
                    co += 8
                res[k] = cap[t][..., co:co + e["cout_pad"]].double()
        return x, res

    def _conv(self, e, cap, out, tag, fam, perturb=None):
        """Compares every output of a conv op with the reference; returns the worst err / bound ratio."""
        x, res = self._inputs(e, cap, perturb)
        ref = conv_ref(self.sd, e, x, res, self.lp, perturb=None if perturb == "shift_res" else perturb)
        c = 2.0 ** -14 + (2.0 ** -16 if e["layer"] == "conv1" else 0.0)
        worst, exact = 0.0, [0, 0]

        def cmp(name, want, bnd):
            nonlocal worst
            got = out[name]
            worst = max(worst, _ratio(got, want, bnd))
            eq = (got == bf16_rn(want)).sum().item()
            exact[0] += eq
            exact[1] += got.numel()

        if "out_pre" in out:
            cmp("out_pre", ref["pre"], bound(ref["pre"], ref["A_pre"], c=c))
        if e.get("pool2"):
            cmp("out_raw", maxpool(ref["v"]), maxpool(bound(ref["v"], ref["A"], c=c)))
        elif "out_raw" in out:
            cmp("out_raw", ref["v"], bound(ref["v"], ref["A"], c=c))
        if "out_post" in out and not e.get("pool2"):
            cmp("out_post", ref["post"], bound(ref["post"], ref["A_post"], c=c))
        if perturb is not None:
            return worst
        assert worst <= 1.0, f"{tag}: off by {worst:.3g} x its bound"
        self.note(fam, worst, exact)
        cout = e["cout_pad"]
        if e.get("pool2") and "out_post" in out:
            s, t = bn_affine(self.sd, *e["terms"]["post"], cout)
            self._act(tag, fam, out["out_post"], out["out_raw"], s, t)
        if e.get("aux_mode"):
            s, t = bn_affine(self.sd, *e["terms"]["aux"], cout)
            if e["aux_mode"] == 1:
                self._act(tag, fam, out["out_aux1"], out["out_raw"], s, t)
            else:
                assert torch.equal(out["out_aux1"], maxpool(out["out_raw"])), f"{tag}: pooled copy differs"
                self._act(tag, fam, out["out_aux2"], out["out_aux1"], s, t)
        return worst

    def _phase(self, i, e, cap, tag, perturb=None):
        a, b = e["phase"]
        x = cap[e["reads"]["in"][0]].double()
        ref = conv_ref(self.sd, e, x, {}, self.lp, perturb=perturb)
        want = ref["v"][..., :self.L].permute(0, 3, 1, 2)
        bnd = bound(want, ref["A"][..., :self.L].permute(0, 3, 1, 2), bf16_out=False)
        got = self.hm[:, :, a::2, b::2].double()
        worst = _ratio(got, want, bnd)
        if perturb is not None:
            return worst
        assert worst <= 1.0, f"{tag}: heat maps off by {worst:.3g} x their bound"
        self.note("conv11 phase", worst)
        # keys = the running arg-max over the phases so far, from the plan's own fp32 maps
        done = [(p // 2, p % 2) for p in range(2 * a + b + 1)]
        idx = torch.arange(self.h * self.w, device="cuda").view(self.h, self.w)
        mask = torch.zeros((self.h, self.w), dtype=torch.bool, device="cuda")
        for (pa, pb) in done:
            mask[pa::2, pb::2] = True
        vals = self.hm.view(self.V, self.L, -1)[:, :, mask.view(-1)]
        keys = ordered_keys(vals, idx.view(-1)[mask.view(-1)].expand_as(vals)).max(-1).values
        got_keys = self.region("keys") ^ (-(2 ** 63))
        assert torch.equal(got_keys, keys), f"{tag}: arg-max keys differ from the running maximum of the maps"
        return worst

    def teeth(self):
        """Re-runs the plan and, for the first op of each family, checks that a perturbed reference fails the bound."""
        seen = set()
        for i, e in enumerate(self.exp):
            p = _teeth(e) if e["kind"] == "conv" else None
            fam = _family(e)
            if p is None or fam in seen:
                continue
            seen.add(fam)
            yield i, e, fam, p


@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: "L%d-%s-%dx%d-v%d-%s-%s" % (c[0], c[1], c[2], c[3], c[4], c[5],
                                                                                   "fused" if c[6] else "unfused"))
def test_plan_launch_by_launch(lib, cfg):
    run = _Run(lib, *cfg)
    teeth = {i: (fam, p) for i, _e, fam, p in run.teeth()}
    run.teeth_results = {}
    orig_check = run.check

    def check(i, e, cap, tag):
        orig_check(i, e, cap, tag)
        if i in teeth:
            fam, p = teeth[i]
            if e["layer"] == "conv11":
                r = run._phase(i, e, cap, tag, perturb=p)
            else:
                out = {name: run.region(t)[..., co:co + e["cout_pad"]].double()
                       for name, (t, co) in e["writes"].items()}
                r = run._conv(e, cap, out, tag, fam, perturb=p)
            run.teeth_results[fam] = (p, r)

    run.check = check
    run.run()
    for fam, (p, r) in sorted(run.teeth_results.items()):
        print(f"teeth {fam}: {p} -> {r:.3g} x bound")
        assert r > 1.0, f"{fam}: the reference perturbed by {p} still passes ({r:.3g} x bound)"
    for fam, (worst, eq, n) in sorted(run.stats.items()):
        frac = eq / n if n else float("nan")
        print(f"{cfg} {fam}: worst err/bound {worst:.3g}, bit-exact {frac:.4f}")
        if n:
            assert frac >= EXACT_FLOOR, f"{fam}: only {frac:.3f} of the outputs equal bf16_rn(reference)"
    assert {"stem conv", "resample", "rb conv", "up-residual", "pool2", "conv11 phase"} <= set(run.teeth_results)
