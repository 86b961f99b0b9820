"""The CNN plan's op list as the reference model defines it, and an fp64 reference of each op.

`expected_ops` walks oracle/hourglass_ref.py (written in the plan's producer / consumer order) and lists, op by op,
what the plan must launch: the layer, its bias, every BatchNorm affine with its channel offset, and which named tensor
(slice) each operand reads or writes.  Tensors are named after the reference's variables ("hg1.rb5.y" = the output of
hg1.rb5, "conv2.a_in" = relu(conv2.bn1(x0)), ...).  `plan_ops` reads the records the library keeps for every op
(mvlm_debug_hourglass_dry_ops / _ops), so the tests compare the two lists without trusting the plan's own bookkeeping.

`conv_ref` computes one convolution op in fp64 on the device from tensors captured from the plan's own earlier outputs
(teacher forcing): weights bf16_rn(w_fp32) as the packers store them, conv11's phase weights summed in fp32 in the
packer's order and then rounded, BatchNorm folded from the state_dict, the stem reading the fp32 image.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn.functional as F

OPERANDS = ("in", "res1", "res2", "res_up", "out_pre", "out_raw", "out_post", "out_aux1", "out_aux2", "keys")
TERMS = ("mid", "pre", "post", "aux", "scale")
KINDS = ("conv", "pool", "bnrelu", "stem", "memset", "peaks")
READS = ("in", "res1", "res2", "res_up")
BN_EPS = 1e-5


def padded_landmarks(n):
    lp = (n + 15) // 16 * 16
    return {16: 32, 48: 64, 112: 128}.get(lp, lp)


# ---- the plan's records -----------------------------------------------------------------------------------------------

def _decode(ops, bufs, n_ops, n_bufs):
    out = []
    for o in ops[:n_ops]:
        out.append({
            "kind": KINDS[o.kind], "layer": o.layer.decode(), "bias": o.bias.decode(), "phase": (o.phase_a, o.phase_b),
            "terms": {TERMS[k]: (t.bn.decode(), t.off) for k, t in enumerate(o.terms) if t.bn},
            **{f: getattr(o, f) for f in ("h", "w", "cin", "in_cs", "kh", "kw", "y_off0", "x_off0", "cout_pad",
                                         "n_tile", "cout_real", "pool2", "aux_mode")},
            "operands": {OPERANDS[k]: (p.buf, p.cs, p.co, p.ws_offset) for k, p in enumerate(o.operands) if p.cs},
        })
    return out, [(b.bytes, b.offset) for b in bufs[:n_bufs]]


def _fetch(call):
    from mvlm_b200 import _lib

    n, nb = C.c_int(), C.c_int()
    _lib.check(call(None, 0, C.byref(n), None, 0, C.byref(nb)), "op records")
    ops, bufs = (_lib.HgOp * n.value)(), (_lib.HgBuffer * nb.value)()
    _lib.check(call(ops, n.value, C.byref(n), bufs, nb.value, C.byref(nb)), "op records")
    return _decode(ops, bufs, n.value, nb.value)


def plan_ops(lib, n_landmarks, cin, n_views, h, w):
    """(op records, [(bytes, offset)] per buffer) of a dry plan: no device, honours the MVLM_HG_* switches."""
    return _fetch(lambda *a: lib.mvlm_debug_hourglass_dry_ops(n_landmarks, cin, n_views, h, w, *a))


def net_ops(lib, net):
    """The same for a created plan (mvlm_b200.ops.Hourglass); ws_offset then comes from the pointers the ops use."""
    return _fetch(lambda *a: lib.mvlm_debug_hourglass_ops(net._h, *a))


# ---- the expected op list ---------------------------------------------------------------------------------------------

class _List:
    def __init__(self):
        self.ops, self.tensors = [], {}

    def t(self, name, h, w, c):
        assert name not in self.tensors, name
        self.tensors[name] = (h, w, c)
        return name

    def op(self, kind, **kw):
        op = {"kind": kind, "layer": "", "bias": "", "phase": (-1, -1), "terms": {}, "reads": {}, "writes": {}}
        op.update(kw)
        self.ops.append(op)
        return op

    def conv(self, layer, src, cin, cout, k, h, w, bias=True, terms=None, reads=None, writes=None, **kw):
        reads = dict(reads or {})
        reads["in"] = (src, 0)
        kw.setdefault("y_off0", -(k // 2))
        kw.setdefault("x_off0", -(k // 2))
        return self.op("conv", layer=layer, bias=f"{layer}.bias" if bias else "", terms=terms or {}, reads=reads,
                       writes=writes or {}, h=h, w=w, cin=cin, cout_pad=cout, kh=k, kw=k, **kw)


def expected_ops(n_landmarks, cin, h, w, fusion=True):
    """(ops, tensors): the plan of (n_landmarks, cin, h, w) as oracle/hourglass_ref.py computes it.  fusion = the
    default plan, whose producers also write the max-pools and conv4's resample activation (MVLM_HG_ELT_FUSION)."""
    lp = padded_landmarks(n_landmarks)
    G = _List()
    h2, w2 = h // 2, w // 2

    def rb(p, x, a_in, cin_, cout, hh, ww, post=None, up=None, pool=False, ar=None, aux=None):
        """ResidualBlock (:267-273) as hourglass_ref.rb: returns the names of (y, relu(post(y)), aux outputs)."""
        oh, ow = (hh // 2, ww // 2) if pool else (hh, ww)
        c1, c2 = cout // 2, cout // 4
        if cin_ != cout:
            y = G.t(f"{p}.y" if not pool else f"{p}.y_full", hh, ww, cout)
            G.conv(f"{p}.resample.2", ar, cin_, cout, 1, hh, ww, bias=False, writes={"out_raw": (y, 0)})
            skip = y
        else:
            skip = x
            y = None
        out = G.t(f"{p}.y", oh, ow, cout) if (pool or y is None) else y
        post_t = G.t(f"{p}.post", oh, ow, cout) if post else None
        aux_t = None
        if aux:
            mode, bn_name, names = aux
            aux_t = [G.t(names[0], *((hh // 2, ww // 2) if mode == 2 else (hh, ww)), cout)]
            if mode == 2:
                aux_t.append(G.t(names[1], hh // 2, ww // 2, cout))
        a1, a2 = G.t(f"{p}.a1", hh, ww, c1), G.t(f"{p}.a2", hh, ww, c2)
        widths, offs, cins, ins = (c1, c2, c2), (0, c1, c1 + c2), (cin_, c1, c2), (a_in, a1, a2)
        pres = ((a1, f"{p}.bn2"), (a2, f"{p}.bn3"), None)
        for i in range(3):
            terms, writes, reads = {}, {}, {"res1": (skip, offs[i])}
            if pres[i]:
                terms["pre"] = (pres[i][1], 0)
                writes["out_pre"] = (pres[i][0], 0)
            if up:
                reads["res_up"] = (up, offs[i])
            writes["out_raw"] = (out, offs[i])
            if post:
                terms["post"] = (post, offs[i])
                writes["out_post"] = (post_t, offs[i])
            mode = 0
            if aux:
                mode = aux[0]
                terms["aux"] = (aux[1], offs[i])
                writes["out_aux1"] = (aux_t[0], offs[i])
                if mode == 2:
                    writes["out_aux2"] = (aux_t[1], offs[i])
            G.conv(f"{p}.conv{i + 1}", ins[i], cins[i], widths[i], 3, hh, ww, bias=False, terms=terms, reads=reads,
                   writes=writes, pool2=int(pool), aux_mode=mode)
        return out, post_t

    def pool_op(src, bn_name, raw, act):
        hh, ww, c = G.tensors[src]
        G.op("pool", terms={"scale": (bn_name, 0)}, reads={"in": (src, 0)},
             writes={"out_raw": (raw, 0), "out_post": (act, 0)}, h=hh, w=ww, cin=c)

    def hourglass(p, x, a_x, hh, ww, in_pooled):
        """HourGlassModule.forward (:301-361) in hourglass_ref.hourglass's order."""
        F_ = 256
        cur, lows, a_lows = x, [], []
        low_blocks, skip_blocks = (2, 4, 6, 8, 10), (3, 5, 7, 9)
        for lvl, lb in enumerate(low_blocks):
            lbn = f"{p}.rb{lb}"
            ch, cw = G.tensors[cur][:2]
            if not (fusion and (lvl > 0 or in_pooled)):
                G.t(f"{lbn}.in", ch // 2, cw // 2, F_)
                G.t(f"{lbn}.a_in", ch // 2, cw // 2, F_)
                pool_op(cur, f"{lbn}.bn1", f"{lbn}.in", f"{lbn}.a_in")
            nxt = skip_blocks[lvl] if lvl < 4 else 11
            aux = None
            if fusion and lvl < 4:
                nb = f"{p}.rb{low_blocks[lvl + 1]}"
                aux = (2, f"{nb}.bn1", (f"{nb}.in", f"{nb}.a_in"))
            low, a_low = rb(lbn, f"{lbn}.in", f"{lbn}.a_in", F_, F_, ch // 2, cw // 2, post=f"{p}.rb{nxt}.bn1", aux=aux)
            lows.append(low)
            a_lows.append(a_low)
            cur = low
        ch, cw = G.tensors[cur][:2]
        low2, a2 = rb(f"{p}.rb11", cur, a_lows[4], F_, F_, ch, cw, post=f"{p}.rb12.bn1")
        cur, _ = rb(f"{p}.rb12", low2, a2, F_, F_, ch, cw)
        for lvl, (b1, b2) in enumerate(((13, 14), (15, 16), (17, 18), (19, 20))):
            sk = lows[3 - lvl]
            ch, cw = G.tensors[sk][:2]
            s, a = rb(f"{p}.rb{skip_blocks[3 - lvl]}", sk, a_lows[3 - lvl], F_, F_, ch, cw, post=f"{p}.rb{b1}.bn1", up=cur)
            l1, a1 = rb(f"{p}.rb{b1}", s, a, F_, F_, ch, cw, post=f"{p}.rb{b2}.bn1")
            cur, _ = rb(f"{p}.rb{b2}", l1, a1, F_, F_, ch, cw)
        out, _ = rb(f"{p}.rb1", x, a_x, F_, F_, hh, ww, up=cur)
        return out

    # stem (:405-407): image -> hi / lo staging, conv1 + bn1 + ReLU -> the conv2 block's two activations
    img16 = G.t("img16", h, w, 16)
    G.op("stem", writes={"out_raw": (img16, 0)}, h=h, w=w, cin=cin)
    a_c2, ar_c2 = G.t("conv2.a_in", h, w, 64), G.t("conv2.ar", h, w, 64)
    G.conv("conv1", img16, 16, 64, 3, h, w, terms={"mid": ("bn1", 0), "pre": ("conv2.bn1", 0),
                                                  "post": ("conv2.resample.0", 0)},
           writes={"out_pre": (a_c2, 0), "out_post": (ar_c2, 0)})
    # conv2 block, consumed only through its max-pool (:410-411)
    x1, a3 = rb("conv2", None, a_c2, 64, 128, h, w, post="conv3.bn1", pool=True, ar=ar_c2)
    if fusion:
        y3, a4 = rb("conv3", x1, a3, 128, 128, h2, w2, post="conv4.bn1",
                    aux=(1, "conv4.resample.0", ("conv4.ar",)))
    else:
        y3, a4 = rb("conv3", x1, a3, 128, 128, h2, w2, post="conv4.bn1")
        G.t("conv4.ar", h2, w2, 128)
        G.op("bnrelu", terms={"scale": ("conv4.resample.0", 0)}, reads={"in": (y3, 0)},
             writes={"out_post": ("conv4.ar", 0)}, h=h2, w=w2, cin=128)
    aux4 = (2, "hg1.rb2.bn1", ("hg1.rb2.in", "hg1.rb2.a_in")) if fusion else None
    r3, a_h1 = rb("conv4", y3, a4, 128, 256, h2, w2, post="hg1.rb1.bn1", ar="conv4.ar", aux=aux4)
    hg1 = hourglass("hg1", r3, a_h1, h2, w2, fusion)
    ll1, x6 = G.t("ll1", h2, w2, 256), G.t("x6", h2, w2, lp)
    G.conv("conv5", hg1, 256, 256, 3, h2, w2, terms={"pre": ("bn2", 0)}, writes={"out_pre": (ll1, 0)})
    G.conv("conv6", ll1, 256, lp, 3, h2, w2, writes={"out_raw": (x6, 0)})
    s, a_h2 = G.t("sum_temp", h2, w2, 256), G.t("hg2.a_x", h2, w2, 256)
    terms, writes = {"post": ("hg2.rb1.bn1", 0)}, {"out_raw": (s, 0), "out_post": (a_h2, 0)}
    if fusion:
        G.t("hg2.rb2.in", h2 // 2, w2 // 2, 256)
        G.t("hg2.rb2.a_in", h2 // 2, w2 // 2, 256)
        terms["aux"] = ("hg2.rb2.bn1", 0)
        writes.update(out_aux1=("hg2.rb2.in", 0), out_aux2=("hg2.rb2.a_in", 0))
    G.conv("conv7", x6, lp, 256, 3, h2, w2, terms=terms, reads={"res1": (r3, 0), "res2": (ll1, 0)}, writes=writes,
           aux_mode=2 if fusion else 0)
    hg2 = hourglass("hg2", s, a_h2, h2, w2, fusion)
    ll2, x10 = G.t("ll2", h2, w2, 256), G.t("x10", h2, w2, lp)
    G.conv("conv9", hg2, 256, 256, 3, h2, w2, terms={"pre": ("bn3", 0)}, writes={"out_pre": (ll2, 0)})
    G.conv("conv10", ll2, 256, lp, 3, h2, w2, writes={"out_raw": (x10, 0)})
    # conv11 on nearest-x2(conv10) (:428-429) as four 2x2 phase convolutions with the fused arg-max
    G.tensors["keys"] = (1, 1, n_landmarks)
    G.op("memset", writes={"keys": ("keys", 0)})
    for a in range(2):
        for b in range(2):
            G.op("conv", layer="conv11", bias="conv11.bias", phase=(a, b), reads={"in": (x10, 0), "keys": ("keys", 0)},
                 writes={"keys": ("keys", 0)}, h=h2, w=w2, cin=lp, cout_pad=lp, kh=2, kw=2, y_off0=a - 1,
                 x_off0=b - 1, cout_real=n_landmarks)
    G.op("peaks", reads={"in": (x10, 0), "keys": ("keys", 0)})
    return G.ops, G.tensors


# ---- fp64 references --------------------------------------------------------------------------------------------------

def bf16_rn(t):
    return t.to(torch.bfloat16).to(t.dtype)


def bn_affine(sd, name, off, c):
    """Folded BatchNorm channels [off, off + c) in fp64 (fp32 state_dict values)."""
    g = lambda k: sd[f"{name}.{k}"].double()[off:off + c]  # noqa: E731
    s = g("weight") / torch.sqrt(g("running_var") + BN_EPS)
    return s, g("bias") - g("running_mean") * s


def layer_weight(sd, op, lp):
    """The op's weights as the plan stores them, fp64 OIHW (cout_pad, cin, kh, kw) with zero padding."""
    cout, cin, kh = op["cout_pad"], op["cin"], op["kh"]
    if op["layer"] == "conv11":
        w = sd["conv11.weight"].float()
        a, b = op["phase"]
        rows = ((0,), (1, 2)) if a == 0 else ((0, 1), (2,))
        cols = ((0,), (1, 2)) if b == 0 else ((0, 1), (2,))
        wp = torch.zeros((w.shape[0], w.shape[1], 2, 2), dtype=torch.float32, device=w.device)
        for ky in range(2):
            for kx in range(2):
                acc = torch.zeros_like(w[:, :, 0, 0])
                for rr in rows[ky]:             # the packer's order: rr outer, cc inner, fp32
                    for cc in cols[kx]:
                        acc = acc + w[:, :, rr, cc]
                wp[:, :, ky, kx] = acc
        w = bf16_rn(wp)
    elif op["layer"] == "conv1":
        w = bf16_rn(sd["conv1.weight"].float())
    else:
        w = bf16_rn(sd[f"{op['layer']}.weight"].float())
    out = torch.zeros((cout, cin, kh, kh), dtype=torch.float64, device=w.device)
    out[:w.shape[0], :w.shape[1]] = w.double()
    return out


def conv(x_nhwc, w, y_off0, x_off0):
    """NHWC fp64 conv whose tap (ky, kx) reads input (y + y_off0 + ky, x + x_off0 + kx), zero outside."""
    kh, kw = w.shape[-2:]
    x = x_nhwc.permute(0, 3, 1, 2)
    x = F.pad(x, (-x_off0, kw - 1 + x_off0, -y_off0, kh - 1 + y_off0))
    return F.conv2d(x, w).permute(0, 2, 3, 1)


def maxpool(t):
    return F.max_pool2d(t.permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1)


def up2(t):
    return t.repeat_interleave(2, 1).repeat_interleave(2, 2)


def conv_ref(sd, op, x, res, lp, perturb=None):
    """fp64 reference of a convolution op.  x: the input (V, h, w, cin) (stem: the fp32 image in NHWC); res: the
    residual slices {"res1": .., "res2": .., "res_up": ..} as (V, *, *, cout_pad).  Returns {"v": the value the raw
    output stores (before pooling), "A": the sum of absolute products, "pre": .., "post": .. (unpooled outputs),
    "A_pre" / "A_post"}.  perturb (the tests' check that the bound has teeth): "bias" drops the bias, "shift_in" moves
    the input by one pixel, "phase" uses another phase's weights, ("bn", term, name) replaces one BatchNorm."""
    cout = op["cout_pad"]
    terms = dict(op["terms"])
    if perturb and perturb[0] == "bn":
        terms[perturb[1]] = (perturb[2], terms[perturb[1]][1])
    if op["layer"] == "conv1":
        w = layer_weight(sd, op, lp)[:, :x.shape[-1]]
    else:
        wop = dict(op, phase=(1 - op["phase"][0], op["phase"][1])) if perturb == "phase" else op
        w = layer_weight(sd, wop, lp)
    if perturb == "shift_in":
        x = torch.roll(x, 1, dims=2)
    v = conv(x, w, op["y_off0"], op["x_off0"])
    A = conv(x.abs(), w.abs(), op["y_off0"], op["x_off0"])
    if op["bias"] and perturb != "bias":
        b = torch.zeros(cout, dtype=torch.float64, device=v.device)
        bb = sd[op["bias"]].double()
        b[:bb.numel()] = bb
        v, A = v + b, A + b.abs()
    out = {}

    def affine(term, val, a):
        s, t = bn_affine(sd, *terms[term], cout)
        return torch.relu(val * s + t), a * s.abs() + t.abs()

    if "mid" in terms:
        v, A = affine("mid", v, A)
    if "pre" in terms:
        out["pre"], out["A_pre"] = affine("pre", v, A)
    for k, r in res.items():
        r = r.double()
        if k == "res_up":
            r = up2(r)
        v, A = v + r, A + r.abs()
    out["v"], out["A"] = v, A
    if "post" in terms:
        out["post"], out["A_post"] = affine("post", v, A)
    return out


def bound(ref, A, bf16_out=True, c=2.0 ** -14):
    """|got - ref| allowed: bf16 output rounding (2^-8 |ref|) + fp32 / tensor-core accumulation (c * A)."""
    return (2.0 ** -8 * ref.abs() if bf16_out else 0.0) + c * A


def ordered_keys(vals, idx):
    """u64 arg-max keys (ordered fp32 value << 32 | ~index) as int64 with the top bit flipped, so that signed
    comparison is the kernel's unsigned order.  vals fp32, idx int64 pixel index."""
    b = vals.contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    neg = (b >> 31) == 1
    o = torch.where(neg, (~b) & 0xFFFFFFFF, b | 0x80000000)
    k = (o << 32) | (0xFFFFFFFF - idx)
    return k ^ (-(2 ** 63))
