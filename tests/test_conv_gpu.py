"""Parity of the tcgen05 implicit-GEMM conv (mvlm_conv2d_bf16) against an fp64 reference on the same bf16-rounded
operands, element by element (plan_ref.bound): |err| <= 2^-8 |ref| (bf16 output rounding; none for fp32 outputs)
+ 2^-14 A, A = the same computation on absolute values (fp32 / tensor-core accumulation).  The upsample-phase and
max-pool tests keep their own tolerances (summed phase weights; pools bit-exact).
"""
import pytest
import torch
import torch.nn.functional as F

from plan_ref import bf16_rn, bound, conv

pytestmark = pytest.mark.gpu


def _ref(x_nhwc, w_oihw, bias, y_off0, x_off0):
    """fp64 conv of the operands the kernel reads (weights rounded to bf16 as the packer stores them) whose tap
    (ky, kx) reads input (y + y_off0 + ky, x + x_off0 + kx), and A, the same sum over absolute values."""
    x = x_nhwc.double()
    w = bf16_rn(w_oihw.float()).double()
    v, A = conv(x, w, y_off0, x_off0), conv(x.abs(), w.abs(), y_off0, x_off0)
    if bias is not None:
        v, A = v + bias.double(), A + bias.double().abs()
    return v, A


def _affine(v, A, s, t):
    """relu(v * s + t) and its A."""
    s, t = s.double(), t.double()
    return torch.relu(v * s + t), A * s.abs() + t.abs()


def _check(got, ref, A, what, bf16_out=True):
    """Every element of got within plan_ref.bound of ref."""
    got = got.double()
    assert torch.isfinite(got).all(), f"{what}: NaN / inf"
    err = (got - ref).abs()
    r = torch.where(err == 0, 0.0, err / bound(ref, A, bf16_out)).max().item()
    assert r <= 1.0, f"{what}: off by {r:.3g} x its bound"


CASES = [
    # n, h, w, cin, cs_in, cout, n_tile, kh, kw
    (2, 32, 32, 64, 64, 64, 64, 3, 3),
    (1, 16, 16, 256, 256, 128, 128, 3, 3),
    (3, 64, 64, 128, 128, 64, 64, 3, 3),
    (2, 32, 48, 256, 256, 256, 128, 3, 3),   # two N tiles, non-square
    (2, 32, 32, 64, 64, 32, 32, 3, 3),
    (2, 16, 16, 32, 64, 32, 32, 3, 3),       # cin 32 read from a 64-stride buffer
    (2, 32, 32, 80, 80, 256, 128, 3, 3),     # cin = 64 + 16 (partial last chunk)
    (2, 32, 32, 256, 256, 73, 80, 3, 3),     # cout 73 padded to 80
    (1, 32, 32, 96, 96, 84, 96, 3, 3),
    (2, 32, 32, 64, 64, 128, 128, 1, 1),     # 1x1 resample conv
    (5, 8, 8, 256, 256, 128, 128, 3, 3),     # map smaller than the 8x32 tile
    (5, 4, 4, 128, 128, 64, 64, 3, 3),
    (2, 24, 40, 64, 64, 64, 64, 3, 3),       # ragged: rows not a multiple of the tile height
    (2, 80, 20, 64, 64, 64, 64, 3, 3),       # ragged: width not a multiple of 8, 2.5 tiles high
    (3, 2, 2, 256, 256, 128, 128, 3, 3),     # 2x2 map (hourglass bottom of a 64^2 image)
    # cout <= 64: tcgen05.mma.ws, M = 64 (33..64 channels) or M = 32, accumulator tile spread over all four lane groups
    (2, 32, 32, 64, 64, 48, 48, 3, 3),       # M = 64 with 48 weight rows
    (2, 32, 32, 64, 64, 16, 16, 3, 3),       # M = 32 with 16 weight rows
    (3, 2, 2, 128, 128, 32, 32, 3, 3),       # 8-row tile (N = 64, the .ws minimum) on a 2x2 map
    (2, 16, 24, 16, 16, 64, 64, 3, 3),       # the stem's shape: one 16-channel (32-byte row) chunk, stationary weights
    (2, 40, 16, 128, 128, 64, 64, 3, 3),     # streamed weights, one ring slot per column of taps
    (2, 32, 32, 64, 64, 64, 64, 2, 2),       # 2x2 taps: two-tap columns
    (2, 32, 32, 96, 96, 32, 32, 1, 1),       # 1x1, 64 + 32-channel tail chunk
]


@pytest.mark.parametrize("n,h,w,cin,cs,cout,n_tile,kh,kw", CASES)
def test_conv_raw(lib, n, h, w, cin, cs, cout, n_tile, kh, kw):
    from mvlm_b200 import ops

    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    g = torch.Generator(device="cuda").manual_seed(1234 + n * 7 + h + cin)
    x = torch.randn((n, h, w, cs), generator=g, device="cuda").to(torch.bfloat16)
    wt = (torch.randn((cout, cin, kh, kw), generator=g, device="cuda") / (cin * kh * kw) ** 0.5)
    bias = torch.randn((cout,), generator=g, device="cuda")
    cout_pad = ((cout + n_tile - 1) // n_tile) * n_tile
    wp = ops.pack_conv_weight(wt, cout_pad, cin)
    bias_p = torch.zeros(cout_pad, device="cuda")
    bias_p[:cout] = bias
    out = torch.full((n, h, w, cout_pad), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.conv2d_bf16(x, wp, cin=cin, n_tile=n_tile, kh=kh, kw=kw, bias=bias_p, out_raw=(out, 0))
    torch.cuda.synchronize()
    ref, A = _ref(x[..., :cin], wt, bias, -(kh // 2), -(kw // 2))
    _check(out[..., :cout], ref, A, "out_raw")
    if cout_pad > cout:
        assert (out[..., cout:].float() == 0).all()


def test_conv_full_epilogue(lib):
    """bias + act_pre + two residuals + raw + act_post; and fp32 NCHW out + fused argmax keys."""
    from mvlm_b200 import ops

    torch.backends.cudnn.allow_tf32 = False
    n, h, w, cin, cout, n_tile = 2, 32, 32, 128, 128, 128
    g = torch.Generator(device="cuda").manual_seed(7)
    x = torch.randn((n, h, w, cin), generator=g, device="cuda").to(torch.bfloat16)
    wt = torch.randn((cout, cin, 3, 3), generator=g, device="cuda") / (cin * 9) ** 0.5
    bias = torch.randn((cout,), generator=g, device="cuda")
    s1, t1, s2, t2 = (torch.randn((cout,), generator=g, device="cuda") for _ in range(4))
    r1 = torch.randn((n, h, w, 256), generator=g, device="cuda").to(torch.bfloat16)
    r2 = torch.randn((n, h, w, 128), generator=g, device="cuda").to(torch.bfloat16)
    wp = ops.pack_conv_weight(wt, cout, cin)
    out_pre = torch.zeros((n, h, w, 128), device="cuda", dtype=torch.bfloat16)
    out_raw = torch.zeros((n, h, w, 256), device="cuda", dtype=torch.bfloat16)
    out_post = torch.zeros((n, h, w, 256), device="cuda", dtype=torch.bfloat16)
    ops.conv2d_bf16(x, wp, n_tile=n_tile, bias=bias, pre=(s1, t1, out_pre, 0), res1=(r1, 128), res2=(r2, 0),
                    out_raw=(out_raw, 64), post=(s2, t2, out_post, 128))
    torch.cuda.synchronize()
    v, A = _ref(x, wt, bias, -1, -1)
    _check(out_pre, *_affine(v, A, s1, t1), "out_pre")
    r = r1[..., 128:256].double() + r2.double()
    v2, A2 = v + r, A + r1[..., 128:256].double().abs() + r2.double().abs()
    _check(out_raw[..., 64:192], v2, A2, "out_raw")
    assert (out_raw[..., :64] == 0).all() and (out_raw[..., 192:] == 0).all()
    _check(out_post[..., 128:], *_affine(v2, A2, s2, t2), "out_post")
    # fp32 + fused arg-max path (conv11): argmax == argmax of the fp32 map the same kernel wrote
    for co in (128, 73, 32):
        wt2 = wt[:co]
        cp = ((co + 15) // 16) * 16
        wp2 = ops.pack_conv_weight(wt2, cp, cin)
        b2 = torch.zeros(cp, device="cuda")
        b2[:co] = bias[:co]
        out_f32 = torch.zeros((n, co, h, w), device="cuda")
        keys = torch.zeros((n * co,), device="cuda", dtype=torch.int64)
        ops.conv2d_bf16(x, wp2, n_tile=cp, bias=b2, out_f32=out_f32, argmax_keys=keys, cout_real=co)
        torch.cuda.synchronize()
        _check(out_f32, v[..., :co].permute(0, 3, 1, 2), A[..., :co].permute(0, 3, 1, 2), f"fp32 map ({co})",
               bf16_out=False)
        k = keys.view(n, co)
        idx = 0xFFFFFFFF - (k & 0xFFFFFFFF)
        assert torch.equal(idx, out_f32.view(n, co, -1).argmax(dim=-1))
    with pytest.raises(Exception, match="cannot be combined"):
        ops.conv2d_bf16(x, wp, n_tile=n_tile, res1=(r1, 0), out_f32=torch.zeros((n, cout, h, w), device="cuda"), cout_real=cout)


def test_conv_upsample_phase(lib):
    """conv3x3(nearest_up2(x)) == four 2x2 phase convs at the low resolution (conv11 path,
    paulsenpredictor.py:428-429)."""
    from mvlm_b200 import ops

    torch.backends.cudnn.allow_tf32 = False
    n, h, w, c, cout = 2, 32, 32, 80, 73
    g = torch.Generator(device="cuda").manual_seed(11)
    x = torch.randn((n, h, w, c), generator=g, device="cuda").to(torch.bfloat16)
    x[..., 73:] = 0
    wt = torch.randn((cout, 73, 3, 3), generator=g, device="cuda") / (73 * 9) ** 0.5
    bias = torch.randn((cout,), generator=g, device="cuda")
    bias_p = torch.zeros(80, device="cuda")
    bias_p[:cout] = bias
    out = torch.zeros((n, cout, 2 * h, 2 * w), device="cuda")
    for a in range(2):
        for b in range(2):
            # rows: a=0 -> offsets {-1: w0, 0: w1+w2}; a=1 -> {0: w0+w1, +1: w2}
            wr = torch.stack([wt[:, :, 0], wt[:, :, 1] + wt[:, :, 2]], 2) if a == 0 else \
                torch.stack([wt[:, :, 0] + wt[:, :, 1], wt[:, :, 2]], 2)      # (co,ci,2,3)
            wc = torch.stack([wr[..., 0], wr[..., 1] + wr[..., 2]], 3) if b == 0 else \
                torch.stack([wr[..., 0] + wr[..., 1], wr[..., 2]], 3)          # (co,ci,2,2)
            wp = ops.pack_conv_weight(wc.contiguous(), 80, 80)
            ops.conv2d_bf16(x, wp, n_tile=80, kh=2, kw=2, y_off0=a - 1, x_off0=b - 1, bias=bias_p,
                            out_f32=out, cout_real=cout, up=(2, 2, a, b))
    torch.cuda.synchronize()
    xu = F.interpolate(x[..., :73].float().permute(0, 3, 1, 2), scale_factor=2, mode="nearest")
    ref = F.conv2d(xu, wt.to(torch.bfloat16).float(), bias, padding=1)
    scale = ref.abs().max().item()
    # combined phase weights are rounded to bf16 after summation -> bf16-level difference
    assert (out - ref).abs().max().item() <= 1.5e-2 * scale


def test_conv_fused_maxpool(lib):
    """pool2 epilogue == F.max_pool2d of the bf16 raw output (+ BN+ReLU of the pooled values)."""
    from mvlm_b200 import ops

    torch.backends.cudnn.allow_tf32 = False
    for (n, h, w, cin, cout) in ((2, 32, 32, 64, 64), (1, 48, 32, 64, 32), (2, 16, 32, 128, 128)):
        g = torch.Generator(device="cuda").manual_seed(3 + cout)
        x = torch.randn((n, h, w, cin), generator=g, device="cuda").to(torch.bfloat16)
        wt = torch.randn((cout, cin, 3, 3), generator=g, device="cuda") / (cin * 9) ** 0.5
        s2, t2 = (torch.randn((cout,), generator=g, device="cuda") for _ in range(2))
        res = torch.randn((n, h, w, 256), generator=g, device="cuda").to(torch.bfloat16)
        wp = ops.pack_conv_weight(wt, cout, cin)
        full = torch.zeros((n, h, w, cout), device="cuda", dtype=torch.bfloat16)
        ops.conv2d_bf16(x, wp, n_tile=cout, res1=(res, 16), out_raw=(full, 0))
        praw = torch.zeros((n, h // 2, w // 2, 256), device="cuda", dtype=torch.bfloat16)
        pact = torch.zeros((n, h // 2, w // 2, 256), device="cuda", dtype=torch.bfloat16)
        ops.conv2d_bf16(x, wp, n_tile=cout, res1=(res, 16), out_raw=(praw, 32), post=(s2, t2, pact, 32), pool2=True)
        torch.cuda.synchronize()
        ref = F.max_pool2d(full.float().permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1)
        assert torch.equal(praw[..., 32:32 + cout].float(), ref)          # bit-exact: max of the same bf16 values
        act = torch.relu(ref * s2 + t2).to(torch.bfloat16).float()
        assert (pact[..., 32:32 + cout].float() - act).abs().max().item() <= act.abs().max().item() * 2.0 ** -7
        assert (praw[..., :32] == 0).all() and (praw[..., 32 + cout:] == 0).all()


def test_conv_upsampled_residual(lib):
    """res_up epilogue: out = conv + res1 + nearest_up2(low) (hourglass up path, paulsenpredictor.py:334-359),
    with the pre / post activations around it; ragged map so that partial tiles are covered."""
    from mvlm_b200 import ops

    torch.backends.cudnn.allow_tf32 = False
    for (n, h, w, cin, cout, with_pre, with_post) in ((2, 32, 32, 128, 128, True, True), (1, 48, 24, 64, 64, False, True),
                                                       (3, 8, 8, 256, 128, True, False), (2, 64, 64, 64, 32, False, False)):
        g = torch.Generator(device="cuda").manual_seed(17 + cout + h)
        x = torch.randn((n, h, w, cin), generator=g, device="cuda").to(torch.bfloat16)
        wt = torch.randn((cout, cin, 3, 3), generator=g, device="cuda") / (cin * 9) ** 0.5
        s1, t1, s2, t2 = (torch.randn((cout,), generator=g, device="cuda") for _ in range(4))
        res = torch.randn((n, h, w, 256), generator=g, device="cuda").to(torch.bfloat16)
        low = torch.randn((n, h // 2, w // 2, 256), generator=g, device="cuda").to(torch.bfloat16)
        wp = ops.pack_conv_weight(wt, cout, cin)
        out_pre = torch.zeros((n, h, w, cout), device="cuda", dtype=torch.bfloat16)
        out_raw = torch.zeros((n, h, w, 256), device="cuda", dtype=torch.bfloat16)
        out_post = torch.zeros((n, h, w, 256), device="cuda", dtype=torch.bfloat16)
        ops.conv2d_bf16(x, wp, n_tile=cout, pre=(s1, t1, out_pre, 0) if with_pre else None, res1=(res, 64),
                        res_up=(low, 96), out_raw=(out_raw, 32), post=(s2, t2, out_post, 32) if with_post else None)
        torch.cuda.synchronize()
        tag = (n, h, w, cin, cout)
        v, A = _ref(x, wt, None, -1, -1)
        if with_pre:
            _check(out_pre, *_affine(v, A, s1, t1), f"out_pre {tag}")
        up = F.interpolate(low[..., 96:96 + cout].double().permute(0, 3, 1, 2), scale_factor=2, mode="nearest").permute(0, 2, 3, 1)
        r = res[..., 64:64 + cout].double()
        v2, A2 = v + r + up, A + r.abs() + up.abs()
        _check(out_raw[..., 32:32 + cout], v2, A2, f"out_raw {tag}")
        assert (out_raw[..., :32] == 0).all() and (out_raw[..., 32 + cout:] == 0).all()
        if with_post:
            _check(out_post[..., 32:32 + cout], *_affine(v2, A2, s2, t2), f"out_post {tag}")


def test_conv_random_shape_sweep(lib):
    """Seeded sweep over ragged map sizes / channel counts / kernel sizes and the epilogue combinations the plan uses
    (both the M = 128 and the M = 64 kernels, stationary and streamed weights): bias + pre + res1 [+ up] + raw + post."""
    from mvlm_b200 import ops

    torch.backends.cudnn.allow_tf32 = False
    rng = torch.Generator().manual_seed(2024)

    def pick(seq):
        return seq[int(torch.randint(0, len(seq), (1,), generator=rng))]

    for case in range(28):
        k = pick([1, 3, 3, 3])
        cin = pick([16, 32, 64, 80, 96, 128, 256])
        cout = pick([32, 64, 64, 128, 128, 256])
        n = pick([1, 2, 3])
        even = case % 2 == 0                      # res_up needs even H, W
        h = int(torch.randint(1, 36, (1,), generator=rng)) * (2 if even else 1)
        w = int(torch.randint(1, 20, (1,), generator=rng)) * (2 if even else 1)
        with_pre, with_post, with_up = pick([True, False]), pick([True, False]), even and pick([True, False])
        g = torch.Generator(device="cuda").manual_seed(100 + case)
        cs_in = max(cin, 64) if cin % 64 else cin
        x = torch.randn((n, h, w, cs_in), generator=g, device="cuda").to(torch.bfloat16)
        wt = torch.randn((cout, cin, k, k), generator=g, device="cuda") / (cin * k * k) ** 0.5
        bias = torch.randn((cout,), generator=g, device="cuda")
        s1, t1, s2, t2 = (torch.randn((cout,), generator=g, device="cuda") for _ in range(4))
        res = torch.randn((n, h, w, cout + 32), generator=g, device="cuda").to(torch.bfloat16)
        low = torch.randn((n, max(h // 2, 1), max(w // 2, 1), cout + 16), generator=g, device="cuda").to(torch.bfloat16)
        wp = ops.pack_conv_weight(wt, cout, cin)
        out_pre = torch.full((n, h, w, cout), float("nan"), device="cuda", dtype=torch.bfloat16)
        out_raw = torch.full((n, h, w, cout + 8), float("nan"), device="cuda", dtype=torch.bfloat16)
        out_post = torch.full((n, h, w, cout), float("nan"), device="cuda", dtype=torch.bfloat16)
        ops.conv2d_bf16(x, wp, cin=cin, n_tile=min(cout, 128), kh=k, kw=k, bias=bias,
                        pre=(s1, t1, out_pre, 0) if with_pre else None, res1=(res, 32),
                        res_up=(low, 16) if with_up else None, out_raw=(out_raw, 8),
                        post=(s2, t2, out_post, 0) if with_post else None)
        torch.cuda.synchronize()
        tag = (case, n, h, w, cin, cout, k, with_pre, with_post, with_up)
        v, A = _ref(x[..., :cin], wt, bias, -(k // 2), -(k // 2))
        if with_pre:
            _check(out_pre, *_affine(v, A, s1, t1), f"out_pre {tag}")
        r = res[..., 32:].double()
        v2, A2 = v + r, A + r.abs()
        if with_up:
            up = F.interpolate(low[..., 16:].double().permute(0, 3, 1, 2), scale_factor=2, mode="nearest").permute(0, 2, 3, 1)
            v2, A2 = v2 + up, A2 + up.abs()
        _check(out_raw[..., 8:], v2, A2, f"out_raw {tag}")
        assert torch.isnan(out_raw[..., :8].float()).all(), tag           # neighbouring channels untouched
        if with_post:
            _check(out_post, *_affine(v2, A2, s2, t2), f"out_post {tag}")


def test_conv_fused_argmax_fast_path_matches_exact_search(lib):
    """The arg-max-only epilogue (unit maximum + position lookup, the conv11 phase kernels) must return the keys of the
    exact per-row search (the variant that also writes the fp32 map), bit for bit: ties (also those created by a large
    bias swallowing the low bits), -inf maps, NaN pixels, +0 / -0, ragged widths and heights."""
    from mvlm_b200 import ops

    torch.backends.cudnn.allow_tf32 = False
    g = torch.Generator(device="cuda").manual_seed(77)
    c = 128
    eye = torch.eye(c, device="cuda").reshape(c, c, 1, 1)
    wp = ops.pack_conv_weight(eye, c, c)
    for case, (n, h, w, co) in enumerate(((2, 64, 32, 128), (1, 40, 20, 73), (3, 8, 8, 128), (2, 36, 44, 80))):
        for kind in ("random", "quantised", "equal", "bias_ties", "neg_inf_bias", "nan", "zeros"):
            x = torch.randn((n, h, w, c), generator=g, device="cuda")
            bias = torch.zeros(c, device="cuda")
            if kind == "quantised":
                x = torch.randint(-2, 3, (n, h, w, c), generator=g, device="cuda").float()
            elif kind == "equal":
                x = torch.full((n, h, w, c), 1.5, device="cuda")
            elif kind == "bias_ties":
                bias = torch.full((c,), 3.0e5, device="cuda")       # ulp(3e5) = 1/32: many different v give equal v + b
            elif kind == "neg_inf_bias":
                bias[::3] = float("-inf")
            elif kind == "nan":
                x[0, h // 2, w // 3, :] = float("nan")              # 0 * NaN: every channel is NaN at that pixel
                x[-1, h - 1, w - 1, 5] = float("nan")
            elif kind == "zeros":
                x = torch.where(torch.rand((n, h, w, c), generator=g, device="cuda") < 0.5, 0.0, -0.0) * 1.0
            xb = x.to(torch.bfloat16)
            keys_exact = torch.zeros((n * co,), device="cuda", dtype=torch.int64)
            keys_fast = torch.zeros((n * co,), device="cuda", dtype=torch.int64)
            out_f32 = torch.zeros((n, co, h, w), device="cuda")
            ops.conv2d_bf16(xb, wp, n_tile=c, kh=1, kw=1, bias=bias, out_f32=out_f32, argmax_keys=keys_exact, cout_real=co)
            ops.conv2d_bf16(xb, wp, n_tile=c, kh=1, kw=1, bias=bias, argmax_keys=keys_fast, cout_real=co)
            torch.cuda.synchronize()
            assert torch.equal(keys_exact, keys_fast), (case, kind)
            if kind in ("random", "quantised", "equal", "bias_ties"):
                idx = 0xFFFFFFFF - (keys_fast.view(n, co) & 0xFFFFFFFF)
                assert torch.equal(idx, out_f32.view(n, co, -1).argmax(dim=-1)), (case, kind)
