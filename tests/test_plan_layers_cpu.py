"""CPU: the CNN plan, op by op, against the op list the reference model defines (tests/plan_ref.py), and the workspace
packing against lifetimes derived from the op records alone.

A wrong BatchNorm slice, residual channel offset or buffer, or a buffer the packer hands to someone else while it is
still read, can stay under the statistical bars of the end-to-end tests; here it fails and the message names the op.
"""
import pytest

from mvlm_b200 import ops as mops
from plan_ref import READS, expected_ops, plan_ops
from test_plan_build_cpu import SIZES

# odd landmark counts (Lp = 32, 64, 128 from 1, 40, 100), non-square images, a 3 x 1 bottom map (192 x 64)
EXTRA = [(1, 1, 1, 64, 64), (5, 1, 1, 64, 192), (40, 3, 2, 192, 64), (100, 3, 1, 64, 64), (17, 2, 3, 128, 64),
         (128, 4, 1, 256, 256), (84, 2, 3, 128, 64)]
SHAPES = sorted(SIZES) + EXTRA
CHECKED = ("h", "w", "cin", "cout_pad", "kh", "kw", "y_off0", "x_off0", "pool2", "aux_mode", "cout_real")


def _name(i, op):
    return f"op {i} ({op['kind']} {op['layer']}{' phase %s' % (op['phase'],) if op['phase'][0] >= 0 else ''})"


def check_plan(recs, bufs, exp, tensors, n_landmarks, n_views):
    """Every mismatch between the plan's records and the expected list, as messages naming the op."""
    errs = []
    if len(recs) != len(exp):
        return [f"{len(recs)} ops in the plan, {len(exp)} expected"]
    bound, owner = {}, {}
    for i, (r, e) in enumerate(zip(recs, exp)):
        tag = _name(i, e)
        for k in ("kind", "layer", "bias", "phase", "terms"):
            if r[k] != e[k]:
                errs.append(f"{tag}: {k} {r[k]!r}, expected {e[k]!r}")
        for k in CHECKED:
            if k in e and r[k] != e[k]:
                errs.append(f"{tag}: {k} {r[k]}, expected {e[k]}")
        want = {**e["reads"], **e["writes"]}
        if set(r["operands"]) != set(want):
            errs.append(f"{tag}: operands {sorted(r['operands'])}, expected {sorted(want)}")
            continue
        for name, (tensor, co) in want.items():
            buf, cs, rco, _ = r["operands"][name]
            c = tensors[tensor][2]
            if buf < 0:
                errs.append(f"{tag}: {name} is not the start of a plan buffer")
                continue
            if (cs, rco) != (c, co):
                errs.append(f"{tag}: {name} reads/writes {tensor} at channel stride {cs} offset {rco}, expected {c} {co}")
            if bound.setdefault(tensor, buf) != buf:
                errs.append(f"{tag}: {name} uses buffer {buf} for {tensor}, which lives in buffer {bound[tensor]}")
            if owner.setdefault(buf, tensor) != tensor:
                errs.append(f"{tag}: {name} puts {tensor} into buffer {buf}, which holds {owner[buf]}")
    for tensor, buf in bound.items():
        h, w, c = tensors[tensor]
        need = n_views * n_landmarks * 8 if tensor == "keys" else n_views * h * w * c * 2
        if bufs[buf][0] != (need + 1023) // 1024 * 1024:
            errs.append(f"buffer {buf} ({tensor}) has {bufs[buf][0]} bytes for {need}")
    return errs


def check_lifetimes(recs, bufs):
    """Lifetimes from the records only: buffers live at the same time never share workspace bytes, and no op reads a
    byte range that another buffer wrote after the read buffer's producer did."""
    errs, clobbered = [], []
    first, last = {}, {}
    for i, r in enumerate(recs):
        for name, (buf, *_rest) in r["operands"].items():
            first.setdefault(buf, i)
            last[buf] = i
    live = sorted(first)

    def overlap(a, b):
        return bufs[a][1] < bufs[b][1] + bufs[b][0] and bufs[b][1] < bufs[a][1] + bufs[a][0]

    for x in range(len(live)):
        for y in range(x + 1, len(live)):
            a, b = live[x], live[y]
            if first[a] <= last[b] and first[b] <= last[a] and overlap(a, b):
                errs.append(f"buffers {a} (ops {first[a]}..{last[a]}) and {b} (ops {first[b]}..{last[b]}) share "
                            f"workspace bytes")
    writes = [{buf for name, (buf, *_r) in r["operands"].items() if name not in READS} for r in recs]
    for i, r in enumerate(recs):
        for name, (buf, *_r) in r["operands"].items():
            if name not in READS and not (name == "keys" and r["kind"] == "peaks"):
                continue
            prod = max((j for j in range(i) if buf in writes[j]), default=None)
            if prod is None:
                errs.append(f"op {i} ({r['kind']} {r['layer']}): {name} reads buffer {buf} before any op wrote it")
                continue
            for j in range(prod + 1, i):
                for other in writes[j]:
                    if other != buf and overlap(buf, other):
                        clobbered.append(f"op {i} ({r['kind']} {r['layer']}): {name} reads buffer {buf} (written by op "
                                    f"{prod}) after op {j} ({recs[j]['kind']} {recs[j]['layer']}) wrote buffer "
                                    f"{other} over it")
    return clobbered + errs


@pytest.mark.parametrize("fusion", [True, False], ids=["fused", "unfused"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "L%d-c%d-v%d-%dx%d" % s)
def test_plan_ops_match_reference_and_packing_respects_lifetimes(lib, shape, fusion):
    n_landmarks, cin, views, h, w = shape
    with mops._plan_env(MVLM_HG_ELT_FUSION="1" if fusion else "0"):
        recs, bufs = plan_ops(lib, n_landmarks, cin, views, h, w)
    exp, tensors = expected_ops(n_landmarks, cin, h, w, fusion)
    assert len(recs) == (144 if fusion else 155)
    errs = check_plan(recs, bufs, exp, tensors, n_landmarks, views)
    assert not errs, "\n".join(errs[:20])
    errs = check_lifetimes(recs, bufs)
    assert not errs, "\n".join(errs[:20])
    # the records' workspace offsets are the packed ones
    for i, r in enumerate(recs):
        for name, (buf, _cs, _co, ws) in r["operands"].items():
            assert ws == bufs[buf][1], (i, name)
    assert max(o + b for b, o in bufs) == lib.mvlm_hourglass_workspace_bytes(n_landmarks, cin, views, h, w)


def test_checks_name_the_wrong_op():
    """The checkers report a swapped BatchNorm, a shifted residual slice and a clobbered buffer, naming the op."""
    exp, tensors = expected_ops(73, 4, 64, 64)
    ids = {t: k for k, t in enumerate(tensors)}
    recs, bufs = [], []
    for t, (h, w, c) in tensors.items():
        bufs.append((((2 * h * w * c if t != "keys" else 73 * 8) + 1023) // 1024 * 1024, 0))
    off = 0
    for k, (b, _) in enumerate(bufs):
        bufs[k] = (b, off)
        off += b
    for e in exp:
        ops_ = {n: (ids[t], tensors[t][2], co, bufs[ids[t]][1]) for n, (t, co) in {**e["reads"], **e["writes"]}.items()}
        recs.append({**e, "operands": ops_, "cin": e.get("cin", 0)})
    assert check_plan(recs, bufs, exp, tensors, 73, 1) == [] and check_lifetimes(recs, bufs) == []
    i = next(k for k, e in enumerate(exp) if e["layer"] == "hg1.rb5.conv2")
    bad = [dict(r) for r in recs]
    bad[i]["terms"] = dict(bad[i]["terms"], pre=("hg1.rb5.bn2", 0))
    assert any(m.startswith(f"op {i} (conv hg1.rb5.conv2)") for m in check_plan(bad, bufs, exp, tensors, 73, 1))
    bad = [dict(r) for r in recs]
    buf, cs, co, ws = bad[i]["operands"]["res1"]
    bad[i]["operands"] = dict(bad[i]["operands"], res1=(buf, cs, co + 8, ws))
    assert any("res1" in m and m.startswith(f"op {i} ") for m in check_plan(bad, bufs, exp, tensors, 73, 1))
    # conv7 writing sum_temp over its own input x6
    x6, out = ids["x6"], ids["sum_temp"]
    moved = list(bufs)
    moved[out] = (moved[out][0], moved[x6][1])
    errs = check_lifetimes(recs, moved)
    assert any(f"buffers {x6} " in m and f"and {out} " in m for m in errs), errs[:5]
