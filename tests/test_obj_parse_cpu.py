"""CPU: the per-line code of the GPU OBJ parser (csrc/obj_parse.cu, __host__ __device__, run serially through
mvlm_debug_obj_parse_lines) == the host parser mvlm_obj_load, bit for bit: numbers compared as uint32 (NaN bits count),
face corners through the host's index resolution and vertex de-duplication, errors by message."""
import ctypes as C
import decimal
import random

import numpy as np
import pytest

from mvlm_b200 import synth
from mvlm_b200.io_obj import load_obj

OK, BAD, FALLBACK = 0, 1, 2
V, VT, F = 1, 2, 3


def debug_lines(lib, text: bytes):
    n = text.count(b"\n") + 1
    kind, status, n_tris = (np.zeros(n, np.int32) for _ in range(3))
    values = np.zeros((n, 3), np.float32)
    cap = 3 * (len(text) // 2 + 2)
    corners = np.zeros((cap, 2), np.int64)
    n_lines = C.c_int()
    rc = lib.mvlm_debug_obj_parse_lines(text, len(text), n, C.byref(n_lines), kind.ctypes.data, status.ctypes.data,
                                        values.ctypes.data, n_tris.ctypes.data, corners.ctypes.data, cap)
    assert rc == 0, lib.mvlm_last_error()
    m = n_lines.value
    return kind[:m], status[:m], values[:m], n_tris[:m], corners[:int(n_tris[:m].sum()) * 3]


def load_from_lines(lib, text: bytes, path: str):
    """What the GPU parser returns for `text`: the per-line results, resolved like mvlm_obj_load.
    Returns (verts, uvs | None, tris), or the error message, or FALLBACK."""
    kind, status, values, n_tris, corners = debug_lines(lib, text)
    if (status == FALLBACK).any():
        return FALLBACK
    if (status == BAD).any():
        return f"mvlm_obj_load: malformed v / vt / f line in {path}"
    pos, tex = values[kind == V], values[kind == VT][:, :2]
    if len(pos) == 0:
        return f"File {path} does not contain any points."
    v_seen = np.cumsum(kind == V) - (kind == V)
    vt_seen = np.cumsum(kind == VT) - (kind == VT)
    tri_line = np.repeat(np.arange(len(kind)), n_tris)
    a, b = corners[:, 0], corners[:, 1]
    vs, ts = np.repeat(v_seen[tri_line], 3), np.repeat(vt_seen[tri_line], 3)
    vi = np.where(a > 0, a - 1, vs + a)
    ti = np.where(b == 0, -1, np.where(b > 0, b - 1, ts + b))
    bad_v = ~((vi >= 0) & (vi < len(pos)))
    bad_t = ~((ti >= -1) & (ti < len(tex)))
    bad = np.flatnonzero(bad_v | bad_t)
    if len(bad):
        i = bad[0]
        if bad_v[i]:
            return f"mvlm_obj_load: face references vertex {a[i]} of {len(pos)} in {path}"
        return f"mvlm_obj_load: face references vt {b[i]} of {len(tex)} in {path}"
    if not (ti >= 0).any():
        return pos, None, vi.reshape(-1, 3).astype(np.int32)
    keys = (vi.astype(np.uint64) << np.uint64(32)) | (ti + 1).astype(np.uint64)
    uniq, inv = np.unique(keys, return_inverse=True)
    uv_of = (uniq & np.uint64(0xFFFFFFFF)).astype(np.int64) - 1
    verts = pos[(uniq >> np.uint64(32)).astype(np.int64)]
    uvs = np.where(uv_of[:, None] >= 0, tex[np.clip(uv_of, 0, None)], np.float32(0)).astype(np.float32)
    return verts, uvs, inv.reshape(-1, 3).astype(np.int32)


def check_file(lib, path, text: bytes):
    path.write_bytes(text)
    got = load_from_lines(lib, text, str(path))
    try:
        ref = load_obj(path, load_texture=False, n_threads=1)
    except ValueError as e:
        assert got == FALLBACK or got == str(e), (got, str(e))
        return got
    if got == FALLBACK:
        return got
    assert not isinstance(got, str), got
    verts, uvs, tris = got
    assert np.array_equal(verts.view(np.uint32), ref.verts.view(np.uint32))
    assert (uvs is None) == (ref.uvs is None)
    if uvs is not None:
        assert np.array_equal(uvs.view(np.uint32), ref.uvs.view(np.uint32))
    assert np.array_equal(tris, ref.tris)
    return got


# the OBJ strings of tests/test_host_cpu.py, and the cases of the host parser's language
CORPUS = {
    "forms.obj": "v 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nv 2 2 2\nvt 0 0\nvt 1 0\nvt 1 1\nvt 0 1\nvn 0 0 1\n"
                 "f 1/1/1 2/2/1 3/3/1\nf 1//1 3//1 4//1\nf 2/2 5/4 3\nf 1 2 3 4\n",
    "relative.obj": "v 0 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\nvt 1 0\nvt 0 1\nf -3/-3 -2/-2 -1/-1\n",
    "crlf.obj": "# comment\r\nv +1.5e0 -2.25E-1 3\r\nv 1e-3 2 3\r\nv 0.1 0.2 0.3\r\n\r\nf 1 2 3\r\n",
    "nouv.obj": "v 0 0 0\nv 1 0 0\nv 0 1 0\nv 9 9 9\nvt 0 0\nf 1 2 3\n",
    "b.obj": "v 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nvt 0 0\nvt 1 0\nvt 1 1\nvt 0 1\nvt 0.5 0.5\n"
             "f 1/1 2/2 3/3\nf 1/5 3/3 4/4\n",
    "c.obj": "v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\nf -3 -2 -1\n",
    "d.obj": "# empty\n",
    "n.obj": "v 0 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\nvt 1 1\nusemtl m\nf 1 2 3\n",
    "p.obj": "v 0 0 0\nv 1 0 0\nv 2 1 0\nv 1 2 0\nv 0 1 0\nf 1 2 3 4 5\n",
    "bad.obj": "v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 7\n",
    "bad_vt.obj": "v 0 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\nf 1/1 2/1 3/-2\n",
    "bad_neg.obj": "v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 -4\nf 1 2 9\n",
    "malformed.obj": "v 0 0 0\nv 1 x 0\nv 0 1 0\nf 1 2 3\nf 1 2 99\n",
    "malformed_f.obj": "v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3x\n",
    "no_final_newline.obj": "v 0 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\nvt 1 0\nf 1/1 2/2 3/1",
    "tabs.obj": "v\t0 0 0\n\tv 1 1 1\nv 0 0 0\nv 1 0 0\t\nv 0 1 0 1 0.5 0.2\nf 2 3 4 \n",
    "tokens.obj": "v 1-2-3\nv .5 5. -0\nv 1e 1 1\nvt 1-2\nf 1-2-3\nf 1/1-2-3\nf 0 1 2\nf 1/0 2 3\nf 3/ 1// 2/1/\n",
    "vt_minus1.obj": "v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1/-1 2 3\n",
    "points_only.obj": "v 0 0 0\nv 1 0 0\n",
    "long_digits.obj": "v 1.00000005960464477539062500001 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\n",
    "empty.obj": "",
}


@pytest.mark.parametrize("name", sorted(CORPUS))
def test_corpus_matches_host(lib, tmp_path, name):
    got = check_file(lib, tmp_path / name, CORPUS[name].encode())
    if name == "long_digits.obj":
        assert got == FALLBACK


def test_synthetic_scan_matches_host(lib, tmp_path):
    v, uv, t = synth.face_mesh(grid=60, seed=3)
    synth.write_obj(tmp_path / "s.obj", v, uv, t, None)
    assert check_file(lib, tmp_path / "s.obj", (tmp_path / "s.obj").read_bytes()) != FALLBACK


def _num(rng: random.Random) -> str:
    r = rng.random()
    if r < 0.5:
        return f"{rng.uniform(-100, 100):.6f}"
    if r < 0.7:
        return str(rng.randint(-5, 5))
    if r < 0.8:
        return f"{rng.uniform(-1, 1):.9g}"
    if r < 0.98:
        return f"{rng.uniform(-1, 1):.17g}"
    return rng.choice(["1e3", "-2.5E-2", "+7", ".5", "5.", "-0", "nan", "inf", "1e", "0x1p3"])


def _ws(rng):
    return "".join(rng.choice([" ", " ", "\t", "\r"]) for _ in range(rng.randint(1, 2)))


def _random_obj(seed: int) -> str:
    rng = random.Random(seed)
    nv, nvt = rng.randint(3, 30), rng.randint(0, 20)
    lines, v_seen, vt_seen = [], 0, 0
    order = ["v"] * nv + ["vt"] * nvt + ["f"] * rng.randint(0, 25) + ["x"] * rng.randint(0, 8)
    rng.shuffle(order)
    for what in order:
        if what == "v":
            lines.append("v " + _ws(rng).join(_num(rng) for _ in range(rng.choice([3, 3, 4, 5, 6]))) + _ws(rng) * rng.randint(0, 1))
            v_seen += 1
        elif what == "vt":
            lines.append("vt " + _ws(rng).join(_num(rng) for _ in range(rng.choice([2, 2, 3]))))
            vt_seen += 1
        elif what == "f":
            toks = []
            for _ in range(rng.randint(1, 8)):
                a = rng.randint(1, nv) if rng.random() < 0.7 or not v_seen else -rng.randint(1, v_seen)
                if rng.random() < 0.02:
                    a = nv + 5
                form = rng.randrange(4) if nvt else rng.choice([0, 2])
                b = rng.randint(1, max(nvt, 1)) if rng.random() < 0.7 or not vt_seen else -rng.randint(1, vt_seen)
                toks.append([f"{a}", f"{a}/{b}", f"{a}//{rng.randint(1, 9)}", f"{a}/{b}/{rng.randint(1, 9)}"][form])
            lines.append("f " + _ws(rng).join(toks))
        else:
            lines.append(rng.choice(["# comment v 1 2 3", "vn 0 0 1", "usemtl skin", " v 1 2 3", "v\t1 2 3", "o obj",
                                     "", "g group", "s off", "vp 0.5"]))
    eol = "\r\n" if rng.random() < 0.3 else "\n"
    text = eol.join(lines)
    return text if rng.random() < 0.3 else text + eol


def test_random_files_match_host(lib, tmp_path):
    outcomes = {"arrays": 0, "error": 0}
    for seed in range(400):
        got = check_file(lib, tmp_path / f"r{seed}.obj", _random_obj(seed).encode())
        outcomes["error" if isinstance(got, str) else "arrays"] += got != FALLBACK
    assert outcomes["arrays"] > 100 and outcomes["error"] > 20, outcomes


PROBES = ["1e400", "-1e400", "1e-400", "2e-324", "4.9e-324", "1e-320", "0." + "0" * 44 + "1", "nan", "nan(123)", "-nan",
          "inf", "INF", "infinity", "-inf", "-0", "3.4028236e38", ".5", "5.", "0x1p3", "1e", "-", "+-1", "++1",
          "nan(", "nan(a b)", "-.", ".", "0e999999999999", "1e-99999999999", "1e+", "1E-", "-infinityx", "Infinit",
          "nAn()", "-nan(_x9)", "00000000000000000000000000.5", "0.000000000000000000000000000000000000001e39",
          "9007199254740993", "9007199254740992e-22", "1e23", "8.98846567431158e307", "1.7976931348623157e308",
          "1.7976931348623158e308", "1.7976931348623159e308", "2.2250738585072011e-308", "2.2250738585072012e-308",
          "4.9406564584124654e-324", "2.4703282292062327e-324", "2.4703282292062328e-324", "1.4e-45", "7e-46",
          "7.006492321624085e-46", "1.1754942e-38", "3.4028235677973366e38", "3.4028235677973367e38", "1e22", "1e-22",
          "123456789012345678", "1234567890123456789", "18446744073709551615", "0.1e-342", "1e-343", "10e-344"]


def _tokens(n: int, seed: int) -> list[str]:
    """Random decimal tokens: 1-19-digit mantissas with exponents across the double range, %.6f / %.9g / %.17g writes
    of random floats and doubles, and midpoints between neighbouring floats and between neighbouring doubles."""
    rng = np.random.default_rng(seed)
    out = []
    q = n // 5
    digits = rng.integers(1, 20, q)
    exps = rng.integers(-360, 330, q)
    points = rng.random(q)
    for d, e, pnt in zip(digits, exps, points):
        m = "".join(map(str, rng.integers(0, 10, d)))
        if pnt < 0.4:
            k = int(rng.integers(0, d + 1))
            m = m[:k] + "." + m[k:]
        out.append(("-" if pnt < 0.2 else "") + m + ("" if pnt > 0.9 else f"e{e}"))
    f32 = rng.integers(0, 2 ** 32, q, dtype=np.uint64).astype(np.uint32).view(np.float32)
    f32 = f32[np.isfinite(f32)]
    f64 = rng.integers(0, 2 ** 63, q, dtype=np.uint64).view(np.float64)
    out += [f"{x:.6f}" for x in f32[: q // 3].astype(np.float64)]
    out += [f"{x:.9g}" for x in f32[q // 3:].astype(np.float64)]
    out += [f"{x:.17g}" for x in f64]
    # midpoints between neighbouring floats: exact in double (repr round-trips), so the cast sees the tie
    f = np.abs(f32[np.isfinite(f32)])
    nxt = np.nextafter(f, np.float32(np.inf))
    mid = (f.astype(np.float64) + nxt.astype(np.float64)) / 2
    out += [repr(float(x)) for x in mid[np.isfinite(mid)]]
    # midpoints between neighbouring doubles, written to 19 significant digits just below / above the tie (the exact
    # midpoint needs more digits: that token takes the host fallback)
    decimal.getcontext().prec = 60
    dd = np.abs(f64[np.isfinite(f64)])[: n // 10]
    for x in dd:
        y = np.nextafter(x, np.inf)
        if not np.isfinite(y):
            continue
        m = (decimal.Decimal(float(x)) + decimal.Decimal(float(y))) / 2
        out.append(f"{m:.18e}")
        out.append(f"{m.next_plus():.18e}" if rng.random() < 0.5 else f"{m.next_minus():.18e}")
    return out


def test_token_corpus_matches_from_chars(lib, tmp_path):
    """>= 1e6 number tokens, three per `v` line: every line the GPU code accepts gives the host's float bits; every
    line it rejects is rejected by the host too (checked one file per line on a sample); only tokens of more than 19
    significant digits take the host fallback."""
    toks = PROBES * 4 + _tokens(1_020_000, seed=7)
    assert len(toks) >= 1_000_000
    rng = random.Random(11)
    rng.shuffle(toks)
    toks += ["0"] * (-len(toks) % 3)
    lines = [f"v {toks[i]} {toks[i + 1]} {toks[i + 2]}" for i in range(0, len(toks), 3)]
    kind, status, values, _, _ = debug_lines(lib, ("\n".join(lines) + "\n").encode())
    assert len(kind) == len(lines) and (kind == V).all()
    ok = np.flatnonzero(status == OK)
    good = tmp_path / "good.obj"
    good.write_text("\n".join(lines[i] for i in ok) + "\n")
    ref = load_obj(good, load_texture=False)
    assert np.array_equal(values[ok].view(np.uint32), ref.verts.view(np.uint32))
    # sig digits: the fallback is taken for long tokens and for nothing else
    bad = np.flatnonzero(status == BAD)
    fb = np.flatnonzero(status == FALLBACK)
    assert len(ok) > 0.5 * len(lines) and len(bad) > 1000 and len(fb) > 1000
    for i in list(fb[:2000]):
        sig = [len(t.lstrip("+-").split("e")[0].split("E")[0].replace(".", "").lstrip("0")) for t in lines[i].split()[1:]]
        assert max(sig) > 19, lines[i]
    one = tmp_path / "one.obj"
    for i in list(bad[:1500]) + [j for j in bad if any(p in lines[j].split() for p in PROBES)][:1500]:
        one.write_text(lines[i] + "\n")
        with pytest.raises(ValueError, match="malformed"):
            load_obj(one, load_texture=False)


def test_probe_results(lib):
    """The host's from_chars results for the edge cases (GCC 13 / libstdc++), as float bits after the cast."""
    want = {"4.9e-324": 0x00000000, "1e-320": 0x00000000, "0." + "0" * 44 + "1": 0x00000001, "nan": 0x7fc00000,
            "nan(123)": 0x7fc00000, "-nan": 0xffc00000, "inf": 0x7f800000, "INF": 0x7f800000, "infinity": 0x7f800000,
            "-inf": 0xff800000, "-0": 0x80000000, "3.4028236e38": 0x7f800000, ".5": 0x3f000000, "5.": 0x40a00000}
    for tok, bits in want.items():
        _, status, values, _, _ = debug_lines(lib, f"v 0 0 {tok}".encode())
        assert status[0] == OK and values[0].view(np.uint32)[2] == bits, tok
    for tok in ["1e400", "-1e400", "1e-400", "2e-324", "-"]:
        assert debug_lines(lib, f"v 0 0 {tok}".encode())[1][0] == BAD, tok
    for tok in ["0x1p3", "1e"]:  # partial consume: an error unless it is the last number of the line
        assert debug_lines(lib, f"v 0 0 {tok}".encode())[1][0] == OK
        assert debug_lines(lib, f"v 0 {tok} 0".encode())[1][0] == BAD
    assert debug_lines(lib, b"v 0 0 1.00000005960464477539062500001")[1][0] == FALLBACK  # host: 3f800000
