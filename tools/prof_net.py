"""Per-op timing of the CNN plan at the headline workload (GPU box): where do the ms go?"""
import ctypes as C
import sys
from collections import defaultdict
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from mvlm_b200 import _lib, build, ops  # noqa: E402
from mvlm_b200.weights import seeded_state_dict  # noqa: E402

build.build()
V = int(sys.argv[1]) if len(sys.argv) > 1 else 100
S = int(sys.argv[2]) if len(sys.argv) > 2 else 256
lib = _lib.load()
net = ops.Hourglass(seeded_state_dict(73, "RGB+depth", 1234), 73, 4, V, S, S)
img = torch.randint(0, 256, (V, S, S, 4), dtype=torch.uint8, device="cuda")
peaks = torch.empty((73, V, 3), dtype=torch.float32, device="cuda")
n = net.num_launches
ms = (C.c_float * n)()
roles = (C.c_double * (8 * n))()
trace_op = -1
for a in sys.argv:
    if a.startswith("--trace="):
        trace_op = int(a.split("=")[1])
trace = (C.c_longlong * (64 * 16))()
_lib.check(lib.mvlm_debug_hourglass_profile(net._h, img.data_ptr(), None, peaks.data_ptr(), 5, ms, roles, trace_op, trace,
                                            torch.cuda.current_stream().cuda_stream), "profile")
if trace_op >= 0:
    lib.mvlm_debug_hourglass_describe(net._h, trace_op, C.create_string_buffer(256), 256)
    print(f"timeline of CTA 0, op {trace_op} (cycles since kernel start): tile | P halo-issued, P weights-issued | "
          "M acc-acquired, M halo-landed, M issued | E acc-ready, E released")
    for t in range(24):
        r = [trace[t * 16 + k] for k in range(16)]
        print(f"  tile {t:2d} | {r[0]:8d} {r[1]:8d} | {r[2]:8d} {r[3]:8d} {r[4]:8d} | pre-wait {r[7]:8d} {r[5]:8d} {r[6]:8d}   "
              f"mma-span {r[4] - r[2]:6d} epi-span {r[6] - r[5]:6d} | unit0: ld {r[8] - r[5]:5d} sts {r[9] - r[8]:5d} "
              f"out {r[10] - r[9]:5d} end {r[11] - r[10]:5d} | unit1: ld {r[12] - r[11]:5d} sts {r[13] - r[12]:5d} "
              f"out {r[14] - r[13]:5d} end {r[15] - r[14]:5d}")
buf = C.create_string_buffer(256)
agg = defaultdict(lambda: [0, 0.0, [0.0] * 8])
total = sum(ms)
for i in range(n):
    lib.mvlm_debug_hourglass_describe(net._h, i, buf, 256)
    d = buf.value.decode()
    agg[d][0] += 1
    agg[d][1] += ms[i]
    for k in range(8):
        agg[d][2][k] += roles[i * 8 + k]
    if "-v" in sys.argv:
        print(f"{i:4d} {ms[i]:8.4f}  {d}")
print(f"total {total:.3f} ms over {n} ops (event-bracketed, so each op pays its launch gap)")
print("roles (kcycles per CTA per op): prod-wait-A/B-empty | mma-wait-operands / acc-free / total | epi-wait-acc-full / total")
for d, (cnt, t, r) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
    r = [x / cnt / 1e3 for x in r]
    rs = f"  P {r[0]:6.0f} {r[1]:6.0f} | M {r[2]:6.0f} {r[3]:6.0f} {r[4]:6.0f} | E {r[5]:6.0f} {r[6]:6.0f}" if d.startswith("conv") else ""
    print(f"{t:8.3f} ms {100 * t / total:5.1f}%  x{cnt:3d}  {t / cnt * 1000:8.1f} us/op  {d:62s}{rs}")
