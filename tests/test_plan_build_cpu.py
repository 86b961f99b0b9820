"""CPU: the plan's size queries, pinned.  The workspace bytes follow from every buffer's size and first / last use and
the FLOPs from every convolution the plan emits, so a change in how the plan is built that moves either shows here."""
import pytest

from mvlm_b200 import ops

# (L, cin, V, H, W): (workspace bytes, algorithmic FLOPs per view)
SIZES = {
    (73, 4, 100, 256, 256): (4404019200, 146105827328),
    (84, 2, 100, 256, 256): (4404019200, 150483501056),
    (73, 4, 8, 256, 256): (352321536, 146105827328),
    (73, 3, 2, 64, 64): (5505024, 9126895616),
    (84, 1, 200, 512, 512): (35232153600, 601632014336),
    (73, 4, 6, 128, 128): (66060288, 36526456832),
    (5, 4, 3, 64, 128): (16515072, 15555936256),
}

# plan switches: workspace bytes at (73, 4, 100, 256, 256) and (73, 4, 6, 128, 128)
SWITCHES = {
    "MVLM_HG_KEEP_PROBES": ("1", 8021606400, 120324096),
    "MVLM_HG_NO_REUSE": ("1", 23057672192, 345868288),
    "MVLM_HG_ELT_FUSION": ("0", 4404019200, 66060288),
}


@pytest.mark.parametrize("shape", sorted(SIZES))
def test_workspace_and_flops_are_pinned(lib, shape):
    l, cin, v, h, w = shape
    ws, flops = SIZES[shape]
    assert lib.mvlm_hourglass_workspace_bytes(l, cin, v, h, w) == ws
    assert lib.mvlm_hourglass_flops_per_view(l, cin, h, w) == flops


@pytest.mark.parametrize("name", sorted(SWITCHES))
def test_plan_switch_workspace_is_pinned(lib, name):
    value, big, small = SWITCHES[name]
    with ops._plan_env(**{name: value}):
        assert lib.mvlm_hourglass_workspace_bytes(73, 4, 100, 256, 256) == big
        assert lib.mvlm_hourglass_workspace_bytes(73, 4, 6, 128, 128) == small
