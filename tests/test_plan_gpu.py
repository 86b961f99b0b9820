"""Whole-plan variants of the CNN that must not change a single bit: the packed workspace against one buffer per tensor,
and the producer-epilogue pool / activation copies against the stand-alone passes.  The default plan is in turn checked
against the reference-pinned oracle in tests/test_hourglass_gpu.py.
"""
import pytest
import torch

from mvlm_b200.weights import IMAGE_CHANNELS, seeded_state_dict

pytestmark = pytest.mark.gpu

PROBES = ("x1", "y3", "r3", "hg1", "sum_temp", "x10")


def _build(env, *args):
    from mvlm_b200 import ops

    with ops._plan_env(**env):
        return ops.Hourglass(*args, keep_probes=True)


def test_workspace_packing_is_bit_identical_and_small(lib):
    """Buffer reuse (hourglass.cu, ws_alloc / assign_offsets) changes addresses only: peaks and heat maps of the packed
    plan equal those of the plan where every buffer has its own memory; the headline plan fits 6 GB."""
    from mvlm_b200 import ops

    assert lib.mvlm_hourglass_workspace_bytes(73, 4, 100, 256, 256) <= 6e9
    sd = seeded_state_dict(73, "RGB+depth", seed=1234)
    g = torch.Generator().manual_seed(3)
    img = torch.randint(0, 256, (6, 128, 128, 4), generator=g, dtype=torch.uint8).cuda()
    args = (sd, 73, 4, 6, 128, 128)
    flat = _build({"MVLM_HG_NO_REUSE": "1"}, *args)
    packed = ops.Hourglass(*args)
    assert packed.workspace.numel() < 0.35 * flat.workspace.numel()
    pk0, hm0 = flat.forward(img, want_heatmaps=True)
    for _ in range(2):
        pk1, hm1 = packed.forward(img, want_heatmaps=True)
        torch.cuda.synchronize()
        assert torch.equal(pk0.view(torch.int32), pk1.view(torch.int32))
        assert torch.equal(hm0.view(torch.int32), hm1.view(torch.int32))
    with pytest.raises(Exception):
        packed.probe("r3")


@pytest.mark.parametrize("n_landmarks,mode,size,views", [(73, "RGB+depth", 128, 3), (84, "geometry+depth", 64, 2),
                                                        (73, "RGB", 256, 2)])
def test_fused_pool_and_act_copies_equal_standalone_passes(lib, n_landmarks, mode, size, views):
    """The hourglass max-pools (paulsenpredictor.py:309-329) and the BatchNorm+ReLU copy of conv4's resample branch
    (:263-265) written by their producers' epilogues (ConvEpilogue::aux_mode, the default plan) == the stand-alone
    pool2_act / bn_relu passes of MVLM_HG_ELT_FUSION=0: every probe tensor, the heat maps and the peaks bit-identical."""
    sd = seeded_state_dict(n_landmarks, mode, seed=77)
    cin = IMAGE_CHANNELS[mode]
    g = torch.Generator().manual_seed(13)
    img = torch.randint(0, 256, (views, size, size, 4), generator=g, dtype=torch.uint8)
    img[..., cin:] = 0
    img = img.cuda()
    args = (sd, n_landmarks, cin, views, size, size)
    unfused = _build({"MVLM_HG_ELT_FUSION": "0"}, *args)
    fused = _build({"MVLM_HG_ELT_FUSION": "1"}, *args)
    assert fused.num_launches == unfused.num_launches - 11   # ten max-pools and one BatchNorm+ReLU pass are gone
    pk0, hm0 = unfused.forward(img, want_heatmaps=True)
    pk1, hm1 = fused.forward(img, want_heatmaps=True)
    torch.cuda.synchronize()
    for name in PROBES:
        assert torch.equal(unfused.probe(name).view(torch.int16), fused.probe(name).view(torch.int16)), name
    assert torch.equal(hm0.view(torch.int32), hm1.view(torch.int32))
    assert torch.equal(pk0.view(torch.int32), pk1.view(torch.int32))
