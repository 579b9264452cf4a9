"""The per-stage numerics model (tests/quant_model.py) and its stage comparator, on the CPU.

1. Composing the stage functions reproduces the end-to-end model bit for bit (a restatement of the network as one
   function is kept here as the fixed point of that refactor).
2. The comparator passes the noise of a different summation order (the same stage accumulated in fp32 and in fp64) and
   fails the local defects that global pooling hides from the descriptor bar: a 64-channel block of one 8x16 tile off by
   10 %, the last (ragged) output row zeroed, one 8x16 tile zeroed - and a small shift of one channel, which only the
   per-channel mean statistic sees."""
import pytest
import torch
import torch.nn.functional as F

import quant_model as QM
import synthdata as synth
from oracle import dir_oracle as O
from conftest import rel_l2


@torch.no_grad()
def _extract_monolithic(x, sd, arch="resnet50_rmac", fuse_shortcut=True, **head_kw):
    """The Bottleneck network of quant_model as one function, as it was written before the split into stages."""
    h, fold, conv = QM.h, QM._fold, QM._conv
    blocks = O.BLOCKS[arch.split("_")[0]]
    s, b = fold(sd, "bn1")
    t = conv(h(x), sd["conv1.weight"], s, b, stride=2, padding=3)
    t = F.max_pool2d(t, kernel_size=3, stride=2, padding=1)
    for li, nblk in enumerate(blocks, start=1):
        for bi in range(nblk):
            p = "layer%d.%d." % (li, bi)
            stride = 2 if (li > 1 and bi == 0) else 1
            s1, b1 = fold(sd, p + "bn1")
            s2, b2 = fold(sd, p + "bn2")
            s3, b3 = fold(sd, p + "bn3")
            t1 = conv(t, sd[p + "conv1.weight"], s1, b1)
            t2 = conv(t1, sd[p + "conv2.weight"], s2, b2, stride=stride, padding=1)
            if bi == 0:
                sdn, bdn = fold(sd, p + "downsample.1")
                if fuse_shortcut:
                    y = F.conv2d(t2, h(sd[p + "conv3.weight"] * s3.view(-1, 1, 1, 1))) + \
                        F.conv2d(t, h(sd[p + "downsample.0.weight"] * sdn.view(-1, 1, 1, 1)), stride=stride)
                    t = h(F.relu(y + (b3 + bdn).view(1, -1, 1, 1)))
                else:
                    r = conv(t, sd[p + "downsample.0.weight"], sdn, bdn, stride=stride, relu=False)
                    t = conv(t2, sd[p + "conv3.weight"], s3, b3, res16=r)
            else:
                t = conv(t2, sd[p + "conv3.weight"], s3, b3, res16=t)
    return O.head(t, sd, **head_kw)


@pytest.mark.parametrize("fused", [True, False], ids=["fused_shortcut", "two_convs"])
def test_stage_functions_compose_to_the_model_bit_for_bit(fused):
    sd = synth.make_state_dict("resnet50_rmac", seed=4)
    x = synth.make_images(2, 100, 132, seed=5)
    ref = _extract_monolithic(x, sd, fuse_shortcut=fused, squeeze=False)
    assert torch.equal(QM.extract(x, sd, fuse_shortcut=fused, squeeze=False), ref)
    t = QM.stem(x, sd)
    for li in range(1, 5):
        # a stage takes its input as the GPU tap holds it: NHWC fp16
        t = QM.stage(QM.nchw(t.permute(0, 2, 3, 1).half()), sd, "resnet50_rmac", li, fuse_shortcut=fused)
    assert torch.equal(O.head(t, sd, squeeze=False), ref)


def test_basic_block_and_fpn_stages_follow_the_oracle():
    """The BasicBlock stages and the FPN lateral carry the same roundings: against the fp32 oracle they land at the
    fp16 level (well inside the descriptor bar, not at fp32 level)."""
    x = synth.make_images(2, 128, 96, seed=6)
    sd = synth.make_state_dict("resnet18_rmac", seed=2)
    err = rel_l2(O.head(QM.stages(x, sd, "resnet18_rmac")["layer4"], sd).numpy(), O.extract(x, sd, "resnet18_rmac").numpy())
    assert 1e-5 < err < 1e-3, err
    sd = synth.make_state_dict("resnet50_fpn_rmac", seed=3)
    st = QM.stages(x, sd, "resnet50_fpn_rmac")
    _, ref = O.trunk(x, sd, "resnet50", return_stages=True)
    c5 = F.relu(F.conv2d(F.interpolate(ref["layer4"], size=ref["layer3"].shape[-2:], mode="nearest"), sd["conv1x5.weight"]))
    ref_c4 = F.relu(F.conv2d(ref["layer3"] + c5, sd["conv3c4.weight"], None, padding=1))
    err = rel_l2(QM.fpn_c4(st["layer3"], st["layer4"], sd).numpy(), ref_c4.numpy())
    assert 1e-5 < err < 1e-2, err


@pytest.fixture(scope="module")
def r50_stages():
    sd = synth.make_state_dict("resnet50_rmac", seed=7)
    x = synth.make_images(1, 200, 328, seed=8)
    return sd, x, QM.stages(x, sd, "resnet50_rmac")


def test_comparator_passes_summation_order_noise(r50_stages):
    """Every stage accumulated in fp64 from the fp32 model's previous stage: the summation-order noise the kernels add
    is of this kind, and must pass all three bars."""
    sd, x, st = r50_stages
    prev = {"layer1": "stem", "layer2": "layer1", "layer3": "layer2", "layer4": "layer3"}
    worst = {"elem": 0.0, "rel_l2": 0.0, "chan_mean": 0.0}
    r = QM.stem(x.double(), sd)
    e = QM.assert_stage_close(st["stem"], r, "stem")
    for li in range(1, 5):
        name = "layer%d" % li
        r = QM.stage(st[prev[name]].double(), sd, "resnet50_rmac", li)
        e = QM.assert_stage_close(st[name], r, name)
        for k in worst:
            worst[k] = max(worst[k], e[k])
    print("fp32 vs fp64 stage noise:", worst)
    assert worst["elem"] > 0 and worst["rel_l2"] > 0      # the two orders do differ: the check is not vacuous


def _tile_block_off(t):
    g = t.clone()
    g[0, 64:128, 8:16, 16:32] *= 1.1                       # one 64-channel block of one 8x16 tile, 10 % off
    return g


def _last_row_zeroed(t):
    g = t.clone()
    g[:, :, -1, :] = 0
    return g


def _tile_zeroed(t):
    g = t.clone()
    g[0, :, 8:16, 16:32] = 0
    return g


@pytest.mark.parametrize("layer", ["layer1", "layer2", "layer3"])
@pytest.mark.parametrize("defect", [_tile_block_off, _last_row_zeroed, _tile_zeroed], ids=["tile_block_10pct", "last_row_zero", "tile_zero"])
def test_comparator_fails_local_defects(r50_stages, layer, defect):
    _, _, st = r50_stages
    r = st[layer]
    g = defect(r)
    e = QM.stage_errors(g, r)
    assert QM.stage_failures(e), (layer, e)
    with pytest.raises(AssertionError):
        QM.assert_stage_close(g, r, layer)
    # it names where: the worst element and patch lie inside the damaged region
    n, y, x, c = e["worst"]
    if defect is _last_row_zeroed:
        assert y == r.shape[2] - 1 and e["worst_patch"][1] == (r.shape[2] - 1) // 8 * 8
    else:
        assert (n, y // 8, x // 16) == (0, 1, 1) and e["worst_patch"] == (0, 8, 16)
        if defect is _tile_block_off:
            assert 64 <= c < 128


def test_comparator_channel_mean_catches_a_small_shift(r50_stages):
    """A wrong shift in one channel (5e-3 * RMS everywhere) passes the per-element and rel-L2 bars but not the
    per-channel mean bar."""
    _, _, st = r50_stages
    r = st["layer2"]
    g = r.clone()
    rms = float(r.pow(2).mean().sqrt())
    g[:, 77] += 5e-3 * rms
    e = QM.stage_errors(g, r)
    assert QM.stage_failures(e) == ["chan_mean"] and e["worst_channel"] == 77, e
