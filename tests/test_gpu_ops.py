"""Parity of the CUDA operators (through the C ABI) against the CPU oracle.  Needs a B200: -m gpu."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import synthdata as synth
from oracle import dir_oracle as O
from conftest import rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _ops():
    from dirb200 import ops
    ops.require_gpu(0)
    return ops


def _conv_case(ops, B, H, W, Cin, Cout, k, stride, pad, use_res, relu, impl, seed=0):
    r = np.random.RandomState(seed)
    x = torch.from_numpy(r.standard_normal((B, H, W, Cin)).astype(np.float32)).half()
    w = torch.from_numpy((r.standard_normal((Cout, Cin, k, k)) * np.sqrt(2.0 / (Cin * k * k))).astype(np.float32))
    scale = torch.from_numpy(r.uniform(0.5, 1.5, Cout).astype(np.float32))
    shift = torch.from_numpy((0.2 * r.standard_normal(Cout)).astype(np.float32))
    Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    res = torch.from_numpy(r.standard_normal((B, Ho, Wo, Cout)).astype(np.float32)).half() if use_res else None
    # oracle: fp32 conv of the SAME fp16-rounded operands (resnet.py:56-63,70-85)
    y = F.conv2d(x.float().permute(0, 3, 1, 2), w.half().float(), None, stride=stride, padding=pad)
    y = y * scale.view(1, -1, 1, 1) + shift.view(1, -1, 1, 1)
    if use_res:
        y = y + res.float().permute(0, 3, 1, 2)
    if relu:
        y = F.relu(y)
    y = y.permute(0, 2, 3, 1).contiguous()
    wp = ops.pack_conv_weight(w).to(DEV)
    out = ops.conv_bn_act(x.to(DEV), wp, Cout, k, k, stride, pad, scale.to(DEV), shift.to(DEV),
                          res.to(DEV) if use_res else None, relu, impl)
    torch.cuda.synchronize()
    out = out.float().cpu()
    assert out.shape == y.shape
    err = (out - y).abs().max().item()
    tol = 2e-3 * max(1.0, y.abs().max().item())       # fp16 output rounding (2^-11 relative) + fp32 sum order
    return err, tol


CONV_CASES = [
    # B, H, W, Cin, Cout, k, stride, pad, res, relu
    (2, 16, 16, 64, 64, 1, 1, 0, False, True),
    (2, 14, 14, 256, 64, 1, 1, 0, False, True),      # M = 392: ragged last tile
    (1, 56, 56, 64, 256, 1, 1, 0, True, True),       # conv3 + residual
    (1, 16, 16, 64, 128, 3, 1, 1, False, True),
    (2, 14, 14, 128, 128, 3, 1, 1, False, True),     # patch 7x7-ish, zero padding at the borders
    (3, 7, 7, 512, 512, 3, 1, 1, False, True),       # several images per patch
    (2, 15, 17, 64, 64, 3, 2, 1, False, True),       # odd sizes, stride 2
    (2, 28, 28, 128, 128, 3, 2, 1, False, True),
    (2, 14, 14, 256, 512, 1, 2, 0, False, False),    # downsample branch (no ReLU)
    (1, 32, 32, 1024, 256, 1, 1, 0, False, True),    # long K
    (1, 64, 64, 256, 256, 3, 1, 1, False, True),     # layer3-like at 1024^2 input
    # more tiles than SMs: the persistent kernel wraps its accumulator / staging / ring state across tiles
    (8, 64, 64, 64, 256, 1, 1, 0, True, True),       # 256 tiles x 4 chunks, residual prefetch ring
    (6, 64, 64, 128, 128, 3, 1, 1, False, True),     # 192 tiles, 18 k-iterations each
    (3, 96, 96, 64, 64, 3, 1, 1, False, True),       # BN = 64
    (4, 64, 64, 512, 512, 1, 1, 0, True, True),      # 2 n-tiles per m-tile, residual
    (5, 30, 30, 256, 512, 1, 2, 0, False, False),    # stride-2 projection, ragged patches
    # 3x3/s1 through the halo kernel (8x16 patches, one input patch load per tile): ragged sizes, several
    # channel blocks, two n-tiles, resident and streamed weights
    (2, 33, 21, 64, 64, 3, 1, 1, False, True),
    (2, 17, 9, 128, 256, 3, 1, 1, False, True),
    (1, 40, 24, 512, 512, 3, 1, 1, False, False),
    (2, 32, 48, 64, 128, 3, 1, 1, False, True),
]


@pytest.mark.parametrize("impl", [0, 1, 2], ids=["tcgen05", "mma", "tcgen05np"])
@pytest.mark.parametrize("case", CONV_CASES, ids=lambda c: "x".join(str(v) for v in c[:8]))
def test_conv_bn_act(case, impl):
    err, tol = _conv_case(_ops(), *case, impl=impl)
    assert err <= tol, (err, tol)


EPI_KNOBS = [dict(epi_mode=0), dict(epi_mode=1), dict(epi_mode=2), dict(epi_mode=3),
             dict(epi_mode=3, l2_prefetch=1), dict(epi_mode=2, res_variant=1), dict(epi_mode=3, res_variant=2),
             dict(epi_mode=3, res_variant=3, l2_prefetch=8), dict(epi_mode=0, res_variant=3),
             dict(epi_warps=8), dict(epi_warps=16), dict(epi_warps=16, epi_mode=2), dict(epi_warps=8, epi_mode=1)]


@pytest.mark.parametrize("knobs", EPI_KNOBS, ids=lambda k: ",".join("%s=%d" % kv for kv in k.items()))
def test_conv_epilogue_and_tile_variants(knobs):
    """Every epilogue organisation (one / two warp groups, late / early release of the residual staging buffers), residual
    tile variant and the next-tile L2 prefetch compute the same convolution: the residual and many-tile cases of
    CONV_CASES vs the oracle, under each knob setting (process-wide selectors, restored afterwards)."""
    ops = _ops()
    cases = [c for c in CONV_CASES if c[8] or c[0] * c[1] * c[2] >= 128 * 148] + [(16, 64, 64, 256, 1024, 1, 1, 0, True, True)]
    saved = {k: ops.get_global_option(k) for k in ("epi_mode", "res_variant", "l2_prefetch", "epi_warps")}
    try:
        for k, v in knobs.items():
            ops.set_global_option(k, v)
        for case in cases:
            err, tol = _conv_case(ops, *case, impl=0)
            assert err <= tol, (case, err, tol)
    finally:
        for k, v in saved.items():
            ops.set_global_option(k, v)


def test_stem_and_maxpool():
    ops = _ops()
    x = synth.make_images(2, 64, 96, seed=3)
    sd = synth.make_state_dict("resnet50_rmac", seed=0)
    x8 = ops.nchw_to_nhwc8(x.to(DEV))
    torch.cuda.synchronize()
    ref8 = torch.zeros(2, 64, 96, 8)
    ref8[..., :3] = x.permute(0, 2, 3, 1)
    assert torch.equal(x8.cpu(), ref8.half())
    w = sd["conv1.weight"]
    s = sd["bn1.weight"] / torch.sqrt(sd["bn1.running_var"] + 1e-5)
    b = sd["bn1.bias"] - sd["bn1.running_mean"] * s
    wp = ops.pack_conv_weight(w, cin_pad=8).to(DEV)
    y = ops.conv_bn_act(x8, wp, 64, 7, 7, 2, 3, s.to(DEV), b.to(DEV), None, True, impl=1)
    yp = ops.maxpool_3x3s2(y)
    torch.cuda.synchronize()
    ref = F.relu(F.conv2d(x.half().float(), w.half().float(), None, stride=2, padding=3) * s.view(1, -1, 1, 1) + b.view(1, -1, 1, 1))
    assert (y.float().cpu() - ref.permute(0, 2, 3, 1)).abs().max().item() < 2e-3 * max(1.0, ref.abs().max().item())
    refp = F.max_pool2d(y.float().cpu().permute(0, 3, 1, 2), 3, 2, 1).permute(0, 2, 3, 1)
    assert torch.equal(yp.float().cpu(), refp)            # max of fp16 values is exact


@pytest.mark.parametrize("shape", [(2, 64, 96), (1, 63, 65), (3, 224, 224), (2, 130, 70)], ids=lambda s: "x".join(map(str, s)))
def test_stem_tcgen05(shape):
    """conv 7x7/s2/p3 + BN + ReLU through the space-to-depth tcgen05 kernel vs the fp32 oracle conv."""
    ops = _ops()
    b, h, w = shape
    x = synth.make_images(b, h, w, seed=4)
    sd = synth.make_state_dict("resnet50_rmac", seed=0)
    wgt = sd["conv1.weight"]
    s = sd["bn1.weight"] / torch.sqrt(sd["bn1.running_var"] + 1e-5)
    sh = sd["bn1.bias"] - sd["bn1.running_mean"] * s
    y = ops.stem_conv(x.to(DEV), wgt, s.to(DEV), sh.to(DEV))
    torch.cuda.synchronize()
    ref = F.relu(F.conv2d(x.half().float(), wgt.half().float(), None, stride=2, padding=3) * s.view(1, -1, 1, 1) + sh.view(1, -1, 1, 1))
    ref = ref.permute(0, 2, 3, 1)
    assert tuple(y.shape) == tuple(ref.shape)
    assert (y.float().cpu() - ref).abs().max().item() < 2e-3 * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("kw", [dict(pooling="gem", p=3.0), dict(pooling="gem", p=2.5), dict(pooling="max"),
                                dict(pooling="avg"), dict(pooling="gem", p=3.0, norm_features=True),
                                dict(pooling="gem", p=3.0, without_fc=True)],
                         ids=["gem3", "gem2.5", "max", "avg", "normfeat", "nofc"])
@pytest.mark.parametrize("shape", [(4, 7, 7), (1, 5, 9), (3, 32, 32)], ids=["4x7x7", "1x5x9", "3x32x32"])
def test_head(shape, kw):
    ops = _ops()
    b, h, w = shape
    r = np.random.RandomState(1)
    feat = torch.from_numpy(np.abs(r.standard_normal((b, h, w, 2048))).astype(np.float32)).half()
    feat[0, 0, 0, :7] = 0.0                                # exercises clamp(min=eps)
    sd = {"adpool.p": torch.tensor([kw.get("p", 3.0)]),
          "fc.weight": torch.from_numpy((r.standard_normal((2048, 2048)) / 45.0).astype(np.float32)),
          "fc.bias": torch.from_numpy((0.01 * r.standard_normal(2048)).astype(np.float32))}
    without_fc = kw.get("without_fc", False)
    ref = O.head(feat.float().permute(0, 3, 1, 2), sd, pooling=kw["pooling"], norm_features=kw.get("norm_features", False),
                 without_fc=without_fc, squeeze=False).numpy()
    out = ops.head_pool_fc_l2(feat.to(DEV), pooling=kw["pooling"], p=kw.get("p", 3.0), eps=1e-6,
                              norm_features=kw.get("norm_features", False),
                              fc_w=None if without_fc else sd["fc.weight"].to(DEV),
                              fc_b=None if without_fc else sd["fc.bias"].to(DEV))
    torch.cuda.synchronize()
    assert rel_l2(out.cpu().numpy(), ref) < 2e-5


@pytest.mark.parametrize("shape", [(1, 32, 32), (5, 7, 9), (19, 16, 12), (64, 8, 8)], ids=["1x32x32", "5x7x9", "19x16x12", "64x8x8"])
@pytest.mark.parametrize("kw", [dict(pooling="gem", p=3.0), dict(pooling="gem", p=2.5, norm_features=True),
                                dict(pooling="max", without_fc=True), dict(pooling="avg")],
                         ids=["gem3", "gem2.5-normfeat", "max-nofc", "avg"])
def test_head_single_kernel_is_bit_identical_to_the_phase_kernels(shape, kw):
    """rmac_resnet.py:59-68 as ONE persistent launch (grid barrier between pooling / FC / L2) vs one kernel per phase:
    the same virtual-block bodies in the same order, so fp32 and fp16 descriptors must agree bit for bit; repeated
    launches check that the self-resetting barrier words are reusable."""
    ops = _ops()
    b, h, w = shape
    r = np.random.RandomState(7)
    feat = torch.from_numpy(np.abs(r.standard_normal((b, h, w, 2048))).astype(np.float32)).half().to(DEV)
    without_fc = kw.get("without_fc", False)
    fc_w = None if without_fc else torch.from_numpy((r.standard_normal((2048, 2048)) / 45.0).astype(np.float32)).to(DEV)
    fc_b = None if without_fc else torch.from_numpy((0.01 * r.standard_normal(2048)).astype(np.float32)).to(DEV)
    args = dict(pooling=kw["pooling"], p=kw.get("p", 3.0), eps=1e-6, norm_features=kw.get("norm_features", False),
                fc_w=fc_w, fc_b=fc_b, want_f16=True)
    saved = ops.get_global_option("head_fused")
    try:
        ops.set_global_option("head_fused", 0)
        ref32, ref16 = ops.head_pool_fc_l2(feat, **args)
        ops.set_global_option("head_fused", 1)
        for _ in range(3):
            out32, out16 = ops.head_pool_fc_l2(feat, **args)
            torch.cuda.synchronize()
            assert torch.equal(out32, ref32) and torch.equal(out16, ref16)
    finally:
        ops.set_global_option("head_fused", saved)
    assert torch.isfinite(ref32).all() and abs(float(ref32[0].norm()) - 1.0) < 1e-5


def test_whiten_tensor_core_path_large():
    """5000 x 2048 rows through the tcgen05 hi/lo-split whitening vs the fp64 oracle, ragged row count."""
    ops = _ops()
    pca64 = synth.make_pca(2048, seed=3, dtype=np.float64)
    pca32 = synth.make_pca(2048, seed=3, dtype=np.float32)
    X = synth._unit_rows(np.random.RandomState(6).standard_normal((5000, 2048))).astype(np.float32)
    ref = O.whiten_features(X.astype(np.float64), pca64, whitenp=0.25, whitenv=1000)
    cs = (1.0 / np.power(pca64.explained_variance_[:1000], 0.25)).astype(np.float32)
    y = ops.whiten(torch.from_numpy(X).to(DEV), torch.from_numpy(pca32.components_[:1000].copy()).to(DEV),
                   torch.from_numpy(pca32.mean_).to(DEV), torch.from_numpy(cs).to(DEV))
    torch.cuda.synchronize()
    assert tuple(y.shape) == (5000, 1000)
    assert rel_l2(y.cpu().numpy(), ref) < 2e-5


@pytest.mark.parametrize("variant", [1, 0], ids=["pair", "single"])
@pytest.mark.parametrize("cm,b,h,w", [(256, 2, 64, 64), (128, 1, 48, 40), (256, 1, 17, 23), (128, 3, 16, 8), (256, 5, 72, 56), (64, 2, 80, 72), (64, 1, 16, 9)])
def test_conv_c23_fused_bottleneck_tail(cm, b, h, w, variant):
    """conv2 (3x3) + BN + ReLU + conv3 (1x1) + BN + residual + ReLU in ONE kernel (resnet.py:75-85) == the two-kernel
    path bit for bit (same fp16 rounding of the intermediate, same K order), and within fp16 tolerance of the oracle;
    ragged tiles (sizes that are not multiples of the 8 x 16 patch) and many tiles per CTA."""
    _conv_c23_case(_ops(), cm, b, h, w, variant, seed=cm + h)


def _conv_c23_case(ops, cm, b, h, w, variant, seed):
    r = np.random.RandomState(seed)
    t1 = torch.from_numpy(np.maximum(r.standard_normal((b, h, w, cm)), 0).astype(np.float16)).to(DEV)
    res = torch.from_numpy(r.standard_normal((b, h, w, 4 * cm)).astype(np.float16)).to(DEV)
    w2 = torch.from_numpy((r.standard_normal((cm, cm, 3, 3)) * np.sqrt(2.0 / (9 * cm))).astype(np.float32))
    w3 = torch.from_numpy((r.standard_normal((4 * cm, cm, 1, 1)) * np.sqrt(2.0 / cm)).astype(np.float32))
    s2 = torch.from_numpy(r.uniform(0.7, 1.3, cm).astype(np.float32)).to(DEV)
    h2 = torch.from_numpy((0.1 * r.standard_normal(cm)).astype(np.float32)).to(DEV)
    s3 = torch.from_numpy(r.uniform(0.2, 0.4, 4 * cm).astype(np.float32)).to(DEV)
    h3 = torch.from_numpy((0.1 * r.standard_normal(4 * cm)).astype(np.float32)).to(DEV)
    w2p, w3p = ops.pack_conv_weight(w2).to(DEV), ops.pack_conv_weight(w3).to(DEV)
    fused = ops.conv_c23(t1, w2p, s2, h2, w3p, s3, h3, res, variant=variant)
    t2 = ops.conv_bn_act(t1, w2p, cm, 3, 3, 1, 1, s2, h2, None, True)
    two = ops.conv_bn_act(t2, w3p, 4 * cm, 1, 1, 1, 0, s3, h3, res, True)
    torch.cuda.synchronize()
    assert torch.equal(fused, two)
    # oracle: fp32 convolutions on the fp16-rounded operands
    x = t1.float().cpu().permute(0, 3, 1, 2)
    mid = torch.relu(torch.nn.functional.conv2d(x, w2.half().float(), padding=1) * s2.cpu().view(1, -1, 1, 1) + h2.cpu().view(1, -1, 1, 1))
    out = torch.nn.functional.conv2d(mid.half().float(), w3.half().float()) * s3.cpu().view(1, -1, 1, 1) + h3.cpu().view(1, -1, 1, 1)
    out = torch.relu(out + res.float().cpu().permute(0, 3, 1, 2)).permute(0, 2, 3, 1)
    err = (fused.float().cpu() - out).abs().max().item()
    assert err < 2e-3 * max(1.0, out.abs().max().item()), err


@pytest.mark.parametrize("mag,spread", [(1.0, 1.0), (1.0, 0.1), (1.0, 0.01), (1.0, 1e-3), (1e-3, 1.0), (300.0, 0.05)])
def test_whiten_tensor_core_path_is_scale_invariant(mag, spread):
    """Rows tightly clustered around their mean and rows of unusual magnitude: the adaptive power-of-two prescale of
    the hi/lo split keeps the fp32-grade accuracy (without it the error grows like 1 / |x - mean|)."""
    ops = _ops()
    r = np.random.RandomState(11)
    centre = synth._unit_rows(r.standard_normal((1, 2048)))
    X = (mag * synth._unit_rows(centre + spread * r.standard_normal((1000, 2048)) / np.sqrt(2048.0))).astype(np.float32)
    mean = X.mean(0).astype(np.float32)
    comp = synth._unit_rows(r.standard_normal((256, 2048))).astype(np.float32)
    ref = (X.astype(np.float64) - mean.astype(np.float64)) @ comp.astype(np.float64).T
    y = ops.whiten(torch.from_numpy(X).to(DEV), torch.from_numpy(comp).to(DEV), torch.from_numpy(mean).to(DEV), None,
                   l2norm=False)
    torch.cuda.synchronize()
    err = np.linalg.norm(y.cpu().numpy().astype(np.float64) - ref, axis=1) / np.linalg.norm(ref, axis=1)
    print("whiten rel err (mag %g, spread %g): max %.3e" % (mag, spread, err.max()))
    assert err.max() < 2e-5, (mag, spread, err.max())        # bar: 2e-5 vs the fp64 oracle (DESIGN 4.4)


def test_pool_scales_l2_whiten(golden):
    ops = _ops()
    g = golden("pool.npz")
    xs = [torch.from_numpy(g[k]).to(DEV) for k in ("x0", "x1", "x2")]
    np.testing.assert_allclose(ops.pool_scales(xs, "mean", 3, l2=False).cpu().numpy(), g["mean"], rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(ops.pool_scales(xs, "gem", 3, l2=False).cpu().numpy(), g["gem3"], rtol=2e-5, atol=1e-6)
    np.testing.assert_allclose(ops.pool_scales(xs[:2], "gem", 2, l2=False).cpu().numpy(), g["gem2"], rtol=2e-5, atol=1e-6)
    np.testing.assert_array_equal(ops.pool_scales(xs[:1], "gem", 3, l2=False).cpu().numpy(), g["single"])
    with pytest.raises(ValueError):
        ops.pool_scales(xs, "bogus")
    pooled = ops.pool_scales(xs, "gem", 3, l2=True).cpu().numpy()
    assert rel_l2(pooled, O.l2n(g["gem3"])) < 1e-5
    # whitening against the golden (D=64) and against the oracle at D=2048
    w = golden("whiten.npz")
    X = torch.from_numpy(w["X"]).to(DEV)
    comp, mean, var = w["comp_f32"], w["mean_f32"], w["var_f32"]
    cs = (1.0 / (1.0 * np.power(var, 0.25))).astype(np.float32)
    y = ops.whiten(X, torch.from_numpy(comp).to(DEV), torch.from_numpy(mean).to(DEV), torch.from_numpy(cs).to(DEV))
    assert rel_l2(y.cpu().numpy(), w["w_p025_f64"]) < 1e-5
    cs2 = (1.0 / (2.0 * np.power(var[:32], 0.5))).astype(np.float32)
    y2 = ops.whiten(X, torch.from_numpy(comp[:32].copy()).to(DEV), torch.from_numpy(mean).to(DEV), torch.from_numpy(cs2).to(DEV))
    assert rel_l2(y2.cpu().numpy(), w["w_p05_v32_m2_f64"]) < 1e-5
    y3 = ops.whiten(X, torch.from_numpy(comp).to(DEV), torch.from_numpy(mean).to(DEV), torch.from_numpy(cs).to(DEV), l2norm=False)
    assert rel_l2(y3.cpu().numpy(), w["w_nol2_f64"]) < 1e-5
    pca = synth.make_pca(2048, seed=11, dtype=np.float32)
    Xb = synth._unit_rows(np.random.RandomState(5).standard_normal((300, 2048))).astype(np.float32)
    ref = O.whiten_features(Xb.astype(np.float64), synth.make_pca(2048, seed=11, dtype=np.float64), whitenp=0.25)
    csb = (1.0 / np.power(pca.explained_variance_.astype(np.float64), 0.25)).astype(np.float32)
    yb, yb16 = ops.whiten(torch.from_numpy(Xb).to(DEV), torch.from_numpy(pca.components_).to(DEV),
                          torch.from_numpy(pca.mean_).to(DEV), torch.from_numpy(csb).to(DEV), want_f16=True)
    assert rel_l2(yb.cpu().numpy(), ref) < 1e-3            # north-star tolerance; the hi/lo split GEMM gives ~1e-6
    assert rel_l2(yb.cpu().numpy(), ref) < 2e-5
    assert rel_l2(yb16.float().cpu().numpy(), ref) < 1e-3


@pytest.mark.parametrize("shape", [(2, 37, 53, 0.7), (1, 100, 80, 1.4), (3, 64, 64, 0.5), (1, 333, 517, 0.7), (2, 224, 224, 1.4)],
                         ids=lambda s: "x".join(str(v) for v in s))
def test_resize_bilinear_matches_pil(shape):
    """GPU bilinear resize == PIL Image.resize(BILINEAR) byte for byte (the `Scale(float)` transform, transforms.py:168,183)."""
    from PIL import Image
    ops = _ops()
    b, h, w, s = shape
    ho, wo = int(0.5 + s * h), int(0.5 + s * w)
    a = np.random.RandomState(1).randint(0, 256, (b, h, w, 3), dtype=np.uint8)
    out = ops.resize_bilinear_u8(torch.from_numpy(a).to(DEV), (ho, wo)).cpu().numpy()
    for i in range(b):
        ref = np.array(Image.fromarray(a[i]).resize((wo, ho), Image.BILINEAR))
        assert np.array_equal(out[i], ref)
