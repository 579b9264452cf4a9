"""The extraction network stage by stage, element for element, and at the benchmark's batch through the host entry points.
-m gpu.

A descriptor averages a local defect away (a wrong K-chunk in one 8x16 tile of layer1 moves it by ~2e-4, inside the
1e-3 descriptor bar), so here every stage output the network records (option debug_taps) is checked on its own: the GPU's
previous tap goes through the per-stage numerics model (tests/quant_model.py) and the result is compared with the next
tap by three statistics - per element, rel L2 and per-channel mean (quant_model.stage_errors) - that name the worst
element and 8x16 patch on failure.  Stages are isolated, so errors do not carry over from earlier stages.

Then the benchmark geometry (ResNet-101, 64 x 1024^2, one chunk of 64: activation tensors of 2^31 bytes), the pipelined
host entry points over several chunks, and the single operators the network tests reached only through descriptors."""
import contextlib
import ctypes as C
import gc
import json

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import quant_model as QM
import synthdata as synth
from oracle import dir_oracle as O
from conftest import rel_l2
from test_gpu_ops import CONV_CASES, EPI_KNOBS, _conv_case, _conv_c23_case

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
STAGES = ("stem", "layer1", "layer2", "layer3", "layer4")

# (id, net options, process-wide kernel selectors).  One line per knob setting: retiring a knob removes its line.
CONFIGS = [
    ("default", {}, {}),
    ("conv_impl1", dict(conv_impl=1), {}),
    ("conv_impl2", dict(conv_impl=2), {}),
    ("fuse_ds0", dict(fuse_ds=0), {}),
    ("fuse_c23_pair", dict(fuse_c23=2, c23_variant=1), {}),
    ("fuse_c23_single", dict(fuse_c23=2, c23_variant=0), {}),
    ("halo0", {}, dict(halo=0)),
    ("epi_warps8", {}, dict(epi_warps=8)),
    ("epi_mode3", {}, dict(epi_mode=3)),
    ("res_variant1", {}, dict(res_variant=1)),
    ("stage_sched_sub1", dict(stage_sched=1, sub1=1, sub2=1, sub3=1, sub4=1), {}),
]
# G1: maps 50x82 -> 25x41 -> 13x21 -> 7x11 (odd input at every stride-2 step; layers 3-4 below the halo kernel's
# H >= 16; several images per tile).  G2: maps 130x98 -> 65x49 -> 33x25 -> 17x13 (ragged 8x16 patches everywhere).
GEOMS = {"G1": (3, 200, 328), "G2": (2, 520, 392)}


@contextlib.contextmanager
def _global_options(opts):
    from dirb200 import ops
    saved = {k: ops.get_global_option(k) for k in opts}
    try:
        for k, v in opts.items():
            ops.set_global_option(k, v)
        yield
    finally:
        for k, v in saved.items():
            ops.set_global_option(k, v)


def _net(arch, seed, **kw):
    from dirb200 import nets, ops
    ops.require_gpu(0)
    net = nets.create_model(arch, **kw)
    sd = synth.make_state_dict(arch, seed=seed, out_dim=net.out_dim)
    net.load_state_dict(sd)
    return net.eval(), sd


def _taps(net, names=STAGES):
    torch.cuda.synchronize()
    return {s: QM.nchw(net.debug_stage(s).cpu()) for s in names}


def _check(tag, stage, g, r):
    """Stage statistics as one parseable line (collected for DESIGN.md section 2), and the bars."""
    e = QM.stage_errors(g, r)
    print("STAGE_ERR " + json.dumps(dict(tag=tag, stage=stage, elem=e["elem"], rel_l2=e["rel_l2"], chan_mean=e["chan_mean"])))
    return e, QM.stage_failures(e)


def _check_stages(tag, net, sd, arch, x, fuse_shortcut):
    """Run x with debug taps; every stage from the previous GPU tap through the model, against the next tap."""
    net.set_backend_option_live("debug_taps", 1)
    net(x.to(DEV))
    taps = _taps(net)
    bad = []
    g = taps["stem"]
    e, f = _check(tag, "stem", g, QM.stem(x[-g.shape[0]:], sd))
    bad += [("stem", f, e)] if f else []
    for li in range(1, 5):
        name, prev = STAGES[li], STAGES[li - 1]
        g = taps[name]                     # with per-stage sub-chunks, layer4 holds the last sub-chunk only
        e, f = _check(tag, name, g, QM.stage(taps[prev][-g.shape[0]:], sd, arch, li, fuse_shortcut))
        bad += [(name, f, e)] if f else []
    assert not bad, (tag, bad)
    return taps


@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
@pytest.mark.parametrize("geom", sorted(GEOMS))
def test_r50_stages_match_the_model(geom, cfg):
    name, opts, gopts = cfg
    net, sd = _net("resnet50_rmac", 11)
    for k, v in opts.items():
        net.set_backend_option(k, v)
    x = synth.make_images(*GEOMS[geom], seed=12)
    fused = opts.get("fuse_ds", 1) != 0 and opts.get("conv_impl", 0) == 0
    with _global_options(gopts):
        _check_stages("r50/%s/%s" % (geom, name), net, sd, "resnet50_rmac", x, fused)


@pytest.mark.parametrize("cfg", [c for c in CONFIGS if not any(k.startswith(("fuse", "c23")) for k in c[1])],
                         ids=lambda c: c[0])
def test_r18_basic_block_stages_match_the_model(cfg):
    """BasicBlock trunk: 3x3 + residual through the halo kernel at widths 64, 128, 256 and 512 (G2)."""
    name, opts, gopts = cfg
    net, sd = _net("resnet18_rmac", 13)
    for k, v in opts.items():
        net.set_backend_option(k, v)
    with _global_options(gopts):
        _check_stages("r18/G2/" + name, net, sd, "resnet18_rmac", synth.make_images(*GEOMS["G2"], seed=14), True)


def test_fpn_lateral_stage_matches_the_model():
    """R50-FPN mode 1 at G1: 1x1 lateral on the 7x11 layer4 map, nearest upsample to 13x21, add, 3x3 smoothing."""
    net, sd = _net("resnet50_fpn_rmac", 15)
    taps = _check_stages("r50fpn/G1/default", net, sd, "resnet50_fpn_rmac", synth.make_images(*GEOMS["G1"], seed=16), True)
    g = _taps(net, ("fpn_c4",))["fpn_c4"]
    e, f = _check("r50fpn/G1/default", "fpn_c4", g, QM.fpn_c4(taps["layer3"][-g.shape[0]:], taps["layer4"][-g.shape[0]:], sd))
    assert not f, e


def test_r101_1024_stages_match_the_model():
    net, sd = _net("resnet101_rmac", 17)
    _check_stages("r101/1x1024/default", net, sd, "resnet101_rmac", synth.make_images(1, 1024, 1024, seed=18), True)


def test_taps_do_not_depend_on_the_chunk():
    """chunk = 1 records the last image alone: its taps equal the last image's taps of one chunk of B, bit for bit."""
    net, _ = _net("resnet50_rmac", 11)
    x = synth.make_images(*GEOMS["G1"], seed=12).to(DEV)
    net.set_backend_option("debug_taps", 1)
    d = net(x)
    whole = {s: net.debug_stage(s) for s in STAGES}
    net.set_backend_option_live("chunk", 1)
    assert torch.equal(net(x), d)
    for s in STAGES:
        one = net.debug_stage(s)
        assert one.shape[0] == 1 and torch.equal(one, whole[s][-1:]), s


def test_debug_stage_reports_the_size_when_the_buffer_is_too_small():
    from dirb200 import lib
    net, _ = _net("resnet50_rmac", 11)
    net.set_backend_option("debug_taps", 1)
    net(synth.make_images(2, 64, 96, seed=1).to(DEV))
    dims = (C.c_int * 4)()
    buf = torch.empty(1024, dtype=torch.uint8, device=DEV)
    with pytest.raises(lib.DirbError):
        lib.call("dirb200_net_debug_stage", net._handle, b"layer1", C.c_void_p(buf.data_ptr()), buf.numel(), dims,
                 C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert list(dims) == [2, 16, 24, 256]
    assert tuple(net.debug_stage("layer1").shape) == (2, 16, 24, 256)


# --------------------------------------------------------------------------- benchmark geometry
BENCH_B, BENCH_HW = 64, 1024
# device bytes this test needs: ~13 GB of activation workspace for a chunk of 64 (net.cu: setup_workspace), 4.6 GB of
# taps, 0.8 GB of input, the host staging buffers and tap copies, with margin; the peak is printed as BENCH_MEM_USED
BENCH_MEM = 40e9


def test_benchmark_geometry_and_host_entry_points():
    """ResNet-101, 64 x 1024^2, auto chunk (one chunk of 64; a layer1 activation is 64*256*256*256*2 B = 2^31 B):
    descriptors against the oracle, the image-63 stages against the model, batch invariance, and the pipelined host
    entry points (chunks 8, 8, 16, 32 / 1, 1, 2, 4, 6, ... / uniform 5 with a ragged tail; buffer and event reuse over
    B = 64 -> 5 -> 64; pageable memory) bit-identical to the device entry points."""
    gc.collect()
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if free < BENCH_MEM:
        print("skipped: %.1f GB free on the device, the 64 x 1024^2 geometry needs %.0f GB" % (free / 1e9, BENCH_MEM / 1e9))
        pytest.skip("needs %.0f GB of free device memory" % (BENCH_MEM / 1e9))
    net, sd = _net("resnet101_rmac", 19)
    u8 = synth.make_images_u8(BENCH_B, BENCH_HW, BENCH_HW, seed=20)
    x = synth.normalise_images(u8)
    net.set_backend_option("debug_taps", 1)
    d = net(x.to(DEV))
    taps = {s: net.debug_stage(s)[63:64].cpu() for s in STAGES}
    torch.cuda.synchronize()
    free_min, _ = torch.cuda.mem_get_info()
    print("BENCH_MEM_USED %.2f GB" % ((free - free_min) / 1e9))
    ref = d.cpu().numpy()
    # against the oracle
    sel = [0, 37, 63]
    assert rel_l2(ref[sel], O.extract(x[sel], sd, "resnet101_rmac", squeeze=False).numpy()) < 1e-3
    # the stages of the last image of the 64-image taps against the model
    t = {s: QM.nchw(v) for s, v in taps.items()}
    bad = []
    e, f = _check("r101/64x1024/img63", "stem", t["stem"], QM.stem(x[63:64], sd))
    bad += [("stem", f, e)] if f else []
    for li in range(1, 5):
        e, f = _check("r101/64x1024/img63", STAGES[li], t[STAGES[li]], QM.stage(t[STAGES[li - 1]], sd, "resnet101_rmac", li))
        bad += [(STAGES[li], f, e)] if f else []
    assert not bad, bad
    # batch invariance: image 63 alone
    d63 = net(x[63:64].to(DEV))
    assert torch.equal(d63, d[63])
    for s in STAGES:
        assert torch.equal(net.debug_stage(s).cpu(), taps[s]), s
    net.set_backend_option_live("debug_taps", 0)
    # host entry points == device entry points, bit for bit
    pinned = torch.empty(x.shape, dtype=torch.float32).pin_memory()
    pinned.copy_(x)
    xp = pinned.numpy()
    pinned8 = torch.empty(u8.shape, dtype=torch.uint8).pin_memory()
    pinned8.copy_(torch.from_numpy(u8))
    up = pinned8.numpy()
    d8 = net.forward_u8(torch.from_numpy(u8).to(DEV)).cpu().numpy()
    assert np.array_equal(d8, ref)                                      # uint8 input == fp32 input
    for label, opts in (("host_chunk 16", {}), ("host_chunk 3", dict(host_chunk=3)), ("chunk 5", dict(chunk=5))):
        for k, v in opts.items():
            net.set_backend_option_live(k, v)
        try:
            assert np.array_equal(net.forward_host(xp), ref), label
            assert np.array_equal(net.forward_host_u8(up), d8), label
        finally:
            net.set_backend_option_live("host_chunk", 16)
            net.set_backend_option_live("chunk", 0)
    for b in (BENCH_B, 5, BENCH_B):                                      # buffer / event reuse across calls
        assert np.array_equal(net.forward_host(xp[:b]), ref[:b]), b
        assert np.array_equal(net.forward_host_u8(up[:b]), d8[:b]), b
    assert np.array_equal(net.forward_host(x.numpy()), ref)             # pageable memory
    assert np.array_equal(net.forward_host_u8(u8), d8)


# --------------------------------------------------------------------------- single operators
# 3x3 / stride 1 convolution + residual (BasicBlock conv2: the halo kernel's residual producer): Cin = Cout at every
# BasicBlock width, ragged sizes, one map below the halo kernel's H >= 16
RES3_CASES = [
    (2, 33, 21, 64, 64, 3, 1, 1, True, True),
    (2, 17, 29, 128, 128, 3, 1, 1, True, True),
    (1, 19, 24, 256, 256, 3, 1, 1, True, True),
    (2, 20, 13, 512, 512, 3, 1, 1, True, True),
    (3, 9, 12, 128, 128, 3, 1, 1, True, True),
]


def _ops():
    from dirb200 import ops
    ops.require_gpu(0)
    return ops


@pytest.mark.parametrize("halo", [1, 0])
@pytest.mark.parametrize("impl", [0, 1, 2], ids=["tcgen05", "mma", "tcgen05np"])
@pytest.mark.parametrize("case", RES3_CASES, ids=lambda c: "x".join(str(v) for v in c[:5]))
def test_conv3x3_with_residual(case, impl, halo):
    ops = _ops()
    with _global_options(dict(halo=halo)):
        err, tol = _conv_case(ops, *case, impl=impl)
    assert err <= tol, (err, tol)


@pytest.mark.parametrize("knobs", EPI_KNOBS, ids=lambda k: ",".join("%s=%d" % kv for kv in k.items()))
def test_conv3x3_with_residual_epilogue_variants(knobs):
    ops = _ops()
    with _global_options(knobs):
        for case in RES3_CASES:
            err, tol = _conv_case(ops, *case, impl=0)
            assert err <= tol, (case, err, tol)


@pytest.mark.parametrize("impl", [0, 2], ids=["tcgen05", "tcgen05np"])
@pytest.mark.parametrize("case", [c for c in CONV_CASES if c[5] == 3 and c[6] == 1], ids=lambda c: "x".join(str(v) for v in c[:8]))
def test_conv3x3_tap_by_tap_path(case, impl):
    """halo = 0: the 3x3 stride-1 convolutions take the tap-by-tap path at every size."""
    ops = _ops()
    with _global_options(dict(halo=0)):
        err, tol = _conv_case(ops, *case, impl=impl)
    assert err <= tol, (err, tol)


@pytest.mark.parametrize("epi_mode", [0, 1, 2, 3])
@pytest.mark.parametrize("cm,b,h,w", [(64, 2, 80, 72), (128, 3, 16, 8), (256, 1, 17, 23)])
def test_conv_c23_under_epi_mode(cm, b, h, w, epi_mode):
    """The fused Bottleneck tail reads the epilogue organisation too: under each setting it equals the two-kernel path
    bit for bit and meets the oracle bound."""
    ops = _ops()
    with _global_options(dict(epi_mode=epi_mode)):
        for variant in (1, 0):
            _conv_c23_case(ops, cm, b, h, w, variant, seed=cm + h + epi_mode)


def test_center_bias():
    """x * (1 + center-bias map) at every small map size: the kernel computes the bilinear weights itself, in fp32."""
    ops = _ops()
    sizes = (1, 2, 3, 7, 13, 32)
    r = np.random.RandomState(3)
    inexact = total = 0
    for b in (0.5, 2.0):
        for hh in sizes:
            for ww in sizes:
                x = torch.from_numpy(np.abs(r.standard_normal((2, hh, ww, 16))).astype(np.float16))
                m = O.center_bias_map(b, hh, ww)[0, 0]                                  # (hh, ww) fp32
                ref = (x.float() * m.view(1, hh, ww, 1)).half()
                out = ops.center_bias(x.to(DEV), b).cpu()
                ulp = (out.view(torch.int16).int() - ref.view(torch.int16).int()).abs()
                assert int(ulp.max()) <= 1, (b, hh, ww)
                inexact += int((ulp > 0).sum())
                total += ulp.numel()
    print("center_bias: %d of %d elements 1 fp16 ulp off h(x * map), the rest exact" % (inexact, total))


@pytest.mark.parametrize("hh", [1, 2, 3, 17])
@pytest.mark.parametrize("ww", [1, 2, 3, 17])
def test_maxpool_with_negative_inputs(hh, ww):
    """Windows at the border and windows whose values are all negative: the maximum, never the padding."""
    ops = _ops()
    r = np.random.RandomState(hh * 31 + ww)
    x = r.standard_normal((2, hh, ww, 64))
    x[0] = -np.abs(x[0]) - 0.5                                           # image 0: every value negative
    x[1, ..., :32] -= 1000.0                                             # large negative channels
    xh = torch.from_numpy(x.astype(np.float16))
    out = ops.maxpool_3x3s2(xh.to(DEV)).cpu()
    ref = F.max_pool2d(xh.float().permute(0, 3, 1, 2), 3, 2, 1).permute(0, 2, 3, 1)
    assert torch.equal(out.float(), ref)
