"""CPU simulation of the NUMERICS of the GPU extraction path (TEST INFRASTRUCTURE): the same network as
oracle/dir_oracle.py, with every rounding the kernels perform - fp16 input, fp16 weights, fp32 accumulation, BatchNorm as
an fp32 (scale, shift) epilogue, fp16 activation stores, BN-scaled fp16 weights for the fused projection shortcut, fp32
head.  It answers "does this precision design meet the 1e-3 descriptor bar, and with what margin" without a GPU
(DESIGN.md section 2); accumulation ORDER inside a dot product is the only thing it does not reproduce.

The network is split into the stages the GPU path records as debug taps (stem, layer1..layer4, the FPN lateral
'fpn_c4'): each stage function takes a stage input holding fp16 values (NCHW; fp32, or fp64 to accumulate in double
precision) and returns the stage output the kernels would store, so a GPU stage can be checked on its own, fed with the
GPU's own previous tap.  stage_errors() / assert_stage_close() compare a GPU stage with the model and locate a defect."""
import torch
import torch.nn.functional as F

from oracle import dir_oracle as O


def h(x):
    """Round to fp16 and come back (what a store to an fp16 tensor + reload does)."""
    return x.to(torch.float16).to(x.dtype if x.dtype != torch.float16 else torch.float32)


def _fold(sd, name):
    s = sd[name + ".weight"] / torch.sqrt(sd[name + ".running_var"] + O.BN_EPS)       # net.cu: pack_conv
    return s, sd[name + ".bias"] - sd[name + ".running_mean"] * s


def _conv(x16, w, scale, shift, stride=1, padding=0, res16=None, relu=True):
    y = F.conv2d(x16, h(w).to(x16.dtype), None, stride=stride, padding=padding)     # fp16 operands, fp32 accumulate
    y = y * scale.view(1, -1, 1, 1) + shift.view(1, -1, 1, 1)                        # epilogue in fp32
    if res16 is not None:
        y = y + res16
    return h(F.relu(y) if relu else y)


def _trunk(arch):
    name = arch.split("_")[0]
    if name in O.BASIC_BLOCKS:
        return O.BASIC_BLOCKS[name], True
    return O.BLOCKS[name], False


def nchw(tap):
    """NHWC fp16 GPU tap -> NCHW fp32 stage input / output of this model."""
    return tap.float().permute(0, 3, 1, 2).contiguous()


@torch.no_grad()
def stem(x, sd):
    """conv 7x7/s2/p3 -> BN -> ReLU on the fp16-rounded image, fp16 store, maxpool 3x3/s2/p1 (exact on fp16 values)."""
    s, b = _fold(sd, "bn1")
    t = _conv(h(x), sd["conv1.weight"], s, b, stride=2, padding=3)
    return F.max_pool2d(t, kernel_size=3, stride=2, padding=1)


@torch.no_grad()
def stage(t, sd, arch, layer, fuse_shortcut=True):
    """layer1..layer4 (`layer` = 1..4) of a Bottleneck or BasicBlock trunk.  fuse_shortcut: block 0 of a Bottleneck
    layer runs conv3 + projection shortcut as one GEMM over K = [conv2 output | block input] with BN-scaled fp16 weights
    (net.cu: wcat; the tcgen05 path with option fuse_ds), else two convolutions with an fp16 shortcut in between."""
    blocks, basic = _trunk(arch)
    t = h(t)
    for bi in range(blocks[layer - 1]):
        p = "layer%d.%d." % (layer, bi)
        stride = 2 if (layer > 1 and bi == 0) else 1
        if basic:                                          # resnet.py:27-44, net.cu: run_chunk (n->basic)
            s1, b1 = _fold(sd, p + "bn1")
            s2, b2 = _fold(sd, p + "bn2")
            t1 = _conv(t, sd[p + "conv1.weight"], s1, b1, stride=stride, padding=1)
            res = t
            if bi == 0 and layer > 1:                      # resnet.py:136-141 (expansion 1)
                sdn, bdn = _fold(sd, p + "downsample.1")
                res = _conv(t, sd[p + "downsample.0.weight"], sdn, bdn, stride=stride, relu=False)
            t = _conv(t1, sd[p + "conv2.weight"], s2, b2, padding=1, res16=res)
            continue
        s1, b1 = _fold(sd, p + "bn1")
        s2, b2 = _fold(sd, p + "bn2")
        s3, b3 = _fold(sd, p + "bn3")
        t1 = _conv(t, sd[p + "conv1.weight"], s1, b1)
        t2 = _conv(t1, sd[p + "conv2.weight"], s2, b2, stride=stride, padding=1)
        if bi == 0:
            sdn, bdn = _fold(sd, p + "downsample.1")
            if fuse_shortcut:      # one GEMM over K = [t2 | x] with BN-scaled fp16 weights (net.cu: wcat)
                y = F.conv2d(t2, h(sd[p + "conv3.weight"] * s3.view(-1, 1, 1, 1)).to(t.dtype)) + \
                    F.conv2d(t, h(sd[p + "downsample.0.weight"] * sdn.view(-1, 1, 1, 1)).to(t.dtype), stride=stride)
                t = h(F.relu(y + (b3 + bdn).view(1, -1, 1, 1)))
            else:
                r = _conv(t, sd[p + "downsample.0.weight"], sdn, bdn, stride=stride, relu=False)
                t = _conv(t2, sd[p + "conv3.weight"], s3, b3, res16=r)
        else:
            t = _conv(t2, sd[p + "conv3.weight"], s3, b3, res16=t)
    return t


@torch.no_grad()
def fpn_c4(layer3, layer4, sd):
    """FPN lateral of mode 1 (rmac_resnet_fpn.py:55-62) as the GPU runs it: h(relu(conv1x5(x5))) on the small map (the
    1x1 convolution commutes with the nearest upsampling), nearest upsample to the layer3 size, h(x4 + up), then
    h(relu(conv3c4(.))).  No BatchNorm: scale 1, shift 0."""
    x4, x5 = h(layer3), h(layer4)
    c3 = x4.shape[1]
    one, zero = torch.ones(c3, dtype=x4.dtype), torch.zeros(c3, dtype=x4.dtype)
    t = _conv(x5, sd["conv1x5.weight"], one, zero)
    up = F.interpolate(t, size=x4.shape[-2:], mode="nearest")
    return _conv(h(x4 + up), sd["conv3c4.weight"], one, zero, padding=1)


@torch.no_grad()
def stages(x, sd, arch="resnet50_rmac", fuse_shortcut=True):
    """{'stem', 'layer1'..'layer4'} of the model run end to end."""
    out = {"stem": stem(x, sd)}
    t = out["stem"]
    for li in range(1, 5):
        t = out["layer%d" % li] = stage(t, sd, arch, li, fuse_shortcut)
    return out


@torch.no_grad()
def extract(x, sd, arch="resnet50_rmac", fuse_shortcut=True, **head_kw):
    return O.head(stages(x, sd, arch, fuse_shortcut)["layer4"], sd, **head_kw)   # fp32 head on the fp16 map


# --------------------------------------------------------------------------- stage comparator
# Bars for a GPU stage against this model fed with the GPU's own previous stage (tests/test_gpu_extract_stages.py).
# The model differs from the kernels only in the order of the fp32 sums; a different order flips the fp16 rounding of
# some stored intermediates, and inside a stage such flips propagate through the following blocks.  The CPU estimate of
# that noise (the same stage accumulated in fp32 and in fp64; R50 at 200x328 and R101 at 256^2) is 5-8e-3 * RMS per
# element, 2-6e-4 stage rel L2 and 2.5e-4 * RMS per channel mean; the bars below are 4-8x that.  The GPU stage tests print
# their statistics (STAGE_ERR lines); keep each bar at 3x or more above the worst value they report on a B200.
ELEM_BAR = 3e-2         # max |g - r| / RMS(r)
REL_L2_BAR = 3e-3       # ||g - r|| / ||r||
CHAN_MEAN_BAR = 2e-3    # max over channels of |mean over pixels of (g - r)| / RMS(r)
PATCH = (8, 16)         # rows x columns of the convolution kernels' output patch


def stage_errors(g, r):
    """g, r: NCHW stage tensors (GPU, model).  -> dict of the three statistics, the worst element (n, y, x, c) and the
    worst 8x16 patch (n, y0, x0) by summed squared error."""
    g = g.double()
    r = r.double()
    d = g - r
    rms = float(r.pow(2).mean().sqrt().clamp(min=1e-30))
    a = d.abs()
    i = int(a.argmax())
    n, c, y, x = [int(v) for v in torch.unravel_index(torch.tensor(i), a.shape)]
    chan = d.mean(dim=(0, 2, 3)).abs()
    e2 = F.pad(d.pow(2).sum(1, keepdim=True), (0, (-d.shape[3]) % PATCH[1], 0, (-d.shape[2]) % PATCH[0]))
    pe = F.avg_pool2d(e2, PATCH, stride=PATCH)[:, 0]
    j = int(pe.argmax())
    pn, py, px = [int(v) for v in torch.unravel_index(torch.tensor(j), pe.shape)]
    return dict(elem=float(a.max()) / rms, rel_l2=float(d.norm() / r.norm().clamp(min=1e-30)),
                chan_mean=float(chan.max()) / rms, rms=rms, worst=(n, y, x, c), worst_channel=int(chan.argmax()),
                worst_patch=(pn, py * PATCH[0], px * PATCH[1]))


def stage_failures(e, elem=ELEM_BAR, rel_l2=REL_L2_BAR, chan_mean=CHAN_MEAN_BAR):
    """Names of the statistics of stage_errors() result `e` that exceed their bars."""
    return [k for k, bar in (("elem", elem), ("rel_l2", rel_l2), ("chan_mean", chan_mean)) if e[k] > bar]


def assert_stage_close(g, r, what, **bars):
    e = stage_errors(g, r)
    bad = stage_failures(e, **bars)
    assert not bad, ("%s: %s over the bar; elem %.3e rel_l2 %.3e chan_mean %.3e (channel %d); worst element (n,y,x,c) = %s, "
                     "worst 8x16 patch (n,y0,x0) = %s" % (what, bad, e["elem"], e["rel_l2"], e["chan_mean"],
                                                           e["worst_channel"], e["worst"], e["worst_patch"]))
    return e
