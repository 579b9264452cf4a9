"""Model API of the extraction path: the duck-type the reference's callers use, backed by libdirb200.

Mirrors ``dirtorch/nets/__init__.py:18-95`` (``model_names``, ``create_model``, ``load_pretrained_weights``)
and the module surface of ``dirtorch/nets/rmac_resnet.py:12-69`` that ``test_dir.py:57-74,185-190`` and
``common.py:150-175`` touch: ``net(imgs) -> (B,D)`` L2-normalised descriptors (``(D,)`` at B=1),
``preprocess``, ``rgb_means/rgb_stds/input_size``, ``iscuda``, ``pca``, ``fc_name``, ``feat_dim``,
``eval()``, ``state_dict()``, ``load_state_dict()``.

The forward pass is NOT torch: the state dict is handed to the C library, which folds BatchNorm, repacks the
convolutions for the tcgen05 implicit-GEMM kernels and runs the whole network on the current CUDA stream.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from collections import OrderedDict

import numpy as np
import torch

from . import lib

RGB_MEANS = [0.485, 0.456, 0.406]            # resnet.py:110-111
RGB_STDS = [0.229, 0.224, 0.225]

_TRUNKS = {"resnet18": ([2, 2, 2, 2], 1), "resnet50": ([3, 4, 6, 3], 4), "resnet101": ([3, 4, 23, 3], 4),
           "resnet152": ([3, 8, 36, 3], 4)}                       # (blocks per layer, block.expansion): resnet.py:15,47
# rmac_resnet.py:74-88 and rmac_resnet_fpn.py:92-110 (the trunk-only classifiers resnet18/50/101/152 of
# nets/__init__.py:14 are ImageNet classifiers, not descriptor networks: not on this path)
_ARCH = {t + "_rmac": (t, False, 1) for t in _TRUNKS}
_ARCH.update({t + "_fpn_rmac": (t, True, 1) for t in _TRUNKS})
_ARCH["resnet101_fpn0_rmac"] = ("resnet101", True, 0)
_ARCH_BLOCKS = {a: _TRUNKS[t][0] for a, (t, _f, _m) in _ARCH.items()}
model_names = set(_ARCH)


def _reference_style_init(arch, out_dim, seed_gen=None, fpn_mode=1):
    """Fresh weights with the statistics of the reference's constructor: conv ~ N(0, sqrt(2/(k*k*Cout)))
    and BN weight 1 / bias 0 (resnet.py:92-99), identity running stats, Linear default init."""
    g = seed_gen or torch.Generator().manual_seed(torch.initial_seed() & 0x7FFFFFFF)
    sd = OrderedDict()
    trunk, fpn, _ = _ARCH[arch]
    blocks, exp = _TRUNKS[trunk]

    def conv(name, cout, cin, k):
        sd[name] = torch.randn((cout, cin, k, k), generator=g) * math.sqrt(2.0 / (k * k * cout))

    def bn(name, c):
        sd[name + ".weight"] = torch.ones(c)
        sd[name + ".bias"] = torch.zeros(c)
        sd[name + ".running_mean"] = torch.zeros(c)
        sd[name + ".running_var"] = torch.ones(c)
        sd[name + ".num_batches_tracked"] = torch.tensor(0, dtype=torch.long)

    conv("conv1.weight", 64, 3, 7)
    bn("bn1", 64)
    inplanes = 64
    for li, (planes, nblk) in enumerate(zip([64, 128, 256, 512], blocks), start=1):
        for b in range(nblk):
            p = "layer%d.%d." % (li, b)
            stride = 2 if (li > 1 and b == 0) else 1
            if exp == 4:                                          # Bottleneck, resnet.py:54-65
                conv(p + "conv1.weight", planes, inplanes, 1)
                bn(p + "bn1", planes)
                conv(p + "conv2.weight", planes, planes, 3)
                bn(p + "bn2", planes)
                conv(p + "conv3.weight", planes * 4, planes, 1)
                bn(p + "bn3", planes * 4)
            else:                                                 # BasicBlock, resnet.py:18-25
                conv(p + "conv1.weight", planes, inplanes, 3)
                bn(p + "bn1", planes)
                conv(p + "conv2.weight", planes, planes, 3)
                bn(p + "bn2", planes)
            if b == 0 and (stride != 1 or inplanes != planes * exp):          # resnet.py:136-141
                conv(p + "downsample.0.weight", planes * exp, inplanes, 1)
                bn(p + "downsample.1", planes * exp)
            inplanes = planes * exp
    feat = 512 * exp
    if fpn:
        if fpn_mode == 1:                                         # rmac_resnet_fpn.py:27-30
            conv("conv1x5.weight", 256 * exp, 512 * exp, 1)
            conv("conv3c4.weight", 256 * exp, 256 * exp, 3)
        feat = 768 * exp                                          # rmac_resnet_fpn.py:46
    bound = 1.0 / math.sqrt(feat)
    sd["fc.weight"] = (torch.rand((out_dim, feat), generator=g) * 2 - 1) * bound
    sd["fc.bias"] = (torch.rand(out_dim, generator=g) * 2 - 1) * bound
    return sd


class ResNetRMAC:
    """ResNet-18/50/101/152 trunk + global pooling + FC + L2 (``ResNet_RMAC``, rmac_resnet.py:12-69), or the FPN head
    over the layer3 and layer4 maps (``ResNet_RMAC_FPN``, rmac_resnet_fpn.py:11-90)."""

    def __init__(self, arch, out_dim=None, norm_features=False, pooling="gem", gemp=3, center_bias=0,
                 dropout_p=None, without_fc=False, mode=None, **kwargs):
        kwargs.pop("scales", None)                              # rmac_resnet.py:75,79,83
        if kwargs:
            raise TypeError("unexpected model options: %s" % sorted(kwargs))
        if arch not in _ARCH:
            raise NameError("unknown model architecture '%s'\nSelect one in %s" % (arch, ",".join(sorted(model_names))))
        trunk, self.fpn, default_mode = _ARCH[arch]
        exp = _TRUNKS[trunk][1]
        if mode is not None and not self.fpn:
            raise TypeError("unexpected model options: ['mode']")          # ResNet_RMAC has no `mode` (rmac_resnet.py:15-17)
        self.mode = default_mode if mode is None else int(mode)
        if self.fpn:
            if pooling != "gem":
                # rmac_resnet_fpn.py:36-43,76-77: forward() uses adpoolx5 / adpoolc4, which only pooling='gem' creates
                raise ValueError("the FPN head supports pooling='gem' only (got %r)" % (pooling,))
            if out_dim is None:
                out_dim = 768 * exp                             # rmac_resnet_fpn.py:25
        else:
            if not (pooling in ("max", "avg") or pooling.startswith("gem")):
                raise ValueError(pooling)                        # rmac_resnet.py:30-31
            if out_dim is None:
                out_dim = 2048                                  # rmac_resnet.py:15
        self.arch = arch
        self.model_name = trunk
        self.trunk_dim = (768 if self.fpn else 512) * exp       # fc.in_features
        self.rgb_means = list(RGB_MEANS)                   # resnet.py:110-112
        self.rgb_stds = list(RGB_STDS)
        self.input_size = (3, 224, 224)
        self.norm_features = bool(norm_features)
        self.without_fc = bool(without_fc)
        self.pooling = pooling
        self.center_bias = center_bias
        self.dropout = None                                      # identity in eval mode (rmac_resnet.py:44-45)
        self.fc_name = "fc"
        self.feat_dim = out_dim
        self.out_dim = out_dim
        self.detach = False
        self.iscuda = False
        self.training = False
        self.preprocess = dict(mean=self.rgb_means, std=self.rgb_stds, input_size=max(self.input_size))
        self._sd = _reference_style_init(arch, out_dim, fpn_mode=self.mode)
        if self.fpn:
            self._sd["adpoolx5.p"] = torch.ones(1) * float(gemp)   # rmac_resnet_fpn.py:41-42
            self._sd["adpoolc4.p"] = torch.ones(1) * float(gemp)
        elif pooling.startswith("gem"):
            self._sd["adpool.p"] = torch.ones(1) * float(gemp)   # pooling.py:54
        self._handle = None
        self._handle_device = None
        self._opts = {}

    # ------------------------------------------------------------------ nn.Module-like surface
    def eval(self):
        self.training = False
        return self

    def train(self, mode=True):
        if mode:
            raise NotImplementedError("the B200 path is inference-only (the reference ships no trainer either)")
        return self

    def cuda(self, device=None):
        self.iscuda = True
        return self

    def to(self, *a, **k):
        return self

    def state_dict(self):
        return OrderedDict((k, v.clone()) for k, v in self._sd.items())

    def load_state_dict(self, state_dict, strict=True):
        new = OrderedDict()
        for k, v in state_dict.items():
            if k.startswith("module."):
                k = k[7:]
            new[k] = v.detach().to("cpu")
        missing = [k for k in self._sd if k not in new]
        unexpected = [k for k in new if k not in self._sd]
        if strict and (missing or unexpected):
            raise RuntimeError("Error(s) in loading state_dict: missing keys %s, unexpected keys %s" % (missing, unexpected))
        for k, v in new.items():
            if k in self._sd:
                if tuple(v.shape) != tuple(self._sd[k].shape):
                    raise RuntimeError("size mismatch for %s: %s vs %s" % (k, tuple(v.shape), tuple(self._sd[k].shape)))
                self._sd[k] = v.to(self._sd[k].dtype).clone()
        self._release()
        return self

    def set_backend_option(self, key, value):
        """Library tuning knobs ('chunk', 'conv_impl'); see include/dirb200.h."""
        self._opts[key] = float(value)
        self._release()

    def set_backend_option_live(self, key, value):
        """Change a tuning knob on the existing native handle (no weight re-upload)."""
        self._opts[key] = float(value)
        if self._handle is not None:
            lib.call("dirb200_net_set_option", self._handle, key.encode(), float(value))

    # ------------------------------------------------------------------ native handle
    def _release(self):
        if self._handle is not None:
            lib.raw("dirb200_net_destroy")(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    def _ensure(self, device_index):
        if self._handle is not None and self._handle_device == device_index:
            return self._handle
        self._release()
        h = C.c_void_p()
        lib.call("dirb200_net_create", self.arch.encode(), int(device_index), C.byref(h))
        try:
            mode = 0 if self.pooling.startswith("gem") else (1 if self.pooling == "max" else 2)
            base = [("pooling", mode), ("norm_features", self.norm_features), ("without_fc", self.without_fc),
                    ("out_dim", self.out_dim), ("center_bias", max(0.0, float(self.center_bias)))]
            if self.fpn:
                base.append(("fpn_mode", self.mode))
            for k, v in base + list(self._opts.items()):
                lib.call("dirb200_net_set_option", h, k.encode(), float(v))
            for name, t in self._sd.items():
                if name.endswith("num_batches_tracked"):
                    continue
                a = np.ascontiguousarray(t.detach().cpu().numpy().astype(np.float32))
                shape = (C.c_int64 * max(1, a.ndim))(*a.shape)
                lib.call("dirb200_net_set_tensor", h, name.encode(), a.ctypes.data_as(C.c_void_p), shape, a.ndim)
            lib.call("dirb200_net_finalize", h)
        except Exception:
            lib.raw("dirb200_net_destroy")(h)
            raise
        self._handle, self._handle_device = h, device_index
        return h

    # ------------------------------------------------------------------ forward
    @property
    def descriptor_dim(self):
        return self.trunk_dim if self.without_fc else self.out_dim

    def forward(self, x, want_f16=False):
        if not isinstance(x, torch.Tensor) or x.dim() != 4 or x.shape[1] != 3:
            raise TypeError("expected a (B,3,H,W) tensor")
        if not x.is_cuda:
            x = x.cuda(non_blocking=True)                        # common.variables, common.py:213-215
        x = x.contiguous().float()
        b, _, hgt, wid = x.shape
        h = self._ensure(x.device.index or 0)
        with torch.cuda.device(x.device):
            desc = torch.empty((b, self.descriptor_dim), dtype=torch.float32, device=x.device)
            d16 = torch.empty((b, self.descriptor_dim), dtype=torch.float16, device=x.device) if want_f16 else None
            lib.call("dirb200_net_forward", h, C.c_void_p(x.data_ptr()), b, hgt, wid, C.c_void_p(desc.data_ptr()),
                     C.c_void_p(d16.data_ptr()) if want_f16 else C.c_void_p(0),
                     C.c_void_p(torch.cuda.current_stream().cuda_stream))
        if want_f16:
            return desc, d16
        if b == 1:
            desc = desc[0]                                       # x.squeeze_() at B=1, rmac_resnet.py:64
        return desc

    __call__ = forward

    def forward_host(self, imgs: np.ndarray, device=0) -> np.ndarray:
        """Host NCHW fp32 array in, host descriptors out; H2D + forward + D2H inside one C call."""
        a = np.ascontiguousarray(imgs, dtype=np.float32)
        b, _, hgt, wid = a.shape
        h = self._ensure(device)
        out = np.empty((b, self.descriptor_dim), dtype=np.float32)
        lib.call("dirb200_net_forward_host", h, a.ctypes.data_as(C.c_void_p), b, hgt, wid, out.ctypes.data_as(C.c_void_p))
        return out

    def forward_u8(self, imgs_u8: torch.Tensor):
        """uint8 HWC CUDA tensor (B,H,W,3) -> descriptors; ToTensor + Normalize(self.preprocess) run inside the stem."""
        if not (imgs_u8.is_cuda and imgs_u8.dtype == torch.uint8 and imgs_u8.dim() == 4 and imgs_u8.shape[3] == 3):
            raise TypeError("expected a (B,H,W,3) uint8 CUDA tensor")
        x = imgs_u8.contiguous()
        b, hgt, wid, _ = x.shape
        h = self._ensure_with_preprocess(x.device.index or 0)
        desc = torch.empty((b, self.descriptor_dim), dtype=torch.float32, device=x.device)
        lib.call("dirb200_net_forward_u8", h, C.c_void_p(x.data_ptr()), b, hgt, wid, C.c_void_p(desc.data_ptr()),
                 C.c_void_p(0), C.c_void_p(torch.cuda.current_stream().cuda_stream))
        return desc[0] if b == 1 else desc

    def forward_u8_multiscale(self, imgs_u8: torch.Tensor, scales=(0.7, 1.0, 1.4), pooling="gem", gemp=3):
        """Multi-scale descriptors entirely on the GPU (BASELINE configs[4]): for every scale s the uint8 batch is
        resized like the reference's `Scale(s)` transform (PIL bilinear, output size int(0.5 + s*w), bit-exact on the
        GPU), run through the network, and the per-scale descriptors are pooled (common.pool) and L2-normalised
        (test_dir.py:121-122)."""
        from . import ops
        b, h, w, _ = imgs_u8.shape
        descs = []
        for sc in scales:
            if float(sc) == 1.0:
                x = imgs_u8
            else:
                x = ops.resize_bilinear_u8(imgs_u8.contiguous(), (int(0.5 + sc * h), int(0.5 + sc * w)))
            d = self.forward_u8(x)
            descs.append(d if d.dim() == 2 else d.unsqueeze(0))
        if len(descs) == 1:
            return ops.l2_normalize(descs[0])
        return ops.pool_scales(descs, pooling, gemp, l2=True)

    def forward_host_u8(self, imgs_u8: np.ndarray, device=0) -> np.ndarray:
        """Host uint8 HWC array (B,H,W,3) in, host descriptors out (H2D of 3 bytes/pixel instead of 12)."""
        a = np.ascontiguousarray(imgs_u8, dtype=np.uint8)
        b, hgt, wid, _ = a.shape
        h = self._ensure_with_preprocess(device)
        out = np.empty((b, self.descriptor_dim), dtype=np.float32)
        lib.call("dirb200_net_forward_host_u8", h, a.ctypes.data_as(C.c_void_p), b, hgt, wid, out.ctypes.data_as(C.c_void_p))
        return out

    def _ensure_with_preprocess(self, device_index):
        h = self._ensure(device_index)
        for i in range(3):
            lib.call("dirb200_net_set_option", h, ("mean%d" % i).encode(), float(self.preprocess["mean"][i]))
            lib.call("dirb200_net_set_option", h, ("std%d" % i).encode(), float(self.preprocess["std"][i]))
        return h

    def debug_stage(self, what):
        """NHWC fp16 activation after 'stem' / 'layer1'..'layer4' ('fpn_c4': the merged layer3 map of an FPN head) of
        the last chunk of the last forward (needs set_backend_option('debug_taps', 1))."""
        dims = (C.c_int * 4)()
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        lib.call("dirb200_net_debug_stage", self._handle, what.encode(), C.c_void_p(0), 0, dims, stream)   # size query
        n, hh, ww, c = [int(v) for v in dims]
        out = torch.empty((n, hh, ww, c), dtype=torch.float16, device=torch.device("cuda", self._handle_device))
        lib.call("dirb200_net_debug_stage", self._handle, what.encode(), C.c_void_p(out.data_ptr()), out.numel() * 2, dims,
                 stream)
        return out

    def profile(self):
        """Per-class timing of the last forward (needs set_backend_option('profile', 1)):
        {class: dict(launches, ms, flops, bytes)}."""
        arr = (C.c_double * 16)()
        lib.call("dirb200_net_profile", self._handle, arr)
        names = ["conv_tcgen05", "stem_conv", "layout_maxpool", "head"]
        return {nm: dict(launches=int(arr[4 * i]), ms=arr[4 * i + 1], flops=arr[4 * i + 2], bytes=arr[4 * i + 3])
                for i, nm in enumerate(names)}

    def profile_table(self):
        """Per launch type of the profiled forward(s): list of dict(tag, cls, launches, ms, flops, bytes)."""
        import json
        need = C.c_size_t()
        lib.call("dirb200_net_profile_table", self._handle, C.c_void_p(0), 0, C.byref(need))
        buf = C.create_string_buffer(need.value)
        lib.call("dirb200_net_profile_table", self._handle, buf, need.value, C.byref(need))
        return json.loads(buf.value.decode())

    def last_launch_stats(self):
        n, f = C.c_int64(), C.c_double()
        lib.call("dirb200_net_last_launches", self._handle, C.byref(n), C.byref(f))
        return int(n.value), float(f.value)


def _factory(arch):
    def make(**kwargs):
        return ResNetRMAC(arch, **kwargs)
    make.__name__ = arch
    return make


for _a in _ARCH:                                    # resnet18_rmac ... resnet152_fpn_rmac, as nets/__init__.py:14-16 lists them
    globals()[_a] = _factory(_a)


def create_model(arch, pretrained="", delete_fc=False, *args, **kwargs):
    """nets.create_model, dirtorch/nets/__init__.py:24-64."""
    if arch not in model_names:
        raise NameError("unknown model architecture '%s'\nSelect one in %s" % (arch, ",".join(sorted(model_names))))
    model = ResNetRMAC(arch, *args, **kwargs)
    if os.path.isfile(pretrained or ""):
        weights = torch.load(pretrained, map_location="cpu", weights_only=False)["state_dict"]
        load_pretrained_weights(model, weights, delete_fc=delete_fc)
    elif pretrained:
        raise AssertionError("Model %s must be initialized with a valid model file (not %s)" % (arch, pretrained))
    return model


def load_pretrained_weights(net, state_dict, delete_fc=False):
    """Tolerant load: strips 'module.', keeps the net's own tensor when a layer is missing or mis-shaped
    (dirtorch/nets/__init__.py:67-95)."""
    new = OrderedDict()
    for k, v in state_dict.items():
        new[k[7:] if k.startswith("module.") else k] = v
    own = net.state_dict()
    for k, v in own.items():
        if k not in new:
            if not k.endswith("num_batches_tracked"):
                print("Loading weights for %s: Missing layer %s" % (type(net).__name__, k))
            new[k] = v
        elif tuple(v.shape) != tuple(new[k].shape):
            print("Loading weights for %s: Bad shape for layer %s, skipping" % (type(net).__name__, k))
            new[k] = v
    net.load_state_dict({k: v for k, v in new.items() if k in own})
