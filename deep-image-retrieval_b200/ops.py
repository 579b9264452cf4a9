"""Torch-tensor front-end of the single operators of the C ABI (device memory + streams come from torch).

Every function takes CUDA tensors, hands raw pointers to libdirb200.so and launches on torch's
current stream.  Nothing here computes with torch.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import lib


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(0) if t is None else C.c_void_p(t.data_ptr())


def _chk(t, dtype, name):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dtype and t.is_contiguous()):
        raise TypeError("%s must be a contiguous CUDA tensor of dtype %s" % (name, dtype))
    return t


def require_gpu(device=0):
    lib.call("dirb200_device_check", int(device))


def set_global_option(key, value):
    """Process-wide kernel selectors ('halo', 'pdl', 'res_variant', 'l2_prefetch', 'head_fused'); include/dirb200.h."""
    lib.call("dirb200_set_global_option", key.encode(), float(value))


def get_global_option(key):
    v = C.c_double()
    lib.call("dirb200_get_global_option", key.encode(), C.byref(v))
    return v.value


def nchw_to_nhwc8(x):
    _chk(x, torch.float32, "x")
    b, c, h, w = x.shape
    assert c == 3
    out = torch.empty((b, h, w, 8), dtype=torch.float16, device=x.device)
    lib.call("dirb200_nchw_to_nhwc8", _ptr(x), b, h, w, _ptr(out), _stream())
    return out


def pack_conv_weight(w_oihw: torch.Tensor, cin_pad=None) -> torch.Tensor:
    """OIHW fp32 -> [Cout][KH][KW][CinPad] fp16, rows zero-padded to a multiple of 32 (the layout
    dirb200_conv_bn_act expects).  Host-side repack (weights are packed once)."""
    o, i, kh, kw = w_oihw.shape
    cp = cin_pad or i
    w = torch.zeros((o, kh, kw, cp), dtype=torch.float32)
    w[..., :i] = w_oihw.detach().float().cpu().permute(0, 2, 3, 1)
    k = kh * kw * cp
    kpad = (k + 31) // 32 * 32
    out = torch.zeros((o, kpad), dtype=torch.float16)
    out[:, :k] = w.reshape(o, k).half()
    return out


def conv_bn_act(x, w_packed, cout, kh, kw, stride, pad, scale, shift, res=None, relu=True, impl=0):
    """x NHWC fp16 (B,H,W,Cin) -> NHWC fp16 (B,Ho,Wo,Cout)."""
    _chk(x, torch.float16, "x")
    _chk(w_packed, torch.float16, "w_packed")
    _chk(scale, torch.float32, "scale")
    _chk(shift, torch.float32, "shift")
    b, h, w, cin = x.shape
    ho = (h + 2 * pad - kh) // stride + 1
    wo = (w + 2 * pad - kw) // stride + 1
    out = torch.empty((b, ho, wo, cout), dtype=torch.float16, device=x.device)
    if res is not None:
        _chk(res, torch.float16, "res")
        assert res.shape == out.shape
    lib.call("dirb200_conv_bn_act", _ptr(x), b, h, w, cin, _ptr(w_packed), cout, kh, kw, stride, pad, _ptr(scale),
             _ptr(shift), _ptr(res), int(bool(relu)), int(impl), _ptr(out), _stream())
    return out


def conv_c23(t1, w2_packed, scale2, shift2, w3_packed, scale3, shift3, res, variant=1):
    """Fused Bottleneck tail: relu(bn3(conv1x1(relu(bn2(conv3x3(t1))))) + res).  t1 NHWC fp16 (B,H,W,Cm) -> (B,H,W,4Cm)."""
    _chk(t1, torch.float16, "t1")
    _chk(res, torch.float16, "res")
    b, h, w, cm = t1.shape
    assert tuple(res.shape) == (b, h, w, 4 * cm)
    out = torch.empty_like(res)
    lib.call("dirb200_conv_c23", _ptr(t1), b, h, w, cm, _ptr(_chk(w2_packed, torch.float16, "w2")), _ptr(scale2), _ptr(shift2),
             _ptr(_chk(w3_packed, torch.float16, "w3")), _ptr(scale3), _ptr(shift3), _ptr(res), _ptr(out), int(variant), _stream())
    return out


def stem_conv(x_nchw, w_oihw, scale, shift):
    """Conv 7x7/s2/p3 (3->64) + BN + ReLU on tensor cores: NCHW fp32 (B,3,H,W) -> NHWC fp16 (B,Ho,Wo,64)."""
    _chk(x_nchw, torch.float32, "x_nchw")
    b, c, h, w = x_nchw.shape
    assert c == 3 and tuple(w_oihw.shape) == (64, 3, 7, 7)
    wh = np.ascontiguousarray(w_oihw.detach().cpu().numpy().astype(np.float32))
    w2 = np.empty((64, 256), dtype=np.float16)
    lib.call("dirb200_stem_pack_weight", wh.ctypes.data_as(C.c_void_p), w2.ctypes.data_as(C.c_void_p))
    w2d = torch.from_numpy(w2).to(x_nchw.device)
    ws = torch.empty(lib.raw("dirb200_stem_workspace_bytes")(b, h, w), dtype=torch.uint8, device=x_nchw.device)
    ho, wo = (h + 6 - 7) // 2 + 1, (w + 6 - 7) // 2 + 1
    out = torch.empty((b, ho, wo, 64), dtype=torch.float16, device=x_nchw.device)
    lib.call("dirb200_stem_conv", _ptr(x_nchw), b, h, w, _ptr(w2d), _ptr(_chk(scale, torch.float32, "scale")),
             _ptr(_chk(shift, torch.float32, "shift")), _ptr(ws), _ptr(out), _stream())
    return out


def resize_bilinear_u8(x_u8, size):
    """uint8 HWC CUDA tensor (B,H,W,3) -> (B,Ho,Wo,3), byte-identical to PIL Image.resize((Wo,Ho), BILINEAR)."""
    _chk(x_u8, torch.uint8, "x_u8")
    b, h, w, c = x_u8.shape
    assert c == 3
    ho, wo = int(size[0]), int(size[1])
    out = torch.empty((b, ho, wo, 3), dtype=torch.uint8, device=x_u8.device)
    lib.call("dirb200_resize_bilinear_u8", _ptr(x_u8), b, h, w, ho, wo, _ptr(out), _stream())
    return out


def resize_coeffs(in_size, out_size):
    """Host-only: PIL's fixed-point bilinear coefficient table of one axis -> (bounds [out,2], kk [out,ksize])."""
    ks = C.c_int()
    lib.call("dirb200_resize_coeffs", int(in_size), int(out_size), C.c_void_p(0), C.c_void_p(0), C.byref(ks))
    bounds = np.zeros((out_size, 2), dtype=np.int32)
    kk = np.zeros((out_size, ks.value), dtype=np.int32)
    lib.call("dirb200_resize_coeffs", int(in_size), int(out_size), bounds.ctypes.data_as(C.c_void_p),
             kk.ctypes.data_as(C.c_void_p), C.byref(ks))
    return bounds, kk


def maxpool_3x3s2(x):
    _chk(x, torch.float16, "x")
    b, h, w, c = x.shape
    out = torch.empty((b, (h - 1) // 2 + 1, (w - 1) // 2 + 1, c), dtype=torch.float16, device=x.device)
    lib.call("dirb200_maxpool_3x3s2", _ptr(x), b, h, w, c, _ptr(out), _stream())
    return out


def center_bias(x, b):
    """In place on x (NHWC fp16 (B,H,W,C)): x *= 1 + the center-bias map of rmac_resnet.py:52-56; returns x."""
    _chk(x, torch.float16, "x")
    bb, h, w, c = x.shape
    lib.call("dirb200_center_bias", _ptr(x), bb, h, w, c, float(b), _stream())
    return x


POOLING = {"gem": 0, "max": 1, "avg": 2}


def head_pool_fc_l2(feat, pooling="gem", p=3.0, eps=1e-6, norm_features=False, fc_w=None, fc_b=None, want_f16=False):
    """feat NHWC fp16 (B,h,w,C) -> (B,D) fp32 L2-normalised (rmac_resnet.py:59-68)."""
    _chk(feat, torch.float16, "feat")
    b, h, w, c = feat.shape
    out_dim = fc_w.shape[0] if fc_w is not None else c
    if fc_w is not None:
        _chk(fc_w, torch.float32, "fc_w")
        _chk(fc_b, torch.float32, "fc_b")
    nws = lib.raw("dirb200_head_workspace_floats")(b, h * w, c, out_dim)
    ws = torch.empty(nws, dtype=torch.float32, device=feat.device)
    desc = torch.empty((b, out_dim), dtype=torch.float32, device=feat.device)
    d16 = torch.empty((b, out_dim), dtype=torch.float16, device=feat.device) if want_f16 else None
    mode = POOLING["gem" if pooling.startswith("gem") else pooling]
    lib.call("dirb200_head_pool_fc_l2", _ptr(feat), b, h * w, c, mode, float(p), float(eps), int(bool(norm_features)),
             _ptr(fc_w), _ptr(fc_b), out_dim, _ptr(ws), _ptr(desc), _ptr(d16), _stream())
    return (desc, d16) if want_f16 else desc


def pool_scales(xs, pooling="mean", gemp=3, l2=True):
    """common.pool (+ F.normalize when l2): list of (N,D) fp32 CUDA tensors -> (N,D)."""
    if pooling not in ("mean", "gem"):
        raise ValueError("Bad pooling mode: " + str(pooling))
    stacked = torch.stack([_chk(x, torch.float32, "xs[i]") for x in xs], dim=0).contiguous()
    s, n, d = stacked.shape
    out = torch.empty((n, d), dtype=torch.float32, device=stacked.device)
    lib.call("dirb200_pool_scales", _ptr(stacked), s, n, d, 0 if pooling == "mean" else 1, float(gemp), int(bool(l2)),
             _ptr(out), _stream())
    return out


def l2_normalize(x, eps=1e-12, want_f16=False):
    _chk(x, torch.float32, "x")
    n, d = x.shape
    out = torch.empty_like(x)
    o16 = torch.empty((n, d), dtype=torch.float16, device=x.device) if want_f16 else None
    lib.call("dirb200_l2_normalize", _ptr(x), n, d, float(eps), _ptr(out), _ptr(o16), _stream())
    return (out, o16) if want_f16 else out


def f32_to_f16(x):
    _chk(x, torch.float32, "x")
    out = torch.empty(x.shape, dtype=torch.float16, device=x.device)
    lib.call("dirb200_f32_to_f16", _ptr(x), x.numel(), _ptr(out), _stream())
    return out


def whiten(x, comp, mean=None, colscale=None, l2norm=True, want_f16=False):
    """((x - mean) . comp^T) * colscale, row L2 (common.py:221-239).  x (N,D), comp (Dout,D) fp32 CUDA."""
    _chk(x, torch.float32, "x")
    _chk(comp, torch.float32, "comp")
    n, d = x.shape
    dout = comp.shape[0]
    y = torch.empty((n, dout), dtype=torch.float32, device=x.device)
    y16 = torch.empty((n, dout), dtype=torch.float16, device=x.device) if want_f16 else None
    lib.call("dirb200_whiten", _ptr(x), n, d, _ptr(comp), _ptr(mean), _ptr(colscale), dout, int(bool(l2norm)), _ptr(y),
             _ptr(y16), _stream())
    return (y, y16) if want_f16 else y


def scores_exact(q, db):
    """Dense exact scores (Q,N) fp32 = q . db^T (fp64 accumulation).  Any D: the kernel reads rows as float4, so both
    operands are zero-padded to a multiple of 4 columns (zero columns change no score)."""
    _chk(q, torch.float32, "q")
    _chk(db, torch.float32, "db")
    if q.shape[1] != db.shape[1]:
        raise ValueError("descriptor dimensions differ: %d vs %d" % (q.shape[1], db.shape[1]))
    pad = (-q.shape[1]) % 4
    if pad:
        q = torch.nn.functional.pad(q, (0, pad)).contiguous()
        db = torch.nn.functional.pad(db, (0, pad)).contiguous()
    out = torch.empty((q.shape[0], db.shape[0]), dtype=torch.float32, device=q.device)
    lib.call("dirb200_scores_exact", _ptr(q), q.shape[0], _ptr(db), db.shape[0], q.shape[1], _ptr(out), _stream())
    return out


def topk_merge(scores, idx, k):
    """scores/idx: (G,Q,k) fp64 / int64 per-shard lists with global indices -> merged (Q,k)."""
    _chk(scores, torch.float64, "scores")
    _chk(idx, torch.int64, "idx")
    g, q, kk = scores.shape
    assert kk == k
    os_ = torch.empty((q, k), dtype=torch.float64, device=scores.device)
    oi = torch.empty((q, k), dtype=torch.int64, device=scores.device)
    lib.call("dirb200_topk_merge", _ptr(scores), _ptr(idx), g, q, k, 0, _ptr(os_), _ptr(oi), _stream())
    return os_, oi


def topk_merge_packed(packed, k):
    """packed: (G,2,Q,k) int64 all-gather buffer, [:,0] = fp64 score bits, [:,1] = global indices -> merged (Q,k)."""
    _chk(packed, torch.int64, "packed")
    g, two, q, kk = packed.shape
    assert two == 2 and kk == k
    os_ = torch.empty((q, k), dtype=torch.float64, device=packed.device)
    oi = torch.empty((q, k), dtype=torch.int64, device=packed.device)
    base = packed.data_ptr()
    lib.call("dirb200_topk_merge", C.c_void_p(base), C.c_void_p(base + q * k * 8), g, q, k, 2 * q * k, _ptr(os_),
             _ptr(oi), _stream())
    return os_, oi


def aqe_expand(q, db32, nn_idx, nn_scores, alpha, partial=False, row_offset=0, n_rows=0):
    _chk(q, torch.float32, "q")
    _chk(db32, torch.float32, "db32")
    _chk(nn_idx, torch.int64, "nn_idx")
    _chk(nn_scores, torch.float64, "nn_scores")
    out = torch.empty_like(q)
    lib.call("dirb200_aqe_expand", _ptr(q), q.shape[0], q.shape[1], _ptr(db32), _ptr(nn_idx), _ptr(nn_scores),
             nn_idx.shape[1], float(alpha), int(bool(partial)), int(row_offset), int(n_rows), _ptr(out), _stream())
    return out


class Exchange:
    """This rank's window of the peer-memory exchange of a sharded search (include/dirb200.h: dirb200_exchange_*)."""

    def __init__(self, device_index: int, world: int, rank: int, max_q: int, max_k: int):
        self.world, self.rank, self.max_q, self.max_k = int(world), int(rank), int(max_q), int(max_k)
        self._h = C.c_void_p()
        lib.call("dirb200_exchange_create", int(device_index), self.world, self.rank, self.max_q, self.max_k, C.byref(self._h))

    def ipc_handle(self) -> bytes:
        buf = C.create_string_buffer(64)
        lib.call("dirb200_exchange_ipc_handle", self._h, buf)
        return buf.raw

    def open(self, handles) -> None:
        """handles: the 64-byte IPC handles of all ranks in rank order (this rank's own entry is ignored)."""
        blob = b"".join(bytes(h) for h in handles)
        assert len(blob) == 64 * self.world
        lib.call("dirb200_exchange_open", self._h, C.c_char_p(blob))

    @staticmethod
    def open_local(group) -> None:
        """Same-process group: `group` = the exchange objects of all ranks, in rank order."""
        arr = (C.c_void_p * len(group))(*[x._h for x in group])
        for x in group:
            lib.call("dirb200_exchange_open_local", x._h, arr)

    def close_peers(self):
        """Unmap the other ranks' windows (every rank, then a barrier, then close())."""
        if self._h:
            lib.call("dirb200_exchange_close_peers", self._h)

    def close(self):
        if self._h:
            lib.raw("dirb200_exchange_destroy")(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Index:
    """One row shard of a descriptor database on one GPU (dirb200_index)."""

    def __init__(self, db32: torch.Tensor, index_offset: int = 0, db16: torch.Tensor = None, check_norms: bool = True):
        """check_norms: the exactness of the top-k rests on |fp16-path score - exact score| <= eps16 = 1.2e-3, which is
        derived for UNIT-NORM rows and queries (what pooling / whitening / query expansion produce).  Rows with larger
        norms are refused here instead of silently returning an inexact list; pass check_norms=False and set option
        'eps16' to 1.2e-3 * max|q| * max|row| to search un-normalised data."""
        _chk(db32, torch.float32, "db32")
        if check_norms and db32.shape[0]:
            worst = float(torch.linalg.vector_norm(db32, dim=1).max())
            if worst > 1.0 + 1e-3:
                raise ValueError("database rows are not unit-norm (max norm %.4g): the exact-top-k error bound assumes |row| <= 1; "
                                 "normalise them, or pass check_norms=False and set option 'eps16' accordingly" % worst)
        self.db32 = db32
        self.n, self.dim = db32.shape
        if db16 is None:                      # an empty shard (more ranks than rows) has nothing to convert
            db16 = f32_to_f16(db32) if self.n else torch.empty((0, self.dim), dtype=torch.float16, device=db32.device)
        self.db16 = db16
        self.offset = int(index_offset)
        self._h = C.c_void_p()
        lib.call("dirb200_index_create", db32.device.index or 0, self.dim, C.byref(self._h))
        lib.call("dirb200_index_set_db", self._h, _ptr(self.db32), _ptr(self.db16), self.n, self.offset)

    def set_option(self, key, value):
        lib.call("dirb200_index_set_option", self._h, key.encode(), float(value))

    def search(self, q32: torch.Tensor, k: int, out=None):
        """-> (scores fp64 (Q,k), idx int64 (Q,k)), exact order: score desc, index asc.
        out: optional (2,Q,k) int64 buffer that receives [score bits, indices] (the all-gather payload)."""
        _chk(q32, torch.float32, "q32")
        nq = q32.shape[0]
        if out is not None:
            _chk(out, torch.int64, "out")
            assert tuple(out.shape) == (2, nq, k)
            scores, idx = out[0].view(torch.float64), out[1]
        else:
            scores = torch.empty((nq, k), dtype=torch.float64, device=q32.device)
            idx = torch.empty((nq, k), dtype=torch.int64, device=q32.device)
        try:
            lib.call("dirb200_index_search", self._h, _ptr(q32), nq, int(k), _ptr(scores), _ptr(idx), _stream())
        except lib.DirbError as e:
            if e.status != -4:                      # DIRB200_EOVERFLOW: candidate lists did not fit after the retry passes
                raise
            # rare (clustered databases whose first rows are not a sample of the rest): run again with more gated
            # retry passes and a larger candidate buffer, then restore the defaults
            self.set_option("retries", 4)
            self.set_option("cand_cap", 1 << 17)
            try:
                lib.call("dirb200_index_search", self._h, _ptr(q32), nq, int(k), _ptr(scores), _ptr(idx), _stream())
                lib.call("dirb200_index_check", self._h)
            finally:
                self.set_option("retries", 1)
                self.set_option("cand_cap", 0)
        return scores, idx

    def search_begin(self, q32: torch.Tensor, k: int, k_shard: int):
        """Phase 1 of a sharded search -> sel (Q,) fp32: local k_shard-th best fp16-path score (MIN-reduce it)."""
        _chk(q32, torch.float32, "q32")
        sel = torch.empty(q32.shape[0], dtype=torch.float32, device=q32.device)
        lib.call("dirb200_index_search_begin", self._h, _ptr(q32), q32.shape[0], int(k), int(k_shard), _ptr(sel), _stream())
        return sel

    def search_finish(self, q32: torch.Tensor, k: int, sel: torch.Tensor, out=None):
        """Phase 2: exact re-scoring of the rows within the band of the (reduced) threshold -> ordered local list."""
        nq = q32.shape[0]
        if out is not None:
            scores, idx = out[0].view(torch.float64), out[1]
        else:
            scores = torch.empty((nq, k), dtype=torch.float64, device=q32.device)
            idx = torch.empty((nq, k), dtype=torch.int64, device=q32.device)
        lib.call("dirb200_index_search_finish", self._h, _ptr(q32), _ptr(_chk(sel, torch.float32, "sel")), _ptr(scores),
                 _ptr(idx), _stream())
        return scores, idx

    def search_sharded(self, exchange: "Exchange", q32: torch.Tensor, k: int, k_shard: int, phase: int = 0):
        """Collective exact top-k over all shards through the peer-memory exchange (no library collective): every rank
        calls it with the same (Q, k, k_shard).  phase 0 = the whole search; 1 .. 4 = one phase (seed bounds, filter +
        selection, re-scoring, merge: several shards driven shard by shard from one process).
        -> (scores fp64, idx int64) (Q,k) after phase 0 / 4, else None.
        Never synchronises: call check() (or the next search) to collect the status."""
        _chk(q32, torch.float32, "q32")
        nq = q32.shape[0]
        scores = idx = None
        if phase in (0, 4):
            scores = torch.empty((nq, k), dtype=torch.float64, device=q32.device)
            idx = torch.empty((nq, k), dtype=torch.int64, device=q32.device)
        if phase == 0:
            lib.call("dirb200_index_search_sharded", self._h, exchange._h, _ptr(q32), nq, int(k), int(k_shard), _ptr(scores),
                     _ptr(idx), _stream())
        else:
            lib.call("dirb200_index_search_sharded_phase", self._h, exchange._h, int(phase), _ptr(q32), nq, int(k), int(k_shard),
                     _ptr(scores), _ptr(idx), _stream())
        return (scores, idx) if scores is not None else None

    def target_scores(self, q32, t_q, t_rows):
        """Exact scores <q32[t_q[t]], db[t_rows[t]]> (fp64) of the target rows this shard owns, 0 for the others.
        t_q int32 (T,), t_rows int64 (T,) global indices - CUDA tensors."""
        _chk(q32, torch.float32, "q32")
        _chk(t_q, torch.int32, "t_q")
        _chk(t_rows, torch.int64, "t_rows")
        out = torch.zeros(t_rows.shape[0], dtype=torch.float64, device=q32.device)
        lib.call("dirb200_index_target_scores", self._h, _ptr(q32), q32.shape[0], _ptr(t_q), _ptr(t_rows), t_rows.shape[0],
                 _ptr(out), _stream())
        return out

    def rank_count(self, q32, t_off, t_rows, t_flags, t_score):
        """above[t] = number of rows of this shard ranking before target t (exact score desc, ties -> lower index) for
        the flagged targets of each query.  t_off: host int32 ndarray (Q+1,), the CSR offsets of the targets; t_rows
        int64 / t_flags uint8 / t_score fp64 CUDA tensors (T,)."""
        _chk(q32, torch.float32, "q32")
        _chk(t_rows, torch.int64, "t_rows")
        _chk(t_flags, torch.uint8, "t_flags")
        _chk(t_score, torch.float64, "t_score")
        off_h = np.ascontiguousarray(t_off, dtype=np.int32)
        assert off_h.shape[0] == q32.shape[0] + 1
        off_d = torch.from_numpy(off_h).to(q32.device)
        above = torch.zeros(t_rows.shape[0], dtype=torch.int64, device=q32.device)
        lib.call("dirb200_index_rank_count", self._h, _ptr(q32), q32.shape[0], off_h.ctypes.data_as(C.c_void_p), _ptr(off_d),
                 _ptr(t_rows), _ptr(t_flags), _ptr(t_score), t_rows.shape[0], _ptr(above), _stream())
        return above

    def rank_counts(self, q32, t_off, t_rows, t_flags):
        """Single-shard convenience: (exact scores fp64 (T,), rows ranking before each flagged target int64 (T,))."""
        off = np.ascontiguousarray(t_off, dtype=np.int32)
        t_q = torch.from_numpy(np.repeat(np.arange(q32.shape[0], dtype=np.int32), np.diff(off))).to(q32.device)
        rows = torch.as_tensor(np.ascontiguousarray(t_rows, dtype=np.int64)).to(q32.device)
        flags = torch.as_tensor(np.ascontiguousarray(t_flags, dtype=np.uint8)).to(q32.device)
        sc = self.target_scores(q32, t_q, rows)
        return sc, self.rank_count(q32, off, rows, flags, sc)

    def check(self):
        """Collect the status of the last search (option deferred_check): raises DirbError on an unresolved overflow."""
        lib.call("dirb200_index_check", self._h)

    def stats(self):
        arr = (C.c_int64 * 5)()
        lib.call("dirb200_index_last_stats", self._h, arr)
        return dict(zip(["dense_rows", "candidates", "survivors", "retries", "launches"], [int(v) for v in arr]))

    def profile(self):
        arr = (C.c_double * 9)()
        lib.call("dirb200_index_last_profile", self._h, arr)
        names = ["prep", "seed_gemm", "seed_kth", "filter_gemm", "cand_select", "retry_gates", "finish"]
        return {n: float(arr[i]) for i, n in enumerate(names)}

    def close(self):
        if self._h:
            lib.raw("dirb200_index_destroy")(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
