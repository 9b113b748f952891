"""``torch.autograd.Function`` wrappers around the C ABI -- host plumbing only.

Every tensor the kernels touch is allocated here through torch's caching allocator on the current stream
(the library never allocates per call, SURVEY.md section 8(b) "ownership").  All feature tensors are fp32
"node-major": ``(N, B, p)`` contiguous, rows ``r = n*B + b``.

Functions (reference lines they replace):
  ObsToNodeMajor   STMGCN.py:36,39 (sum over C, permute) and :47 (row order of the shared LSTM)
  ChebGCN          GCN.py:24-43 on a sparse L~ (recurrence on features) -> out (N,B,q)
  TemporalPool     STMGCN.py:40-42: GCN over time-as-features + residual + sum over regions -> (B,T)
  ContextGate      STMGCN.py:42-43: /N, fc, relu, fc (same weights), sigmoid -> s (B,T)
  SharedLSTM       STMGCN.py:44,47-50: modulate + 3-layer shared LSTM -> SharedLSTM16 (lstm16.cu) or SharedLSTMExact (lstm.cu)
  FuseOut          STMGCN.py:116-118: sum over graphs + output FC -> (B,N,C)
"""
from __future__ import annotations

import os
from collections import OrderedDict
from typing import List, Optional, Sequence

import torch

from . import _lib
from .graph import SupportSet

L = _lib.lib


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


_LSTM_PATH = os.environ.get("STMGCN_LSTM_PATH", "tc")


def lstm_path() -> str:
    """"tc": tcgen05 kernels where shapes allow (LSTM: H = 64, C <= 4; projection: p = q = 64); "fma": exact-fp32 FFMA kernels."""
    return _LSTM_PATH


def set_lstm_path(path: str) -> None:
    global _LSTM_PATH
    if path not in ("tc", "fma"):
        raise ValueError(path)
    _LSTM_PATH = path


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("stmgcn_b200 kernels need CUDA tensors (there is no CPU fallback)")


# --------------------------------------------------------------------------------------------------
# raw helpers (no autograd)
# --------------------------------------------------------------------------------------------------
def spmm_step(g, transpose: bool, alpha: float, x: torch.Tensor, beta: float, z: Optional[torch.Tensor],
              gamma: float, u: Optional[torch.Tensor], y: torch.Tensor) -> None:
    """``y = alpha * op(A) x + beta * z + gamma * u`` on ``(N, F)`` views."""
    n = g.n
    f_total = x.numel() // n
    _lib.check(L.stmgcn_cheb_spmm_step(g.ptr, int(transpose), alpha, x.data_ptr(), beta, _p(z), gamma, _p(u),
                                       y.data_ptr(), f_total, _stream()), "cheb_spmm_step")


def spmm_step16(g, transpose: bool, alpha: float, x16: torch.Tensor, beta: float, z: Optional[torch.Tensor],
                gamma: float, u: Optional[torch.Tensor], y: torch.Tensor, y16: Optional[torch.Tensor]) -> None:
    """:func:`spmm_step` with the gathered operand read from its bf16 copy ``x16``; writes the bf16 copy of ``y`` to ``y16``."""
    f_total = y.numel() // g.n
    _lib.check(L.stmgcn_cheb_spmm_step16(g.ptr, int(transpose), alpha, x16.data_ptr(), beta, _p(z), gamma, _p(u),
                                         y.data_ptr(), _p(y16), f_total, _stream()), "cheb_spmm_step16")


def to_bf16(x: torch.Tensor) -> torch.Tensor:
    y = torch.empty(x.shape, device=x.device, dtype=torch.bfloat16)
    _lib.check(L.stmgcn_to_bf16(x.data_ptr(), y.data_ptr(), x.numel(), _stream()), "to_bf16")
    return y


def _gather16(sset: SupportSet, x: torch.Tensor) -> bool:
    """bf16 gather copies: only in the single-plane (bf16 arithmetic) mode, for the recurrence over one graph."""
    return lstm_planes() == 1 and sset.mode == "cheb" and (x.numel() // sset.graphs[0].n) % 8 == 0 and x.numel() % 8 == 0


def cheb_stack_(sset: SupportSet, s: torch.Tensor, gather16: bool = False) -> None:
    """Fill ``s[1:]`` from ``s[0]``;  s: (Ks, N, B, p).  ``gather16``: allow bf16 gather copies (bf16-arithmetic mode only)."""
    ks = sset.ks
    if sset.mode == "cheb":
        if ks > 1:
            g = sset.graphs[0]
            if gather16 and _gather16(sset, s[0]):
                # bf16 mode: every step gathers from the bf16 copy of the previous term (half the gather volume)
                src = to_bf16(s[0])
                nxt = torch.empty_like(src) if ks > 2 else None
                for k in range(1, ks):
                    out16 = nxt if k < ks - 1 else None
                    spmm_step16(g, False, 1.0 if k == 1 else 2.0, src, 0.0 if k == 1 else -1.0, None if k == 1 else s[k - 2],
                                0.0, None, s[k], out16)
                    src, nxt = out16, src
                return
            spmm_step(g, False, 1.0, s[0], 0.0, None, 0.0, None, s[1])
            for k in range(2, ks):
                spmm_step(g, False, 2.0, s[k - 1], -1.0, s[k - 2], 0.0, None, s[k])
    else:
        raise AssertionError("generic supports are stacked by cheb_stack_generic")


def cheb_stack_generic(sset: SupportSet, x: torch.Tensor) -> torch.Tensor:
    """Generic supports: S_k = A_k x for every k (including k = 0)."""
    s = torch.empty((sset.ks,) + tuple(x.shape), device=x.device, dtype=torch.float32)
    for k in range(sset.ks):
        spmm_step(sset.graphs[k], False, 1.0, x, 0.0, None, 0.0, None, s[k])
    return s


def build_stack(sset: SupportSet, x: torch.Tensor, gather16: bool = False) -> torch.Tensor:
    if sset.mode == "cheb":
        s = torch.empty((sset.ks,) + tuple(x.shape), device=x.device, dtype=torch.float32)
        s[0].copy_(x)
        cheb_stack_(sset, s, gather16)
        return s
    return cheb_stack_generic(sset, x)


def adjoint_stack_(sset: SupportSet, u: torch.Tensor) -> torch.Tensor:
    """Given U_k = dZ W_k^T stacked in ``u`` (Ks, N, B, p) return dX (N, B, p); ``u`` is clobbered.

    cheb: adjoint Clenshaw with L~^T (SURVEY.md section 8(a)); generic: sum_k A_k^T U_k.
    """
    ks = sset.ks
    if sset.mode == "cheb":
        if ks == 1:
            return u[0]
        g = sset.graphs[0]
        k_ord = ks - 1
        # b_K = U_K (in place).  b_k = U_k + 2 L^T b_{k+1} - b_{k+2}  written over U_k.
        # (always fp32 gathers here, also in the bf16-arithmetic mode: rounding b_{k+1} to bf16 before every gather puts
        # ~1.5e-2 into dX on the golden case -- the Clenshaw sum cancels -- and pushed one LSTM weight gradient to 2.2e-2,
        # past the 2e-2 bar of that mode; measured.  The forward stack keeps its bf16 gather copies.)
        for k in range(k_ord - 1, 0, -1):
            z = u[k + 2] if k + 2 <= k_ord else None
            spmm_step(g, True, 2.0, u[k + 1], -1.0 if z is not None else 0.0, z, 1.0, u[k], u[k])
        z = u[2] if k_ord >= 2 else None
        spmm_step(g, True, 1.0, u[1], -1.0 if z is not None else 0.0, z, 1.0, u[0], u[0])
        return u[0]
    out = torch.empty_like(u[0])
    acc = None
    for k in range(ks):
        tgt = out if (k % 2 == 0) else torch.empty_like(out)
        spmm_step(sset.graphs[k], True, 1.0, u[k], 0.0, None, 1.0 if acc is not None else 0.0, acc, tgt)
        acc = tgt
    return acc


_IMAGE_CACHE_SIZE = 24
_PROJ_IMAGES: "OrderedDict" = OrderedDict()
_LSTM16_IMAGES: "OrderedDict" = OrderedDict()


def _cached_images(store: "OrderedDict", params: Sequence[torch.Tensor], extra: tuple, pack, usable=None) -> dict:
    """The dict ``pack()`` returns (operand images of ``params``, packed on the current stream), cached in the LRU ``store``
    on storage + in-place version of every parameter and ``extra``: re-packed only after an optimizer step changed them,
    or when ``usable(hit)`` rejects the hit.  During CUDA-graph capture the cache is bypassed so the pack kernels become
    part of the graph (replays see updated weights)."""
    capturing = torch.cuda.is_current_stream_capturing()
    key = tuple((w.data_ptr(), w._version) for w in params) + extra + (str(params[0].device),)
    if not capturing:
        hit = store.get(key)
        if hit is not None and (usable is None or usable(hit)):
            store.move_to_end(key)
            torch.cuda.current_stream().wait_event(hit["event"])
            return hit
    entry = pack()
    if not capturing:
        entry["event"] = torch.cuda.Event()
        entry["event"].record()
        entry["keep"] = list(params)          # keeps the storages alive: a recycled data_ptr can never alias the key
        store[key] = entry
        while len(store) > _IMAGE_CACHE_SIZE:
            store.popitem(last=False)
    return entry


def _proj_tc(ks: int, p: int, q: int) -> bool:
    """Whether ChebGCN's projection runs on the tcgen05 3xTF32 entries (stmgcn_proj_fwd_tc / _bwd_tc) rather than the
    exact-FFMA ones.  Those entries also require 16-byte aligned pointers and strides that are multiples of 4 floats;
    everything ChebGCN passes them is allocated here (build_stack, torch.empty; stride_k = N*B*64), so that holds by
    construction, except for the incoming gradient d_out.  ChebGCN.backward therefore takes the tensor-core entry only
    when the forward took it (it packed the backward image), dX is needed (the entry always produces U) and d_out is
    16-byte aligned; otherwise it calls the FFMA entry."""
    return lstm_path() == "tc" and p == 64 and q == 64 and ks <= 8


def _proj_images(w: torch.Tensor, ks: int, need_bwd: bool):
    """tcgen05 operand images (forward, backward) of the projection weights (64, 64 per support, ks <= 8).  The backward
    image is packed only when ``need_bwd``; an entry without it is re-packed when a later call needs it."""

    def pack():
        img_f = torch.empty(ks * 64 * 64 * 2, device=w.device, dtype=torch.float32)
        img_b = torch.zeros((2 if ks > 4 else 1) * 2 * 2 * 256 * 32, device=w.device, dtype=torch.float32) if need_bwd else None
        _lib.check(L.stmgcn_proj_pack_tc(w.data_ptr(), ks, img_f.data_ptr(), _p(img_b), _stream()), "proj_pack_tc")
        return dict(fwd=img_f, bwd=img_b)

    img = _cached_images(_PROJ_IMAGES, [w], (ks,), pack, lambda hit: hit["bwd"] is not None or not need_bwd)
    return img["fwd"], img["bwd"]


def _proj_fwd(s: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], act: int, pool: Optional[torch.Tensor],
              b_inner: int) -> torch.Tensor:
    ks, n, b, p = s.shape
    q = w.shape[1]
    out = torch.empty((n, b, q), device=s.device, dtype=torch.float32)
    _lib.check(L.stmgcn_proj_fwd(s.data_ptr(), n * b * p, ks, n * b, p, w.data_ptr(), _p(bias), q, act,
                                 out.data_ptr(), _p(pool), b_inner, _stream()), "proj_fwd")
    return out


def _proj_fwd_tc(s: torch.Tensor, wimg: torch.Tensor, bias: Optional[torch.Tensor], act: int) -> torch.Tensor:
    ks, n, b, _ = s.shape
    out = torch.empty((n, b, 64), device=s.device, dtype=torch.float32)
    _lib.check(L.stmgcn_proj_fwd_tc(s.data_ptr(), n * b * 64, ks, n * b, wimg.data_ptr(), _p(bias), act, out.data_ptr(),
                                    _stream()), "proj_fwd_tc")
    return out


def _proj_bwd(s: torch.Tensor, w: torch.Tensor, act: int, out: torch.Tensor, d_out: Optional[torch.Tensor],
              d_bcast: Optional[torch.Tensor], scale: float, b_inner: int, need_bias: bool, need_u: bool):
    ks, n, b, p = s.shape
    q = w.shape[1]
    dw = torch.zeros_like(w, dtype=torch.float32)
    db = torch.zeros(q, device=s.device, dtype=torch.float32) if need_bias else None
    dz = torch.empty((n * b, q), device=s.device, dtype=torch.float32)
    u = torch.empty_like(s) if need_u else None
    wt = w.t().contiguous() if need_u else None
    _lib.check(L.stmgcn_proj_bwd(s.data_ptr(), n * b * p, ks, n * b, p, _p(wt), q, act, out.data_ptr(), _p(d_out),
                                 _p(d_bcast), scale, b_inner, dz.data_ptr(), dw.data_ptr(), _p(db), _p(u),
                                 n * b * p, _stream()), "proj_bwd")
    return dw, db, u


def _proj_bwd_tc(s: torch.Tensor, w: torch.Tensor, wimg_t: torch.Tensor, act: int, out: torch.Tensor,
                 d_out: torch.Tensor, need_bias: bool):
    ks, n, b, _ = s.shape
    dw = torch.zeros_like(w, dtype=torch.float32)
    db = torch.zeros(64, device=s.device, dtype=torch.float32) if need_bias else None
    dz = torch.empty((n * b, 64), device=s.device, dtype=torch.float32)
    u = torch.empty_like(s)
    _lib.check(L.stmgcn_proj_bwd_tc(s.data_ptr(), n * b * 64, ks, n * b, wimg_t.data_ptr(), act, out.data_ptr(),
                                    d_out.data_ptr(), dz.data_ptr(), dw.data_ptr(), _p(db), u.data_ptr(), n * b * 64,
                                    _stream()), "proj_bwd_tc")
    return dw, db, u


# --------------------------------------------------------------------------------------------------
# autograd Functions
# --------------------------------------------------------------------------------------------------
def obs_to_node_major(obs: torch.Tensor):
    """obs (B,T,N,C) -> xo (N,B,T,C), xt (N,B,T).  Observations are data: no gradient flows back."""
    _require_cuda(obs)
    if obs.requires_grad:
        raise NotImplementedError("stmgcn_b200 treats obs_seq as data; gradients w.r.t. obs_seq are not provided")
    obs = _f32c(obs.detach())
    b, t, n, c = obs.shape
    xt = torch.empty((n, b, t), device=obs.device, dtype=torch.float32)
    xo = torch.empty((n, b, t, c), device=obs.device, dtype=torch.float32) if c > 1 else None
    _lib.check(L.stmgcn_obs_to_node_major(obs.data_ptr(), _p(xo), xt.data_ptr(), b, t, n, c, _stream()),
               "obs_to_node_major")
    return (xo if xo is not None else xt.view(n, b, t, 1)), xt


class ChebGCN(torch.autograd.Function):
    """out (N,B,q) = act( sum_k (T_k x) W_k + b ),  x (N,B,p) node-major."""

    @staticmethod
    def forward(ctx, x, w, bias, sset: SupportSet, act: int):
        _require_cuda(x, w)
        x, w = _f32c(x), _f32c(w)
        bias_c = _f32c(bias) if bias is not None else None
        # bf16-arithmetic mode: the spatial recurrence (F = B*64 features per node: the step's large gather volume) reads its
        # gathered operand from bf16 copies.  Not the temporal GCN (TemporalPool): its output feeds a global mean and the
        # two-layer gate, whose parameter gradients are small differences of large sums -- with bf16 gathers there they
        # moved by 2-3.6e-2 on the golden case (measured), past that mode's 2e-2 bar -- and its F = B*T rows are cheap.
        s = build_stack(sset, x, gather16=True)
        need_grad = any(ctx.needs_input_grad)
        img_b = None
        if _proj_tc(sset.ks, x.shape[2], w.shape[1]):
            img_f, img_b = _proj_images(w, sset.ks, need_grad)
            out = _proj_fwd_tc(s, img_f, bias_c, act)
        else:
            out = _proj_fwd(s, w, bias_c, act, None, x.shape[1])
        ctx.sset, ctx.act, ctx.has_bias = sset, act, bias is not None
        if need_grad:
            ctx.save_for_backward(s, w, out, img_b)
        return out

    @staticmethod
    def backward(ctx, d_out):
        s, w, out, img_b = ctx.saved_tensors
        need_dx = ctx.needs_input_grad[0]
        d_out = _f32c(d_out)
        if img_b is not None and need_dx and d_out.data_ptr() % 16 == 0:      # see _proj_tc
            dw, db, u = _proj_bwd_tc(s, w, img_b, ctx.act, out, d_out, ctx.has_bias)
        else:
            dw, db, u = _proj_bwd(s, w, ctx.act, out, d_out, None, 1.0, s.shape[2], ctx.has_bias, need_dx)
        dx = adjoint_stack_(ctx.sset, u) if need_dx else None
        return dx, dw, db, None, None


class TemporalPool(torch.autograd.Function):
    """pool (B,T) = sum_n ( x + act(GCN_T(x)) )[n,b,:]  (STMGCN.py:40-42 before the division by N).
    x is data (no gradient)."""

    @staticmethod
    def forward(ctx, x, w, bias, sset: SupportSet, act: int):
        _require_cuda(x, w)
        x, w = _f32c(x), _f32c(w)
        bias_c = _f32c(bias) if bias is not None else None
        n, b, t = x.shape
        if w.shape[1] != t:
            raise ValueError("temporal GCN must map seq_len -> seq_len")
        s = build_stack(sset, x)
        if sset.mode == "cheb":
            # s[0] IS x (T_0 = I): the kernel's fused pooling adds the residual from the stack's first segment
            pool = torch.zeros((b, t), device=x.device, dtype=torch.float32)
            out = _proj_fwd(s, w, bias_c, act, pool, b)
        else:
            # generic supports (localpool, hand-made stacks): s[0] = A_0 x is NOT the residual of STMGCN.py:41
            out = _proj_fwd(s, w, bias_c, act, None, b)
            pool = (x + out).sum(dim=0)
        ctx.act, ctx.has_bias = act, bias is not None
        if any(ctx.needs_input_grad):
            ctx.save_for_backward(s, w, out)
        return pool

    @staticmethod
    def backward(ctx, d_pool):
        s, w, out = ctx.saved_tensors
        d_pool = _f32c(d_pool)
        dw, db, _ = _proj_bwd(s, w, ctx.act, out, None, d_pool, 1.0, s.shape[2], ctx.has_bias, False)
        return None, dw, db, None, None


class ContextGate(torch.autograd.Function):
    """s = sigmoid(fc(relu(fc(pool / N))))  -- the same fc twice (STMGCN.py:43)."""

    @staticmethod
    def forward(ctx, pool, fcw, fcb, n_regions: int):
        _require_cuda(pool, fcw, fcb)
        pool, fcw, fcb = _f32c(pool), _f32c(fcw), _f32c(fcb)
        b, t = pool.shape
        z, a1, s = (torch.empty_like(pool) for _ in range(3))
        _lib.check(L.stmgcn_gate_fwd(pool.data_ptr(), b, t, n_regions, fcw.data_ptr(), fcb.data_ptr(),
                                     z.data_ptr(), a1.data_ptr(), s.data_ptr(), _stream()), "gate_fwd")
        ctx.n_regions = n_regions
        ctx.save_for_backward(z, a1, s, fcw)
        return s

    @staticmethod
    def backward(ctx, d_s):
        z, a1, s, fcw = ctx.saved_tensors
        d_s = _f32c(d_s)
        b, t = s.shape
        d_fcw = torch.zeros_like(fcw)
        d_fcb = torch.zeros(t, device=s.device, dtype=torch.float32)
        d_z = torch.empty_like(s)
        _lib.check(L.stmgcn_gate_bwd(d_s.data_ptr(), z.data_ptr(), a1.data_ptr(), s.data_ptr(), b, t,
                                     fcw.data_ptr(), d_fcw.data_ptr(), d_fcb.data_ptr(), d_z.data_ptr(),
                                     _stream()), "gate_bwd")
        return d_z / float(ctx.n_regions), d_fcw, d_fcb, None


def to_blocked(x: torch.Tensor) -> torch.Tensor:
    """(..., R, 64) row-major -> tile-blocked (..., ceil(R/128)*128, 64) flat layout [tile][unit/4][128][4]."""
    *lead, r, h = x.shape
    rp = ((r + 127) // 128) * 128
    if rp != r:
        pad = x.new_zeros(*lead, rp, h)
        pad[..., :r, :] = x
        x = pad
    return x.reshape(*lead, rp // 128, 128, 16, 4).transpose(-3, -2).contiguous().reshape(*lead, rp, h)


def from_blocked(x: torch.Tensor, rows: int) -> torch.Tensor:
    """Inverse of :func:`to_blocked`."""
    *lead, rp, h = x.shape
    return x.reshape(*lead, rp // 128, 16, 128, 4).transpose(-3, -2).reshape(*lead, rp, h)[..., :rows, :].contiguous()


def _pack_lstm(weights: Sequence[torch.Tensor], n_layers: int, hid: int):
    """nn.LSTM parameters -> packed operands (see include/stmgcn_b200.h)."""
    w_ih0 = weights[0]
    c_in = w_ih0.shape[1]
    wx = w_ih0.reshape(4, hid, c_in).permute(2, 1, 0).reshape(c_in, 4 * hid).contiguous()
    wp, bp, wpt = [], [], []
    for l in range(n_layers):
        w_ih, w_hh, b_ih, b_hh = weights[4 * l:4 * l + 4]
        cat = w_hh if l == 0 else torch.cat([w_ih, w_hh], dim=1)
        kd = cat.shape[1]
        packed = cat.reshape(4, hid, kd).permute(2, 1, 0).reshape(kd, 4 * hid).contiguous()
        wp.append(packed)
        wpt.append(packed.t().contiguous())
        bp.append((b_ih + b_hh).reshape(4, hid).t().reshape(4 * hid).contiguous())
    return wx, wp, bp, wpt


def _unpack_lstm_grads(dwx, dwp, dbp, n_layers: int, hid: int, c_in: int):
    grads = []
    for l in range(n_layers):
        kd = dwp[l].shape[0]
        full = dwp[l].reshape(kd, hid, 4).permute(2, 1, 0).reshape(4 * hid, kd)
        if l == 0:
            d_ih = dwx.reshape(c_in, hid, 4).permute(2, 1, 0).reshape(4 * hid, c_in).contiguous()
            d_hh = full.contiguous()
        else:
            d_ih, d_hh = full[:, :hid].contiguous(), full[:, hid:].contiguous()
        d_b = dbp[l].reshape(hid, 4).t().reshape(4 * hid).contiguous()
        grads += [d_ih, d_hh, d_b, d_b.clone()]
    return grads


# --------------------------------------------------------------------------------------------------
# bf16-plane LSTM path (H = 64): resident weight images cached per parameter version
# --------------------------------------------------------------------------------------------------
_PLANES = int(os.environ.get("STMGCN_LSTM_PLANES", "2"))     # 2: 3xBF16 (fp32-grade); 1: single-pass bf16 arithmetic


def lstm_planes() -> int:
    return _PLANES


def set_lstm_planes(planes: int) -> None:
    """2 = hi + lo bf16 planes, three tensor-core passes (fp32-grade, the 1e-4 parity mode);
    1 = hi plane only, one pass (the arithmetic of the bf16-quoted BASELINE configs)."""
    global _PLANES
    if planes not in (1, 2):
        raise ValueError(planes)
    _PLANES = planes


def _lstm16_images(weights: Sequence[torch.Tensor], n_layers: int, c_in: int):
    """Operand images of the shared LSTM's parameters for the bf16-plane kernels (stmgcn_lstm16_pack)."""

    def pack():
        dev = weights[0].device
        wimg = [torch.empty(65536 if l == 0 else 131072, dtype=torch.uint8, device=dev) for l in range(n_layers)]
        bias = [torch.empty(256, dtype=torch.float32, device=dev) for _ in range(n_layers)]
        wih_t = torch.empty(c_in * 256, dtype=torch.float32, device=dev)
        st = _stream()
        for l in range(n_layers):
            w_ih, w_hh, b_ih, b_hh = weights[4 * l:4 * l + 4]
            _lib.check(L.stmgcn_lstm16_pack(w_ih.data_ptr(), w_hh.data_ptr(), b_ih.data_ptr(), b_hh.data_ptr(), l, c_in,
                                            wimg[l].data_ptr(), bias[l].data_ptr(), wih_t.data_ptr() if l == 0 else None,
                                            st), "lstm16_pack")
        return dict(wimg=wimg, bias=bias, wih_t=wih_t, wimg_arr=_lib.ptr_array([v.data_ptr() for v in wimg]),
                    bias_arr=_lib.ptr_array([v.data_ptr() for v in bias]))

    return _cached_images(_LSTM16_IMAGES, weights, (c_in,), pack)


def to_planes(x: torch.Tensor, planes: int) -> torch.Tensor:
    """(..., R, 64) fp32 -> (..., planes, R, 64) bf16: hi = bf16(x), lo = bf16(x - hi)."""
    hi = x.to(torch.bfloat16)
    if planes == 1:
        return hi.unsqueeze(-3).contiguous()
    lo = (x - hi.float()).to(torch.bfloat16)
    return torch.stack([hi, lo], dim=-3).contiguous()


_ZERO_TILES: dict = {}


def _zero_tile(dev: torch.device) -> torch.Tensor:
    """16 KB of zeros per device: the h_prev operand tile at t = 0 without an initial state."""
    key = str(dev)
    if key not in _ZERO_TILES:
        _ZERO_TILES[key] = torch.zeros(128 * 64, device=dev, dtype=torch.bfloat16)
    return _ZERO_TILES[key]


def _lstm_inputs(xo, s_gate, h0, c0, weights):
    """The shared LSTM's inputs as the kernels of both families read them: CUDA, fp32, contiguous."""
    _require_cuda(xo, s_gate, *weights)
    return (_f32c(xo), _f32c(s_gate), _f32c(h0) if h0 is not None else None, _f32c(c0) if c0 is not None else None,
            [_f32c(w) for w in weights])


class SharedLSTM16(torch.autograd.Function):
    """:class:`SharedLSTM` on the tcgen05 bf16-plane kernels of lstm16.cu (H = 64, C <= 4, T <= 64), one library call
    per direction (stmgcn_lstm16_fwd / _bwd run the whole recurrence).  Tape: the hidden states as bf16 planes plus the
    cell state, no gate tape.  The backward recomputes the gates in fused launches (gate recompute + pointwise + data
    gradient + weight gradient), each covering one layer and a run of timesteps -- up to ceil(T / steps per launch) per
    layer, layers top-down -- then one reduction per layer."""

    @staticmethod
    def forward(ctx, xo, s_gate, h0, c0, n_layers: int, hid: int, want_state: bool, *weights):
        xo, s_gate, h0, c0, weights = _lstm_inputs(xo, s_gate, h0, c0, weights)
        n, b, t_len, c_in = xo.shape
        rows = n * b
        dev = xo.device
        rows_pad = ((rows + 127) // 128) * 128
        planes = lstm_planes()
        img = _lstm16_images(weights, n_layers, c_in)
        hp = torch.empty((n_layers, t_len, planes, rows, 64), device=dev, dtype=torch.bfloat16)
        cs = torch.empty((n_layers, t_len, rows_pad, 64), device=dev, dtype=torch.float32)
        h0p = to_planes(h0, planes) if h0 is not None else None        # (L, P, R, 64)
        c0b = to_blocked(c0) if c0 is not None else None
        if want_state:
            h_n = torch.empty((n_layers, rows, 64), device=dev, dtype=torch.float32)
            h_top = h_n[n_layers - 1]
        else:
            h_n = None
            h_top = torch.empty((rows, 64), device=dev, dtype=torch.float32)
        _lib.check(L.stmgcn_lstm16_fwd(t_len, n_layers, rows, c_in, b, planes, xo.data_ptr(), s_gate.data_ptr(),
                                       img["wimg_arr"], img["bias_arr"], img["wih_t"].data_ptr(), _p(h0p), _p(c0b),
                                       hp.data_ptr(), cs.data_ptr(), h_top.data_ptr(), _p(h_n), _stream()), "lstm16_fwd")
        if want_state:
            c_n = from_blocked(cs[:, t_len - 1], rows)
        else:
            h_n = c_n = torch.empty(0, device=dev, dtype=torch.float32)
        ctx.mark_non_differentiable(h_n, c_n)
        if any(ctx.needs_input_grad):
            ctx.n_layers, ctx.planes = n_layers, planes
            ctx.tape = dict(hp=hp, cs=cs, h0p=h0p, c0b=c0b, img=img)
            ctx.save_for_backward(xo, s_gate)
        return h_top.view(n, b, 64), h_n, c_n

    @staticmethod
    def backward(ctx, d_top, _dhn, _dcn):
        xo, s_gate = ctx.saved_tensors
        tape, n_layers, planes = ctx.tape, ctx.n_layers, ctx.planes
        n, b, t_len, c_in = xo.shape
        rows = n * b
        dev = xo.device
        rows_pad = ((rows + 127) // 128) * 128
        img = tape["img"]
        if "event" in img:                 # a cached entry (no event: packed inside the CUDA graph being captured)
            torch.cuda.current_stream().wait_event(img["event"])
        d_top_b = to_blocked(_f32c(d_top).view(rows, 64))
        dh_rec = torch.empty((rows_pad, 64), device=dev, dtype=torch.float32)
        dc = torch.empty((rows_pad, 64), device=dev, dtype=torch.float32)
        # the gradient a layer passes to the layer below, every timestep (two slices alternate down the stack)
        dx_work = (torch.empty((min(2, n_layers - 1), t_len, rows_pad, 64), device=dev, dtype=torch.float32)
                   if n_layers > 1 else None)
        d_s = torch.zeros((b, t_len), device=dev, dtype=torch.float32)
        dbp = torch.zeros((n_layers, 256), device=dev, dtype=torch.float32)
        scratch = torch.empty((n_layers, int(L.stmgcn_lstm16_grid(rows)), 128 * 256), device=dev, dtype=torch.float32)
        w_grads = []
        for l in range(n_layers):
            in_l = c_in if l == 0 else 64
            w_grads += [torch.empty((256, in_l), device=dev, dtype=torch.float32),
                        torch.empty((256, 64), device=dev, dtype=torch.float32),
                        torch.empty(256, device=dev, dtype=torch.float32), torch.empty(256, device=dev, dtype=torch.float32)]
        _lib.check(L.stmgcn_lstm16_bwd(t_len, n_layers, rows, c_in, b, planes, xo.data_ptr(), s_gate.data_ptr(),
                                       img["wimg_arr"], img["bias_arr"], img["wih_t"].data_ptr(), _p(tape["h0p"]),
                                       _p(tape["c0b"]), tape["hp"].data_ptr(), tape["cs"].data_ptr(), d_top_b.data_ptr(),
                                       dh_rec.data_ptr(), dc.data_ptr(), _p(dx_work), d_s.data_ptr(), dbp.data_ptr(),
                                       scratch.data_ptr(), _zero_tile(dev).data_ptr(),
                                       _lib.ptr_array([g.data_ptr() for g in w_grads]), _stream()), "lstm16_bwd")
        return (None, d_s, None, None, None, None, None, *w_grads)


class SharedLSTMExact(torch.autograd.Function):
    """:class:`SharedLSTM` on the exact-fp32 CUDA-core kernels of lstm.cu (any H <= 128), one library call per direction
    (stmgcn_lstm_fwd / _bwd).  Tape: hs, cs and the post-activation gates; the backward overwrites the gate tape in
    place, so it can run only once per forward."""

    @staticmethod
    def forward(ctx, xo, s_gate, h0, c0, n_layers: int, hid: int, want_state: bool, *weights):
        xo, s_gate, h0, c0, weights = _lstm_inputs(xo, s_gate, h0, c0, weights)
        n, b, t_len, c_in = xo.shape
        rows = n * b
        dev = xo.device
        need_grad = any(ctx.needs_input_grad)
        wx, wp, bp, wpt = _pack_lstm(weights, n_layers, hid)
        hs = torch.empty((n_layers, t_len, rows, hid), device=dev, dtype=torch.float32)
        cs = torch.empty((n_layers, t_len, rows, hid), device=dev, dtype=torch.float32)
        gates = torch.empty((n_layers, t_len, rows, 4 * hid), device=dev, dtype=torch.float32) if need_grad else None
        wp_arr, bp_arr = _lib.ptr_array([w.data_ptr() for w in wp]), _lib.ptr_array([v.data_ptr() for v in bp])
        _lib.check(L.stmgcn_lstm_fwd(t_len, n_layers, rows, hid, c_in, b, xo.data_ptr(), s_gate.data_ptr(), wx.data_ptr(),
                                     wp_arr, bp_arr, _p(h0), _p(c0), hs.data_ptr(), cs.data_ptr(), _p(gates), _stream()),
                   "lstm_fwd")
        if need_grad:
            ctx.dims = (n, b, t_len, c_in, n_layers, hid)
            ctx.save_for_backward(xo, s_gate, h0, c0, hs, cs, gates, wx, *wpt)
        h_top = hs[n_layers - 1, t_len - 1].view(n, b, hid)
        if want_state:
            h_n, c_n = hs[:, t_len - 1], cs[:, t_len - 1]
        else:                       # ST_MGCN discards the final state (STMGCN.py:113)
            h_n = c_n = hs.new_empty(0)
        ctx.mark_non_differentiable(h_n, c_n)
        return h_top, h_n, c_n

    @staticmethod
    def backward(ctx, d_top, _dhn, _dcn):
        if getattr(ctx, "tape_consumed", False):
            raise RuntimeError("SharedLSTM (exact-fp32 kernels): the gate tape was overwritten in place by the first backward "
                               "pass; a second backward over the same graph is not supported on this path")
        ctx.tape_consumed = True
        n, b, t_len, c_in, n_layers, hid = ctx.dims
        xo, s_gate, h0, c0, hs, cs, gates, wx, *wpt = ctx.saved_tensors
        rows = n * b
        dev = xo.device
        d_top = _f32c(d_top).view(rows, hid)
        # dh_rec / dc need no initialisation: the step at t = T-1 treats them as zero (stmgcn_lstm_bwd)
        dh_rec = torch.empty((n_layers, rows, hid), device=dev, dtype=torch.float32)
        dc = torch.empty((n_layers, rows, hid), device=dev, dtype=torch.float32)
        dx_work = torch.empty((rows, hid), device=dev, dtype=torch.float32)
        d_s = torch.zeros((b, t_len), device=dev, dtype=torch.float32)
        dwx = torch.zeros_like(wx)
        dbp = [torch.zeros(4 * hid, device=dev, dtype=torch.float32) for _ in range(n_layers)]
        dwp = [torch.zeros((w.shape[1], 4 * hid), device=dev, dtype=torch.float32) for w in wpt]
        wpt_arr, dbp_arr, dwp_arr = (_lib.ptr_array([v.data_ptr() for v in ts]) for ts in (wpt, dbp, dwp))
        # NOTE: gates is overwritten in place with dA (the tape is consumed; see the guard above)
        _lib.check(L.stmgcn_lstm_bwd(t_len, n_layers, rows, hid, c_in, b, xo.data_ptr(), s_gate.data_ptr(), wx.data_ptr(),
                                     wpt_arr, _p(h0), _p(c0), hs.data_ptr(), cs.data_ptr(), gates.data_ptr(),
                                     d_top.data_ptr(), dh_rec.data_ptr(), dc.data_ptr(), dx_work.data_ptr(), d_s.data_ptr(),
                                     dwx.data_ptr(), dbp_arr, dwp_arr, _stream()), "lstm_bwd")
        w_grads = _unpack_lstm_grads(dwx, dwp, dbp, n_layers, hid, c_in)
        return (None, d_s, None, None, None, None, None, *w_grads)


class SharedLSTM:
    """h_top (N,B,H) of the shared multi-layer LSTM over rows r = n*B + b; input ``xo * s[b,t]``.

    apply(xo (N,B,T,C), s (B,T), h0|None, c0|None (L,R,H), n_layers, hid, want_state, *lstm_weights) where
    lstm_weights = [w_ih_l0, w_hh_l0, b_ih_l0, b_hh_l0, w_ih_l1, ...] (nn.LSTM names/shapes).
    Returns (h_top, h_n (L,R,H), c_n (L,R,H)); the last two are not differentiable.

    Picks one of two kernel families (include/stmgcn_b200.h), each its own autograd Function:
    * H = 64, C <= 4, T <= 64 (the reference's configuration, Main.py:62) and ``lstm_path() == "tc"``:
      :class:`SharedLSTM16`, the tcgen05 bf16-plane kernels;
    * anything else, or ``lstm_path() == "fma"``: :class:`SharedLSTMExact`, the exact-fp32 CUDA-core kernels.
    """

    @staticmethod
    def apply(xo, s_gate, h0, c0, n_layers: int, hid: int, want_state: bool, *weights):
        _, _, t_len, c_in = xo.shape
        fn = SharedLSTM16 if hid == 64 and lstm_path() == "tc" and c_in <= 4 and t_len <= 64 else SharedLSTMExact
        return fn.apply(xo, s_gate, h0, c0, n_layers, hid, want_state, *weights)


class FuseOut(torch.autograd.Function):
    """y (B,N,C) = fc( sum_m g_m ),  g_m (N,B,G) node-major  (STMGCN.py:116-118)."""

    @staticmethod
    def forward(ctx, fcw, fcb, *gs):
        _require_cuda(fcw, fcb, *gs)
        fcw, fcb = _f32c(fcw), _f32c(fcb)
        gs = [_f32c(g) for g in gs]
        n, b, gdim = gs[0].shape
        c = fcw.shape[0]
        feat = torch.empty_like(gs[0])
        y = torch.empty((b, n, c), device=feat.device, dtype=torch.float32)
        arr = _lib.ptr_array([g.data_ptr() for g in gs])
        _lib.check(L.stmgcn_fuse_out_fwd(arr, len(gs), n, b, gdim, c, fcw.data_ptr(), fcb.data_ptr(),
                                         feat.data_ptr(), y.data_ptr(), _stream()), "fuse_out_fwd")
        ctx.m = len(gs)
        ctx.save_for_backward(feat, fcw)
        return y

    @staticmethod
    def backward(ctx, d_y):
        feat, fcw = ctx.saved_tensors
        d_y = _f32c(d_y)
        n, b, gdim = feat.shape
        c = fcw.shape[0]
        d_feat = torch.empty_like(feat)
        d_fcw = torch.zeros_like(fcw)
        d_fcb = torch.zeros(c, device=feat.device, dtype=torch.float32)
        _lib.check(L.stmgcn_fuse_out_bwd(d_y.data_ptr(), feat.data_ptr(), n, b, gdim, c, fcw.data_ptr(),
                                         d_feat.data_ptr(), d_fcw.data_ptr(), d_fcb.data_ptr(), _stream()),
                   "fuse_out_bwd")
        return (d_fcw, d_fcb) + tuple(d_feat for _ in range(ctx.m))
