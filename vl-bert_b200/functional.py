"""torch.autograd front ends of the C ABI (include/vlbert_b200.h).

PyTorch is used here only for device memory, streams and autograd bookkeeping; every FLOP of the
hot path runs in libvlbert_b200.so.  All calls enqueue on torch's current CUDA stream.
"""
import ctypes

import os

import torch

from . import _lib

BF16 = torch.bfloat16
F32 = torch.float32


def _p(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _chk(rc):
    if rc != 0:
        _lib.check(rc)


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("vlbert_b200 has no CPU path: expected CUDA tensors (got %s)" % t.device)


def _require_param(t, name, device):
    """Parameters reach the C ABI as raw pointers: the kernels assume contiguous fp32 on the input's device.  A model converted
    with .half() / .bfloat16() / apex amp O2 must be rejected here instead of being reinterpreted (the reference's FP16 cfgs
    rely on amp; this library keeps fp32 master weights and computes its GEMMs in bf16 itself)."""
    if t is None:
        return
    if t.dtype != F32 or not t.is_contiguous() or t.device != device:
        raise RuntimeError("vlbert_b200: parameter %s must be a contiguous float32 tensor on %s (got %s, %s, contiguous=%s); "
                           "half / bfloat16 / amp-O2 converted models are not supported" %
                           (name, device, t.dtype, t.device, t.is_contiguous()))


def _align(n, a=256):
    return (n + a - 1) // a * a


class _Carver(object):
    """Carves typed sub-tensors out of one flat uint8 allocation (256-byte aligned)."""

    def __init__(self, specs, device):
        self.offsets = {}
        off = 0
        for name, shape, dtype in specs:
            n = 1
            for s in shape:
                n *= s
            self.offsets[name] = (off, shape, dtype, n)
            off += _align(n * torch.empty((), dtype=dtype).element_size())
        self.nbytes = off
        self.buf = torch.empty(max(off, 256), dtype=torch.uint8, device=device)
        self.base = self.buf.data_ptr()

    def ptr(self, name):
        """device pointer of a carved region (no tensor view is created: the hot loops only need addresses)"""
        return self.base + self.offsets[name][0]

    def get(self, name):
        off, shape, dtype, n = self.offsets[name]
        esz = torch.empty((), dtype=dtype).element_size()
        return self.buf[off: off + n * esz].view(dtype).view(*shape)


class DropSite(object):
    """One dropout call site (VlbDropout): probability, site id and the DEVICE rng state tensor (int64 [2] = seed, step).
    The kernels read (seed, step) when they run, so the same object serves the forward, its backward and CUDA-graph replays."""

    __slots__ = ("p", "site", "rng", "_struct", "bits", "_bits_shape")

    def __init__(self, p, site, rng):
        if not (0.0 <= p < 1.0):
            raise ValueError("dropout probability has to be in [0, 1), got %r" % (p,))
        if not (rng.is_cuda and rng.dtype == torch.int64 and rng.numel() >= 2 and rng.is_contiguous()):
            raise RuntimeError("vlbert_b200: the dropout rng state must be a contiguous CUDA int64 tensor (seed, step)")
        self.p, self.site, self.rng = float(p), int(site), rng
        d = _lib.Dropout()
        d.p, d.site, d.rng, d.keep_bits = self.p, self.site, rng.data_ptr(), None
        self._struct = d
        self.bits = None
        self._bits_shape = None

    def ref(self):
        return ctypes.byref(self._struct)

    def with_bits(self, rows, cols):
        """Generate (vlb_dropout_bits) the keep flags of this site for a [rows, cols] mask with the CURRENT device (seed, step)
        and attach them: the attention / GEMM-epilogue / LayerNorm-backward consumers read flags, they do not run Philox.
        Returns self.  The backward of an op must be given the same object (same flags) as its forward."""
        if self.p == 0.0:
            return self
        lib = _lib.lib()
        n = int(lib.vlb_dropout_bits_words(rows, cols))
        self.bits = torch.empty((max(n, 1),), dtype=torch.int32, device=self.rng.device)
        self._struct.keep_bits = None
        _chk(lib.vlb_dropout_bits(self.bits.data_ptr(), rows, cols, self.ref(), _stream()))
        self._struct.keep_bits = self.bits.data_ptr()
        self._bits_shape = (rows, cols)
        return self

    def need_bits(self, rows, cols):
        if self.p > 0.0 and self._bits_shape != (rows, cols):
            self.with_bits(rows, cols)
        return self


def _dref(drop):
    return None if drop is None or drop.p == 0.0 else drop.ref()


def dropout_2d(x, drop, col_offset=0, total_cols=None):
    """y = x * keep / (1-p) for a 2-D window x [rows, cols] of a tensor whose mask is indexed over [rows, total_cols]."""
    _require_cuda(x)
    assert x.dim() == 2 and x.stride(1) == 1
    y = torch.empty_like(x, memory_format=torch.contiguous_format)
    total = x.shape[1] if total_cols is None else total_cols
    _chk(_lib.lib().vlb_dropout_2d(_p(x), x.stride(0), _p(y), y.stride(0), x.shape[0], x.shape[1], col_offset, total,
                                   int(x.dtype == BF16), _dref(drop), _stream()))
    return y


# ------------------------------------------------------------------------------------------------
# primitive wrappers (used by tests and by the composites below)
# ------------------------------------------------------------------------------------------------
def gemm(mode, A, B, out, bias=None, resid=None, act=0, aux=None, alpha=1.0, split_k=1, force_bn=0, M=None, N=None, K=None,
         drop=None):
    """See vlb_gemm_bf16.  A/B bf16 2-D (row-major, last dim contiguous); out bf16 or f32 2-D.
    drop: DropSite applied after bias/activation and before the residual add (vlb_gemm_bf16_dropout)."""
    _require_cuda(A, B, out)
    if mode == 0:
        m, k = A.shape; n = B.shape[0]
    elif mode == 1:
        m, k = A.shape; n = B.shape[1]
    else:
        k, m = A.shape; n = B.shape[1]
    M, N, K = M or m, N or n, K or k
    out_kind = 0 if out.dtype == BF16 else (2 if split_k > 1 or getattr(out, "_vlb_accumulate", False) else 1)
    resid_kind = 0 if resid is None else (1 if resid.dtype == BF16 else 2)
    if drop is not None:
        drop.need_bits(M, N)
        _chk(_lib.lib().vlb_gemm_bf16_dropout(mode, M, N, K, _p(A), A.stride(0), _p(B), B.stride(0), _p(out), out.stride(0),
                                              out_kind, _p(bias), _p(resid), resid.stride(0) if resid is not None else 0,
                                              resid_kind, act, _p(aux), aux.stride(0) if aux is not None else 0, float(alpha),
                                              split_k, force_bn, _dref(drop), _stream()))
        return out
    _chk(_lib.lib().vlb_gemm_bf16(mode, M, N, K, _p(A), A.stride(0), _p(B), B.stride(0), _p(out), out.stride(0), out_kind,
                                  _p(bias), _p(resid), resid.stride(0) if resid is not None else 0, resid_kind, act,
                                  _p(aux), aux.stride(0) if aux is not None else 0, float(alpha), split_k, force_bn, _stream()))
    return out


def gemm_bias_residual_f32(A, W, bias, resid32, ln=None, drop=None, force_bn=0):
    """out f32 [M,N] = dropout(A W^T + bias) + R with R = resid32 (fp32 [M,N]) or, when ln = (mean, rstd, gamma, beta),
    R = LayerNorm(resid32) recomputed in the epilogue (vlb_gemm_bias_residual_f32)."""
    _require_cuda(A, W, resid32)
    M, K = A.shape
    N = W.shape[0]
    out = torch.empty((M, N), dtype=F32, device=A.device)
    r = _lib.Residual()
    r.x_f32 = resid32.data_ptr()
    assert resid32.is_contiguous() and resid32.shape == (M, N)
    if ln is not None:
        r.mean, r.rstd, r.gamma, r.beta = [t.data_ptr() for t in ln]
    if drop is not None:
        drop.need_bits(M, N)
    _chk(_lib.lib().vlb_gemm_bias_residual_f32(M, N, K, _p(A), A.stride(0), _p(W), W.stride(0), _p(out), N, _p(bias), ctypes.byref(r),
                                               _dref(drop), force_bn, _stream()))
    return out


def layernorm_forward(x, gamma, beta, eps=1e-12, want_bf16=True, want_f32=False, ldx=None, H=None, drop=None):
    M = x.numel() // x.shape[-1] if ldx is None else x.shape[0]
    H = H or x.shape[-1]
    ldx = ldx or H
    dev = x.device
    y16 = torch.empty((M, H), dtype=BF16, device=dev) if want_bf16 else None
    y32 = torch.empty((M, H), dtype=F32, device=dev) if want_f32 else None
    mean = torch.empty((M,), dtype=F32, device=dev)
    rstd = torch.empty((M,), dtype=F32, device=dev)
    _chk(_lib.lib().vlb_layernorm_forward_dropout(_p(x), ldx, _p(gamma), _p(beta), _p(y16), _p(y32), _p(mean), _p(rstd), M, H,
                                                  float(eps), _dref(drop), _stream()))
    return y16, y32, mean, rstd


def layernorm_backward(dy16, dy32, x, mean, rstd, gamma, dgamma, dbeta, dcolsum=None, want_bf16=True, want_f32=False,
                       ldx=None, H=None, dx32=None, ld_dx=None, in_drop=None, out_drop=None):
    """out_drop: additionally returns dx * keep / (1-p) (bf16) as a third value and makes dcolsum sum that tensor."""
    H = H or x.shape[-1]
    M = mean.numel()
    ldx = ldx or H
    dev = x.device
    dx16 = torch.empty((M, H), dtype=BF16, device=dev) if want_bf16 else None
    if want_f32 and dx32 is None:
        dx32 = torch.empty((M, H), dtype=F32, device=dev)
        ld_dx = H
    dx16_drop = torch.empty((M, H), dtype=BF16, device=dev) if out_drop is not None else None
    if out_drop is not None:
        out_drop.need_bits(M, H)
    _chk(_lib.lib().vlb_layernorm_backward_dropout(_p(dy16), _p(dy32), _p(x), ldx, _p(mean), _p(rstd), _p(gamma), _p(dx16),
                                                   _p(dx32), ld_dx or 0, _p(dgamma), _p(dbeta), _p(dcolsum), M, H, _dref(in_drop),
                                                   _p(dx16_drop), _dref(out_drop), _stream()))
    if out_drop is not None:
        return dx16, dx32, dx16_drop
    return dx16, dx32


def mhsa_forward(qkv, add_mask, B, S, H, heads, drop=None):
    """drop: DropSite; its keep flags for the [B*heads*S, S] probability mask are generated here (and must be re-used by the
    backward: pass the same object to mhsa_backward)."""
    if drop is not None:
        drop.with_bits(B * heads * S, S)
    ctx = torch.empty((B * S, H), dtype=BF16, device=qkv.device)
    lse = torch.empty((B, heads, S), dtype=F32, device=qkv.device)
    _chk(_lib.lib().vlb_mhsa_forward_dropout(_p(qkv), _p(add_mask), _p(ctx), _p(lse), B, S, H, heads, _dref(drop), _stream()))
    return ctx, lse


def mhsa_backward(qkv, add_mask, ctx, lse, dctx, B, S, H, heads, drop=None, dbias=None):
    """dbias: optional f32 [3H], += column sums of dqkv (fused bias gradients)"""
    if drop is not None:
        drop.need_bits(B * heads * S, S)
    dqkv = torch.empty((B * S, 3 * H), dtype=BF16, device=qkv.device)
    scratch = torch.empty((B * S, 3 * H), dtype=F32, device=qkv.device) if S > 128 else None
    _chk(_lib.lib().vlb_mhsa_backward_dropout(_p(qkv), _p(add_mask), _p(ctx), _p(lse), _p(dctx), _p(dqkv), _p(scratch), B, S, H,
                                              heads, _p(dbias), _dref(drop), _stream()))
    return dqkv


def gather_rows(src2d, idx, n_out, out_dtype=F32):
    H = src2d.shape[1]
    out = torch.empty((n_out, H), dtype=out_dtype, device=src2d.device)
    _chk(_lib.lib().vlb_gather_rows(_p(src2d), int(src2d.dtype == BF16), src2d.stride(0), _p(idx), _p(out),
                                    int(out_dtype == BF16), H, n_out, H, _stream()))
    return out


def scatter_rows_add(src2d, idx, out2d):
    H = src2d.shape[1]
    _chk(_lib.lib().vlb_scatter_rows_add(_p(src2d), int(src2d.dtype == BF16), src2d.stride(0), _p(idx), _p(out2d),
                                         out2d.stride(0), src2d.shape[0], H, _stream()))
    return out2d


# ------------------------------------------------------------------------------------------------
# weights: fp32 master parameters -> bf16 GEMM operands (one launch for the whole encoder)
# ------------------------------------------------------------------------------------------------
class EncoderWeights(object):
    """Persistent bf16 operand copies of L BertLayers + the device descriptor table of the cast."""

    PER_LAYER = ("query.w", "query.b", "key.w", "key.b", "value.w", "value.b", "o.w", "o.b", "ln1.w", "ln1.b",
                 "i.w", "i.b", "out.w", "out.b", "ln2.w", "ln2.b")

    def __init__(self, L, H, I, device):
        self.L, self.H, self.I = L, H, I
        self.w_qkv = torch.empty((L, 3 * H, H), dtype=BF16, device=device)
        self.w_o = torch.empty((L, H, H), dtype=BF16, device=device)
        self.w_1 = torch.empty((L, I, H), dtype=BF16, device=device)
        self.w_2 = torch.empty((L, H, I), dtype=BF16, device=device)
        self.b_qkv = torch.empty((L, 3 * H), dtype=F32, device=device)
        self._key = None
        self._table = None
        self._count = 0

    def refresh(self, params):
        """params: flat list, 16 tensors per layer in PER_LAYER order (fp32, contiguous)."""
        L, H = self.L, self.H
        key = tuple(p.data_ptr() for p in params)
        if key != self._key:
            descs = []
            for l in range(L):
                q = params[16 * l: 16 * l + 16]
                for j, (w, b) in enumerate(((q[0], q[1]), (q[2], q[3]), (q[4], q[5]))):
                    descs.append((w.data_ptr(), self.w_qkv[l, j * H].data_ptr(), H * H, 1))
                    descs.append((b.data_ptr(), self.b_qkv[l, j * H:].data_ptr(), H, 0))
                descs.append((q[6].data_ptr(), self.w_o[l].data_ptr(), H * H, 1))
                descs.append((q[10].data_ptr(), self.w_1[l].data_ptr(), self.I * H, 1))
                descs.append((q[12].data_ptr(), self.w_2[l].data_ptr(), H * self.I, 1))
            arr = (_lib.CastDesc * len(descs))()
            for i, (s, d, n, k) in enumerate(descs):
                arr[i].src, arr[i].dst, arr[i].n, arr[i].dst_is_bf16 = s, d, n, k
            host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)
            self._table = host.to(self.w_qkv.device)
            self._count = len(descs)
            self._key = key
        _chk(_lib.lib().vlb_multi_cast(_p(self._table), self._count, 24, _stream()))

    def layer_struct(self, l, params):
        cache = getattr(self, "_structs", None)
        if cache is not None and cache[0] == self._key:
            return cache[1][l]
        structs = [self._layer_struct(i, params) for i in range(self.L)]
        self._structs = (self._key, structs)
        return structs[l]

    def _layer_struct(self, l, params):
        q = params[16 * l: 16 * l + 16]
        w = _lib.LayerWeights()
        w.w_qkv, w.b_qkv = self.w_qkv[l].data_ptr(), self.b_qkv[l].data_ptr()
        w.w_o, w.b_o = self.w_o[l].data_ptr(), q[7].data_ptr()
        w.ln1_g, w.ln1_b = q[8].data_ptr(), q[9].data_ptr()
        w.w_1, w.b_1 = self.w_1[l].data_ptr(), q[11].data_ptr()
        w.w_2, w.b_2 = self.w_2[l].data_ptr(), q[13].data_ptr()
        w.ln2_g, w.ln2_b = q[14].data_ptr(), q[15].data_ptr()
        return w


def _act_specs(l, B, S, H, heads, I, want_f32, drop=False):
    M = B * S
    sp = []
    if drop:
        i32 = torch.int32
        sp = [("ka%d" % l, (B * heads * S, (S + 31) // 32), i32), ("ks%d" % l, (M, (H + 31) // 32), i32), ("ko%d" % l, (M, (H + 31) // 32), i32)]
    sp += [("qkv%d" % l, (M, 3 * H), BF16), ("ctx%d" % l, (M, H), BF16), ("lse%d" % l, (B, heads, S), F32),
          ("a%d" % l, (M, H), F32), ("m1_%d" % l, (M,), F32), ("r1_%d" % l, (M,), F32), ("h%d" % l, (M, H), BF16),
          ("z%d" % l, (M, I), BF16), ("u%d" % l, (M, I), BF16), ("y0_%d" % l, (M, H), F32), ("m2_%d" % l, (M,), F32),
          ("r2_%d" % l, (M,), F32), ("y%d" % l, (M, H), BF16)]
    return sp


def _acts_struct(car, l, y_f32, drop=False):
    a = _lib.LayerActs()
    g = lambda n: car.ptr(n % l)  # noqa: E731
    if drop:
        a.keep_attn, a.keep_self_out, a.keep_out = g("ka%d"), g("ks%d"), g("ko%d")
    a.qkv, a.ctx, a.lse, a.a = g("qkv%d"), g("ctx%d"), g("lse%d"), g("a%d")
    a.ln1_mean, a.ln1_rstd, a.h, a.z, a.u = g("m1_%d"), g("r1_%d"), g("h%d"), g("z%d"), g("u%d")
    a.y0, a.ln2_mean, a.ln2_rstd, a.y = g("y0_%d"), g("m2_%d"), g("r2_%d"), g("y%d")
    a.y_f32 = None if y_f32 is None else y_f32.data_ptr()
    return a


_SIDE_STREAM_BITS = os.environ.get("VLB_BITS_SIDE_STREAM", "1") != "0"
_SIDE_STREAMS = {}


_ZERO_GRADS_IN_FORWARD = os.environ.get("VLB_ZERO_GRADS_IN_FORWARD", "1") != "0"
_CAPTURE_HAS_BACKWARD = False     # set by graphs.GraphedStep while it captures forward + backward into one graph


def _side_stream(device):
    key = (device.type, device.index)
    s = _SIDE_STREAMS.get(key)
    if s is None:
        s = torch.cuda.Stream(device=device)
        _SIDE_STREAMS[key] = s
    return s


def _layer_drop_structs(drop, L):
    """drop: None (eval / p = 0) or an object with p_attn, p_hidden, rng (int64 CUDA tensor: seed, step).  Returns one
    ctypes reference (or None) per layer; sites follow the contract: 1+3l attention, 2+3l self-output, 3+3l output."""
    if drop is None or (drop.p_attn == 0.0 and drop.p_hidden == 0.0):
        return [None] * L
    rng = drop.rng
    if not (rng.is_cuda and rng.dtype == torch.int64 and rng.numel() >= 2 and rng.is_contiguous()):
        raise RuntimeError("vlbert_b200: the dropout rng state must be a contiguous CUDA int64 tensor (seed, step)")
    out = []
    for l in range(L):
        d = _lib.LayerDropout()
        d.p_attn, d.p_hidden = float(drop.p_attn), float(drop.p_hidden)
        d.site_attn, d.site_self_out, d.site_out = 1 + 3 * l, 2 + 3 * l, 3 + 3 * l
        d.rng = rng.data_ptr()
        d.keep_bits_ready = 0
        out.append(d)
    refs = [ctypes.byref(d) for d in out]
    refs.append(out)   # keep the structs alive as long as the reference list is
    return refs


class EncoderFn(torch.autograd.Function):
    """L BertLayers (BertEncoder.forward, modeling.py:406-421) on vlb_bert_layer_forward/backward.

    forward(emb_bf16 [B,S,H], emb_f32 [B,S,H] or None, add_mask f32 [B,S], meta, *params) -> tuple of fp32 [B,S,H] outputs, one
    per requested layer (all layers when meta.all_layers else the last one only).  emb_f32 (the same embedding in fp32)
    selects the fp32 residual stream (csrc/encoder.cu); the gradient then comes back split the same way: the bf16 GEMM part
    for emb_bf16 and the fp32 residual part for emb_f32."""

    @staticmethod
    def forward(ctx, emb, emb32, add_mask, meta, *params):
        _require_cuda(emb, add_mask)
        B, S, H = emb.shape
        L, heads, I = meta.L, meta.heads, meta.I
        lib = _lib.lib()
        st = _stream()
        if emb.dtype != BF16:
            raise RuntimeError("vlbert_b200: EncoderFn expects the bf16 embedding produced by EmbeddingFn (got %s)" % emb.dtype)
        if getattr(meta.weights, "_checked", None) != tuple(p.data_ptr() for p in params):
            for i, p in enumerate(params):
                _require_param(p, "encoder.layer.%d.%s" % (i // 16, EncoderWeights.PER_LAYER[i % 16]), emb.device)
            meta.weights._checked = tuple(p.data_ptr() for p in params)
        emb = emb.contiguous()          # kept alive in ctx: the layer-0 kernels and the backward read this very buffer
        if emb32 is not None:
            if emb32.dtype != F32 or emb32.shape != emb.shape:
                raise RuntimeError("vlbert_b200: EncoderFn expects emb_f32 as a float32 tensor of the embedding's shape")
            emb32 = emb32.contiguous()
        add_mask = add_mask.contiguous()
        meta.weights.refresh(params)
        drops = _layer_drop_structs(getattr(meta, "drop", None), L)
        has_drop = drops[0] is not None
        specs = []
        for l in range(L):
            specs += _act_specs(l, B, S, H, heads, I, False, has_drop)
        car = _Carver(specs, emb.device)
        outs = []
        x_ptr = emb.data_ptr()
        resid = None
        if emb32 is not None:           # layer 0: the embedding itself in fp32
            resid = _lib.Residual()
            resid.x_f32 = emb32.data_ptr()
        bits_ready = None
        if has_drop and _SIDE_STREAM_BITS:
            # The keep flags of every layer are generated up front on a side stream: ten Philox rounds per four elements are
            # instruction-bound work that overlaps the tensor-bound kernels of the earlier layers instead of sitting at the head
            # of each layer's dependency chain.  Layer l waits for its own event only.
            cur = torch.cuda.current_stream()
            side = _side_stream(emb.device)
            side.wait_stream(cur)                     # (seed, step) snapshot and the activation buffer are ordered before
            car.buf.record_stream(side)
            bits_ready = []
            structs = drops[L]
            with torch.cuda.stream(side):
                for l in range(L):
                    a = _acts_struct(car, l, None, True)
                    _chk(lib.vlb_layer_dropout_bits(ctypes.byref(a), B, S, H, heads, drops[l], side.cuda_stream))
                    structs[l].keep_bits_ready = 1
                    ev = torch.cuda.Event()
                    ev.record(side)
                    bits_ready.append(ev)
        # The flat fp32 gradient buffer of the backward (the weight-gradient GEMMs accumulate into it with split-K atomics, so it
        # must start at zero: 340 MB at config 2) is allocated and cleared here, on the side stream, under the forward's
        # tensor-bound kernels, instead of at the head of the backward's dependency chain.  Inside a stream capture this is done
        # only when the capture is known to contain the backward too (GraphedStep sets the flag): the fork is joined there.
        ctx.flat, ctx.flat_ready = None, None
        if _ZERO_GRADS_IN_FORWARD and any(ctx.needs_input_grad) and (_CAPTURE_HAS_BACKWARD or not torch.cuda.is_current_stream_capturing()):
            cur = torch.cuda.current_stream()
            side = _side_stream(emb.device)
            side.wait_stream(cur)
            per = 3 * H * H + 3 * H + H * H + H + 2 * H + I * H + I + H * I + H + 2 * H
            with torch.cuda.stream(side):
                ctx.flat = torch.zeros((L, per), dtype=F32, device=emb.device)
                ctx.flat_ready = torch.cuda.Event()
                ctx.flat_ready.record(side)
            ctx.flat.record_stream(cur)
        for l in range(L):
            want = meta.all_layers or l == L - 1
            y32 = torch.empty((B, S, H), dtype=F32, device=emb.device) if want else None
            w = meta.weights.layer_struct(l, params)
            a = _acts_struct(car, l, y32, has_drop)
            if bits_ready is not None:
                torch.cuda.current_stream().wait_event(bits_ready[l])
            _chk(lib.vlb_bert_layer_forward(ctypes.byref(w), x_ptr, None if resid is None else ctypes.byref(resid), _p(add_mask),
                                            ctypes.byref(a), B, S, H, heads, I, float(meta.eps), drops[l], st))
            x_ptr = car.ptr("y%d" % l)
            if emb32 is not None:       # next layer's residual = this layer's LayerNorm-2 output, recomputed from y0 + statistics
                resid = _lib.Residual()
                resid.x_f32, resid.mean, resid.rstd = car.ptr("y0_%d" % l), car.ptr("m2_%d" % l), car.ptr("r2_%d" % l)
                resid.gamma, resid.beta = params[16 * l + 14].data_ptr(), params[16 * l + 15].data_ptr()
            if want:
                outs.append(y32)
        ctx.meta = meta
        ctx.car = car
        ctx.dims = (B, S, H)
        ctx.drops = drops
        ctx.drop_rng = None if getattr(meta, "drop", None) is None else meta.drop.rng   # keeps the state tensor alive
        ctx.has_drop = has_drop
        ctx.f32_stream = emb32 is not None
        ctx.emb = emb
        ctx.add_mask = add_mask
        ctx.params = params
        return tuple(outs)

    @staticmethod
    def backward(ctx, *grad_outs):
        meta, car = ctx.meta, ctx.car
        B, S, H = ctx.dims
        L, heads, I = meta.L, meta.heads, meta.I
        M = B * S
        lib = _lib.lib()
        st = _stream()
        dev = ctx.emb.device
        params = ctx.params
        per = 3 * H * H + 3 * H + H * H + H + 2 * H + I * H + I + H * I + H + 2 * H
        if ctx.flat is not None:            # cleared under the forward (see there); a second backward gets a fresh buffer
            torch.cuda.current_stream().wait_event(ctx.flat_ready)
            flat, ctx.flat = ctx.flat, None
        else:
            flat = torch.zeros((L, per), dtype=F32, device=dev)
        ws_bytes = int(lib.vlb_bert_layer_backward_workspace(M, H, I))
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        dx = [torch.empty((M, H), dtype=BF16, device=dev), torch.empty((M, H), dtype=BF16, device=dev)]
        dx32 = [torch.empty((M, H), dtype=F32, device=dev), torch.empty((M, H), dtype=F32, device=dev)] if ctx.f32_stream else None
        carry32 = None      # fp32 residual-stream gradient handed down from the layer above
        gouts = list(grad_outs)
        if not meta.all_layers:
            gouts = [None] * (L - 1) + gouts
        dy16 = None
        grads = [None] * (16 * L)
        sizes = [3 * H * H, 3 * H, H * H, H, H, H, I * H, I, H * I, H, H, H]
        emb_ptr = ctx.emb.data_ptr()
        for l in range(L - 1, -1, -1):
            dy32 = gouts[l]
            if dy32 is not None:
                dy32 = dy32.contiguous().float().view(M, H)
                if carry32 is not None:
                    dy32 = dy32 + carry32          # (only when several layers' outputs were requested)
            elif carry32 is not None:
                dy32 = carry32
            if dy16 is None and dy32 is None:
                dy32 = torch.zeros((M, H), dtype=F32, device=dev)
            f = flat[l]
            parts = f.split(sizes)
            dw_qkv, db_qkv = parts[0].view(3 * H, H), parts[1]
            dw_o, db_o, dg1, dbt1 = parts[2].view(H, H), parts[3], parts[4], parts[5]
            dw_1, db_1 = parts[6].view(I, H), parts[7]
            dw_2, db_2, dg2, dbt2 = parts[8].view(H, I), parts[9], parts[10], parts[11]
            g = _lib.LayerGrads()
            g.dw_qkv, g.db_qkv, g.dw_o, g.db_o = dw_qkv.data_ptr(), db_qkv.data_ptr(), dw_o.data_ptr(), db_o.data_ptr()
            g.dln1_g, g.dln1_b, g.dw_1, g.db_1 = dg1.data_ptr(), dbt1.data_ptr(), dw_1.data_ptr(), db_1.data_ptr()
            g.dw_2, g.db_2, g.dln2_g, g.dln2_b = dw_2.data_ptr(), db_2.data_ptr(), dg2.data_ptr(), dbt2.data_ptr()
            w = meta.weights.layer_struct(l, params)
            a = _acts_struct(car, l, None, ctx.has_drop)
            x_ptr = emb_ptr if l == 0 else car.ptr("y%d" % (l - 1))
            out_dx = dx[l & 1]
            out_dx32 = dx32[l & 1] if dx32 is not None else None
            _chk(lib.vlb_bert_layer_backward(ctypes.byref(w), ctypes.byref(a), x_ptr, _p(ctx.add_mask), _p(dy16),
                                             _p(dy32), out_dx.data_ptr(), _p(out_dx32), ctypes.byref(g), ws.data_ptr(), ws_bytes,
                                             B, S, H, heads, I, ctx.drops[l], st))
            dy16 = out_dx
            carry32 = out_dx32
            if meta.reducer is not None:
                meta.reducer.launch(f)
            grads[16 * l: 16 * l + 16] = [dw_qkv[0:H], db_qkv[0:H], dw_qkv[H:2 * H], db_qkv[H:2 * H], dw_qkv[2 * H:],
                                          db_qkv[2 * H:], dw_o, db_o, dg1, dbt1, dw_1, db_1, dw_2, db_2, dg2, dbt2]
        if meta.reducer is not None:
            meta.reducer.drain()
        d_emb = dy16.view(B, S, H)
        d_emb32 = carry32.view(B, S, H) if carry32 is not None else None
        ctx.car = None
        return (d_emb, d_emb32, None, None) + tuple(grads)


# ------------------------------------------------------------------------------------------------
# embedding + packing (VisualLinguisticBert.embedding, common/visual_linguistic_bert.py:173-241)
# ------------------------------------------------------------------------------------------------
class PackIndex(object):
    """Device-side index tensors of the packed sequence (vlb_pack_index)."""

    def __init__(self, text_mask, object_mask, text_token_type_ids, S, pos_offset):
        _require_cuda(text_mask, object_mask, text_token_type_ids)
        B, T = text_mask.shape
        R = object_mask.shape[1]
        dev = text_mask.device
        self.B, self.T, self.R, self.S = B, T, R, S
        self.pos_offset = int(pos_offset)
        i32 = torch.int32
        self.kind = torch.empty((B, S), dtype=i32, device=dev)
        self.src = torch.empty((B, S), dtype=i32, device=dev)
        self.pos_id = torch.empty((B, S), dtype=i32, device=dev)
        self.type_id = torch.empty((B, S), dtype=i32, device=dev)
        self.add_mask = torch.empty((B, S), dtype=F32, device=dev)
        self.obj_row = torch.empty((B, R), dtype=i32, device=dev)
        self.lens = torch.empty((B, 2), dtype=i32, device=dev)
        self.err = torch.zeros((1,), dtype=i32, device=dev)
        self.text_mask_u8 = text_mask.to(torch.uint8).contiguous()
        self.object_mask_u8 = object_mask.to(torch.uint8).contiguous()
        self.type_ids = text_token_type_ids.to(torch.int64).contiguous()
        _chk(_lib.lib().vlb_pack_index(_p(self.text_mask_u8), _p(self.object_mask_u8), _p(self.type_ids), B, T, R, S,
                                       pos_offset, _p(self.kind), _p(self.src), _p(self.pos_id), _p(self.type_id),
                                       _p(self.add_mask), _p(self.obj_row), _p(self.lens), _p(self.err), _stream()))

    ERRORS = ((1, "max_length_hint is smaller than the longest packed sequence (text + regions + [END]): it must be a true upper bound"),
              (2, "position id out of range of position_embeddings"),
              (4, "token id out of range of word_embeddings"),
              (8, "token type id outside 0..2"))

    def check(self):
        """Raise IndexError if any kernel of the embedding flagged bad indices (one device->host sync).  The reference raises
        from the indexing op itself; here the flag is set asynchronously and the offending ids were remapped to row 0."""
        code = int(self.err.item())
        if code:
            raise IndexError("vlbert_b200 embedding: " + "; ".join(m for bit, m in self.ERRORS if code & bit))


class EmbeddingFn(torch.autograd.Function):
    """forward(text_visual f32 [B,T,H], object_vl f32 [B,R,2H], word, end, pos, type, ln_w, ln_b, vt_w, vt_b, vo_w, vo_b,
    ids int64 [B,T], pidx: PackIndex, eps, drop) -> (emb bf16 [B,S,H], emb f32 [B,S,H]): the same embedding twice -- the bf16
    copy is the GEMM operand of layer 0, the fp32 copy its residual operand; their gradients are summed in backward."""

    @staticmethod
    def forward(ctx, text_visual, object_vl, word, end, pos, typ, ln_w, ln_b, vt_w, vt_b, vo_w, vo_b, ids, pidx, eps, drop=None):
        _require_cuda(text_visual, object_vl, word)
        for nm, t in (("word_embeddings.weight", word), ("end_embedding.weight", end), ("position_embeddings.weight", pos),
                      ("token_type_embeddings.weight", typ), ("embedding_LayerNorm.weight", ln_w), ("embedding_LayerNorm.bias", ln_b),
                      ("visual_ln_text.weight", vt_w), ("visual_ln_text.bias", vt_b), ("visual_ln_object.weight", vo_w),
                      ("visual_ln_object.bias", vo_b)):
            _require_param(t, nm, text_visual.device)
        if typ.shape[0] < 3:
            raise RuntimeError("vlbert_b200: token_type_embeddings needs at least 3 rows (types 0/1 text, 2 regions and [END])")
        B, T, R, S = pidx.B, pidx.T, pidx.R, pidx.S
        H = word.shape[1]
        lib = _lib.lib()
        st = _stream()
        tv = text_visual.contiguous().float()
        ov = object_vl.contiguous().float()
        assert tv.shape[-1] == H and ov.shape[-1] == 2 * H
        _, tv_ln, tv_mean, tv_rstd = layernorm_forward(tv.view(B * T, H), vt_w, vt_b, eps, want_bf16=False, want_f32=True)
        _, ov_ln, ov_mean, ov_rstd = layernorm_forward(ov.view(B * R, 2 * H), vo_w, vo_b, eps, want_bf16=False, want_f32=True,
                                                       ldx=2 * H, H=H)
        e = torch.empty((B * S, H), dtype=F32, device=tv.device)
        ids = ids.contiguous()
        _chk(lib.vlb_pack_forward(_p(pidx.kind), _p(pidx.src), _p(pidx.pos_id), _p(pidx.type_id), _p(ids), _p(word), _p(end),
                                  _p(pos), _p(typ), _p(tv_ln), _p(ov_ln), _p(ov), 2 * H, H, _p(e), B, T, R, S, H,
                                  word.shape[0], pos.shape[0], _p(pidx.err), st))
        emb, emb32, e_mean, e_rstd = layernorm_forward(e, ln_w, ln_b, eps, want_f32=True, drop=drop)   # dropout(LayerNorm(.)), :237-239
        ctx.drop = drop
        ctx.save_for_backward(tv, ov, word, end, pos, typ, ln_w, vt_w, vo_w, ids, e, e_mean, e_rstd, tv_mean, tv_rstd,
                              ov_mean, ov_rstd)
        ctx.pidx = pidx
        ctx.dims = (B, T, R, S, H)
        return emb.view(B, S, H), emb32.view(B, S, H)

    @staticmethod
    def backward(ctx, d_emb, d_emb32):
        (tv, ov, word, end, pos, typ, ln_w, vt_w, vo_w, ids, e, e_mean, e_rstd, tv_mean, tv_rstd, ov_mean,
         ov_rstd) = ctx.saved_tensors
        pidx = ctx.pidx
        B, T, R, S, H = ctx.dims
        lib = _lib.lib()
        st = _stream()
        dev = e.device
        z = lambda *s: torch.zeros(s, dtype=F32, device=dev)  # noqa: E731
        d_ln_w, d_ln_b, d_vt_w, d_vt_b, d_vo_w, d_vo_b = z(H), z(H), z(H), z(H), z(H), z(H)
        dy16 = dy32 = None
        if d_emb is not None:
            d16 = d_emb.contiguous().view(B * S, H)
            dy16, dy32 = (d16, None) if d16.dtype == BF16 else (None, d16.float())
        if d_emb32 is not None:
            d32 = d_emb32.contiguous().view(B * S, H).float()
            dy32 = d32 if dy32 is None else dy32 + d32
        if dy16 is None and dy32 is None:
            dy32 = torch.zeros((B * S, H), dtype=F32, device=dev)
        _, de = layernorm_backward(dy16, dy32, e, e_mean, e_rstd, ln_w, d_ln_w, d_ln_b, want_bf16=False, want_f32=True,
                                   in_drop=ctx.drop)
        d_word, d_end, d_pos, d_typ = z(*word.shape), z(*end.shape), z(*pos.shape), z(*typ.shape)
        d_text_vl, d_obj_vl = z(B * T, H), z(B * R, H)
        _chk(lib.vlb_pack_backward(_p(pidx.kind), _p(pidx.src), _p(pidx.pos_id), _p(pidx.type_id), _p(ids), _p(de), _p(d_word),
                                   _p(d_end), _p(d_pos), _p(d_typ), _p(d_text_vl), _p(d_obj_vl), B, T, R, S, H, word.shape[0],
                                   pos.shape[0], pidx.pos_offset, st))
        _, d_tv = layernorm_backward(None, d_text_vl, tv.view(B * T, H), tv_mean, tv_rstd, vt_w, d_vt_w, d_vt_b,
                                     want_bf16=False, want_f32=True)
        d_ov = torch.empty((B * R, 2 * H), dtype=F32, device=dev)
        layernorm_backward(None, d_obj_vl, ov.view(B * R, 2 * H), ov_mean, ov_rstd, vo_w, d_vo_w, d_vo_b, want_bf16=False,
                           want_f32=True, ldx=2 * H, H=H, dx32=d_ov, ld_dx=2 * H)
        d_ov[:, H:] = d_obj_vl
        return (d_tv.view(B, T, H), d_ov.view(B, R, 2 * H), d_word, d_end, d_pos, d_typ, d_ln_w, d_ln_b, d_vt_w, d_vt_b,
                d_vo_w, d_vo_b, None, None, None, None)


class LinearFn(torch.autograd.Function):
    """y = x W^T + b on the tcgen05 GEMM for a small dense layer outside the encoder stack (BertPooler.dense,
    modeling.py:430-434): x f32/bf16 [N, K], W f32 [O, K], b f32 [O] -> y f32 [N, O].  bf16 operands, fp32 accumulation."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        _require_cuda(x, weight, bias)
        _require_param(weight, "dense.weight", x.device)
        _require_param(bias, "dense.bias", x.device)
        N, K = x.shape
        O = weight.shape[0]
        st = _stream()
        lib = _lib.lib()
        x16 = x.contiguous().to(BF16)
        w16 = torch.empty(weight.shape, dtype=BF16, device=x.device)
        _chk(lib.vlb_cast_f32_to_bf16(_p(weight), _p(w16), weight.numel(), st))
        y = torch.empty((N, O), dtype=F32, device=x.device)
        gemm(0, x16, w16, y, bias=bias)
        ctx.save_for_backward(x16, w16)
        return y

    @staticmethod
    def backward(ctx, dy):
        x16, w16 = ctx.saved_tensors
        N, K = x16.shape
        O = w16.shape[0]
        dev = x16.device
        # the reduction dimension of the weight gradient (N rows) is padded to a multiple of 8 (TMA leading dimension)
        Np = (N + 7) // 8 * 8
        dy16 = torch.zeros((Np, O), dtype=BF16, device=dev)
        dy16[:N] = dy
        xp = x16
        if Np != N:
            xp = torch.zeros((Np, K), dtype=BF16, device=dev)
            xp[:N] = x16
        d_b = torch.zeros((O,), dtype=F32, device=dev)
        _chk(_lib.lib().vlb_colsum_bf16(_p(dy16), O, _p(d_b), N, O, _stream()))
        d_w = torch.zeros((O, K), dtype=F32, device=dev)
        d_w._vlb_accumulate = True
        gemm(2, dy16, xp, d_w)
        dx = None
        if ctx.needs_input_grad[0]:
            dx16 = torch.empty((Np, K), dtype=BF16, device=dev)
            gemm(1, dy16, w16, dx16)
            dx = dx16[:N].float()
        return dx, d_w, d_b


class MLMLossFn(torch.autograd.Function):
    """Masked-LM loss of the pre-training task on the labelled positions only (csrc/heads.cu):
    forward(text_out f32 [B,T,H], labels int64 [B,T] (-1 = ignore), transform.dense.weight/bias, transform.LayerNorm.weight/bias,
            decoder weight [V,H] (the tied word embedding), decoder bias [V], cap)
      -> (loss = mean cross-entropy over the labelled positions, n_correct int32[1], n_labelled int32[1])
    i.e. F.cross_entropy(BertLMPredictionHead(text_out).view(-1, V), labels.view(-1), ignore_index=-1) of
    pretrain/modules/resnet_vlbert_for_pretraining.py:165-189 without the logits of the unlabelled positions.
    `cap` = static upper bound of labelled positions (rows the GEMMs run on)."""

    @staticmethod
    def forward(ctx, text_out, labels, tw, tb, ln_w, ln_b, dec_w, dec_b, cap, eps):
        _require_cuda(text_out, labels, dec_w)
        for nm, t in (("transform.dense.weight", tw), ("transform.dense.bias", tb), ("transform.LayerNorm.weight", ln_w),
                      ("transform.LayerNorm.bias", ln_b), ("decoder.weight", dec_w), ("bias", dec_b)):
            _require_param(t, "mlm_head.predictions." + nm, text_out.device)
        B, T, H = text_out.shape
        n, V = B * T, dec_w.shape[0]
        Vp = (V + 7) // 8 * 8
        cap = (int(cap) + 7) // 8 * 8
        dev = text_out.device
        lib, st = _lib.lib(), _stream()
        i32 = torch.int32
        idx = torch.empty((cap,), dtype=i32, device=dev)
        lab = torch.empty((cap,), dtype=i32, device=dev)
        count = torch.empty((1,), dtype=i32, device=dev)
        lbl = labels.contiguous().view(-1).to(torch.int64)
        _chk(lib.vlb_label_compact(_p(lbl), n, -1, _p(idx), _p(lab), cap, _p(count), st))
        x32 = text_out.contiguous().view(n, H).float()
        x16 = gather_rows(x32, idx, cap, BF16)
        tw16 = torch.empty((H, H), dtype=BF16, device=dev)
        _chk(lib.vlb_cast_f32_to_bf16(_p(tw), _p(tw16), tw.numel(), st))
        t32 = torch.empty((cap, H), dtype=F32, device=dev)
        z = torch.empty((cap, H), dtype=BF16, device=dev)
        gemm(0, x16, tw16, t32, bias=tb, act=1, aux=z)                       # dense + bias + erf-GELU (GELU' kept)
        h2, _, mean, rstd = layernorm_forward(t32, ln_w, ln_b, eps)
        w16 = torch.zeros((Vp, H), dtype=BF16, device=dev)                   # tied decoder = word embedding, rows padded to 8
        _chk(lib.vlb_cast_f32_to_bf16(_p(dec_w), _p(w16), dec_w.numel(), st))
        bias_p = torch.full((Vp,), -30000.0, dtype=F32, device=dev)          # padding columns never win the softmax
        bias_p[:V] = dec_b
        logits = torch.empty((cap, Vp), dtype=BF16, device=dev)
        gemm(0, h2, w16, logits, bias=bias_p)
        lse = torch.empty((cap,), dtype=F32, device=dev)
        loss_sum = torch.zeros((1,), dtype=F32, device=dev)
        correct = torch.zeros((1,), dtype=i32, device=dev)
        _chk(lib.vlb_mlm_ce_forward(_p(logits), Vp, V, _p(lab), _p(count), cap, _p(lse), _p(loss_sum), _p(correct), st))
        loss = (loss_sum / count.clamp(min=1).to(F32)).reshape(())
        ctx.save_for_backward(x16, tw16, t32, z, mean, rstd, h2, w16, logits, lab, count, lse, idx, ln_w)
        ctx.dims = (B, T, H, V, Vp, cap)
        ctx.mark_non_differentiable(correct, count)
        return loss, correct, count

    @staticmethod
    def backward(ctx, g_loss, _gc, _gn):
        x16, tw16, t32, z, mean, rstd, h2, w16, logits, lab, count, lse, idx, ln_w = ctx.saved_tensors
        B, T, H, V, Vp, cap = ctx.dims
        dev = x16.device
        lib, st = _lib.lib(), _stream()
        gscale = g_loss.detach().to(F32).reshape(1).contiguous()
        _chk(lib.vlb_mlm_ce_backward(_p(logits), Vp, V, _p(lab), _p(count), cap, _p(lse), _p(gscale), st))
        dlog = logits                                                         # in place: d loss / d logits, bf16 [cap, Vp]
        d_bias = torch.zeros((Vp,), dtype=F32, device=dev)
        _chk(lib.vlb_colsum_bf16(_p(dlog), Vp, _p(d_bias), cap, Vp, st))
        d_w = torch.zeros((Vp, H), dtype=F32, device=dev)
        d_w._vlb_accumulate = True
        gemm(2, dlog, h2, d_w)                                                # dW[v, :] += dlogits[:, v]^T h2
        dh2 = torch.empty((cap, H), dtype=BF16, device=dev)
        gemm(1, dlog, w16, dh2)                                               # dh2 = dlogits W
        d_ln_w, d_ln_b = torch.zeros((H,), dtype=F32, device=dev), torch.zeros((H,), dtype=F32, device=dev)
        _, d_t = layernorm_backward(dh2, None, t32, mean, rstd, ln_w, d_ln_w, d_ln_b, want_bf16=False, want_f32=True)
        d_pre = (d_t * z.float()).to(BF16)                                    # x GELU'(pre-activation)
        d_tb = torch.zeros((H,), dtype=F32, device=dev)
        _chk(lib.vlb_colsum_bf16(_p(d_pre), H, _p(d_tb), cap, H, st))
        d_tw = torch.zeros((H, H), dtype=F32, device=dev)
        d_tw._vlb_accumulate = True
        gemm(2, d_pre, x16, d_tw)
        dx = torch.empty((cap, H), dtype=BF16, device=dev)
        gemm(1, d_pre, tw16, dx)
        d_text = torch.zeros((B * T, H), dtype=F32, device=dev)
        scatter_rows_add(dx, idx, d_text)
        return d_text.view(B, T, H), None, d_tw, d_tb, d_ln_w, d_ln_b, d_w[:V], d_bias[:V], None, None


class MVRCLossFn(torch.autograd.Function):
    """Masked visual region classification loss of the pre-training task on the valid regions only (csrc/heads.cu):
    forward(object_out f32 [B,R,H], mvrc_labels f32 [B,R,C] (soft targets), transform.dense.weight/bias,
            region_cls_pred.weight [C,H] / bias [C], cap, norm_in_batch_first)
      -> (loss, n_correct int32[1], n_valid int32[1])
    i.e. soft_cross_entropy(VisualLinguisticBertMVRCHead(object_out).view(-1, C), mvrc_labels.view(-1, C)) of
    pretrain/modules/resnet_vlbert_for_pretraining.py:191-203 without the logits of the other regions.  A region is valid when
    its target row sums to 1 within 0.1 (common/utils/misc.py:133).
      norm_in_batch_first False: loss = sum of row losses / rows used                       (reduction='mean')
      norm_in_batch_first True : loss = sum_rows row_loss / (rows used in its sample + 1e-4), / (samples with a row + 1e-4)
    `cap` = static upper bound of valid rows (rows the GEMMs run on).  When more rows are valid, the first `cap` (ascending
    flat order) are used and the normalisation counts only those; n_valid still reports the true count.  No valid row:
    loss 0 and all gradients 0."""

    @staticmethod
    def forward(ctx, object_out, mvrc_labels, tw, tb, cw, cb, cap, norm_in_batch_first):
        _require_cuda(object_out, mvrc_labels, cw)
        for nm, t in (("transform.dense.weight", tw), ("transform.dense.bias", tb), ("region_cls_pred.weight", cw),
                      ("region_cls_pred.bias", cb)):
            _require_param(t, "mvrc_head." + nm, object_out.device)
        B, R, H = object_out.shape
        n, C = B * R, cw.shape[0]
        if tuple(mvrc_labels.shape) != (B, R, C):
            raise RuntimeError("vlbert_b200: mvrc_labels must be [B, R, C] = %s (got %s)" % ((B, R, C), tuple(mvrc_labels.shape)))
        Cp = (C + 7) // 8 * 8
        cap = (int(cap) + 7) // 8 * 8
        dev = object_out.device
        lib, st = _lib.lib(), _stream()
        i32 = torch.int32
        tgt = mvrc_labels.contiguous().view(n, C).float()
        arg = torch.empty((n,), dtype=torch.int64, device=dev)
        _chk(lib.vlb_soft_target_rows(_p(tgt), n, C, C, _p(arg), st))
        idx = torch.empty((cap,), dtype=i32, device=dev)
        lab = torch.empty((cap,), dtype=i32, device=dev)
        count = torch.empty((1,), dtype=i32, device=dev)
        _chk(lib.vlb_label_compact(_p(arg), n, -1, _p(idx), _p(lab), cap, _p(count), st))
        x16 = gather_rows(object_out.contiguous().view(n, H).float(), idx, cap, BF16)
        tw16 = torch.empty((H, H), dtype=BF16, device=dev)
        _chk(lib.vlb_cast_f32_to_bf16(_p(tw), _p(tw16), tw.numel(), st))
        h = torch.empty((cap, H), dtype=BF16, device=dev)
        z = torch.empty((cap, H), dtype=BF16, device=dev)
        gemm(0, x16, tw16, h, bias=tb, act=1, aux=z)                         # dense + bias + erf-GELU (GELU' kept)
        w16 = torch.zeros((Cp, H), dtype=BF16, device=dev)                   # classifier rows padded to 8
        _chk(lib.vlb_cast_f32_to_bf16(_p(cw), _p(w16), cw.numel(), st))
        bias_p = torch.full((Cp,), -30000.0, dtype=F32, device=dev)          # padding columns never win the softmax
        bias_p[:C] = cb
        logits = torch.empty((cap, Cp), dtype=BF16, device=dev)
        gemm(0, h, w16, logits, bias=bias_p)
        lse = torch.empty((cap,), dtype=F32, device=dev)
        row_loss = torch.empty((cap,), dtype=F32, device=dev)
        correct = torch.zeros((1,), dtype=i32, device=dev)
        _chk(lib.vlb_soft_ce_forward(_p(logits), Cp, C, _p(tgt), C, _p(idx), _p(lab), _p(count), cap, _p(lse), _p(row_loss),
                                     _p(correct), st))
        # wrow[k] = d loss / d row_loss[k], on the device (rows beyond the rows used have row_loss 0 and get no gradient)
        used = idx >= 0
        if norm_in_batch_first:
            sample = torch.where(used, idx // R, 0).long()
            per_sample = torch.zeros((B,), dtype=F32, device=dev).index_add_(0, sample, used.to(F32))
            n_has = (per_sample > 0).sum().to(F32)
            wrow = used.to(F32) / ((per_sample[sample] + 1e-4) * (n_has + 1e-4))
        else:
            wrow = used.to(F32) / used.sum().clamp(min=1).to(F32)
        loss = (row_loss * wrow).sum()
        ctx.save_for_backward(x16, tw16, h, z, w16, logits, tgt, idx, count, lse, wrow)
        ctx.dims = (B, R, H, C, Cp, cap)
        ctx.mark_non_differentiable(correct, count)
        return loss, correct, count

    @staticmethod
    def backward(ctx, g_loss, _gc, _gn):
        x16, tw16, h, z, w16, logits, tgt, idx, count, lse, wrow = ctx.saved_tensors
        B, R, H, C, Cp, cap = ctx.dims
        dev = x16.device
        lib, st = _lib.lib(), _stream()
        w = (wrow * g_loss.detach().to(F32)).contiguous()
        _chk(lib.vlb_soft_ce_backward(_p(logits), Cp, C, _p(tgt), C, _p(idx), _p(count), cap, _p(lse), _p(w), st))
        dlog = logits                                                         # in place: d loss / d logits, bf16 [cap, Cp]
        d_bias = torch.zeros((Cp,), dtype=F32, device=dev)
        _chk(lib.vlb_colsum_bf16(_p(dlog), Cp, _p(d_bias), cap, Cp, st))
        d_w = torch.zeros((Cp, H), dtype=F32, device=dev)
        d_w._vlb_accumulate = True
        gemm(2, dlog, h, d_w)                                                 # dW = dlogits^T h
        d_pre = torch.empty((cap, H), dtype=BF16, device=dev)
        gemm(1, dlog, w16, d_pre, act=3, aux=z)                               # (dlogits W) x GELU'(pre-activation)
        d_tb = torch.zeros((H,), dtype=F32, device=dev)
        _chk(lib.vlb_colsum_bf16(_p(d_pre), H, _p(d_tb), cap, H, st))
        d_tw = torch.zeros((H, H), dtype=F32, device=dev)
        d_tw._vlb_accumulate = True
        gemm(2, d_pre, x16, d_tw)
        dx = torch.empty((cap, H), dtype=BF16, device=dev)
        gemm(1, d_pre, tw16, dx)
        d_obj = torch.zeros((B * R, H), dtype=F32, device=dev)
        scatter_rows_add(dx, idx, d_obj)
        return d_obj.view(B, R, H), None, d_tw, d_tb, d_w[:C], d_bias[:C], None, None


class GatherRowsFn(torch.autograd.Function):
    """out[i] = idx[i] >= 0 ? src[idx[i]] : 0 ; src 2-D (bf16 or f32) -> f32.  Each source row is referenced at most once."""

    @staticmethod
    def forward(ctx, src2d, idx, n_out):
        ctx.save_for_backward(idx)
        ctx.n_src = src2d.shape[0]
        return gather_rows(src2d.contiguous(), idx, n_out, F32)

    @staticmethod
    def backward(ctx, g):
        (idx,) = ctx.saved_tensors
        out = torch.zeros((ctx.n_src, g.shape[1]), dtype=F32, device=g.device)
        scatter_rows_add(g.contiguous(), idx, out)
        return out, None, None


# ------------------------------------------------------------------------------------------------
# region-feature front end
# ------------------------------------------------------------------------------------------------
class RegionFn(torch.autograd.Function):
    """Precomputed-feature path of FastRCNN.forward (common/fast_rcnn.py:136-193):
    forward(boxes f32 [B,R,4+F], weight f32 [D, 2048+F], bias f32 [D], box_mask bool [B,R], im_info f32 [B,>=2])
      -> obj_reps f32 [B,R,D], obj_reps_raw f32 [B,R,F]   (both re-padded: k-th valid box in slot k)"""

    @staticmethod
    def forward(ctx, boxes, weight, bias, box_mask, im_info, drop=None):
        _require_cuda(boxes, weight, bias, box_mask, im_info)
        _require_param(weight, "obj_downsample.1.weight", boxes.device)
        _require_param(bias, "obj_downsample.1.bias", boxes.device)
        B, R, C = boxes.shape
        Fd = C - 4
        D = weight.shape[0]
        lib = _lib.lib()
        st = _stream()
        dev = boxes.device
        bx = boxes.contiguous().float()
        info = im_info.contiguous().float()
        mask_u8 = box_mask.to(torch.uint8).contiguous()
        A = torch.empty((B * R, 2048 + Fd), dtype=BF16, device=dev)
        gidx = torch.empty((B * R,), dtype=torch.int32, device=dev)
        # (the Dropout(0.1) heading obj_downsample, common/fast_rcnn.py:104-109, is applied while A is written)
        _chk(lib.vlb_region_operand_dropout(_p(bx), C, _p(mask_u8), _p(info), info.shape[1], None, None, _p(A), _p(gidx), B, R, Fd,
                                            _dref(drop), st))
        ctx.drop = drop
        w16 = torch.empty(weight.shape, dtype=BF16, device=dev)
        _chk(lib.vlb_cast_f32_to_bf16(_p(weight.contiguous()), _p(w16), weight.numel(), st))
        Y = torch.empty((B * R, D), dtype=BF16, device=dev)
        gemm(0, A, w16, Y, bias=bias, act=2)
        obj = gather_rows(Y, gidx, B * R, F32).view(B, R, D)
        raw = torch.empty((B * R, Fd), dtype=F32, device=dev)
        _chk(lib.vlb_gather_rows(bx.data_ptr() + 16, 0, C, _p(gidx), _p(raw), 0, Fd, B * R, Fd, st))
        ctx.save_for_backward(A, w16, Y, gidx)
        ctx.dims = (B, R, C, D)
        ctx.mark_non_differentiable(raw)
        return obj, raw.view(B, R, Fd)

    @staticmethod
    def backward(ctx, d_obj, _d_raw):
        A, w16, Y, gidx = ctx.saved_tensors
        B, R, C, D = ctx.dims
        Fd = C - 4
        lib = _lib.lib()
        st = _stream()
        dev = A.device
        # un-gather: dY[gidx[i]] = d_obj[i]
        dY32 = torch.zeros((B * R, D), dtype=F32, device=dev)
        scatter_rows_add(d_obj.contiguous().view(B * R, D).float(), gidx, dY32)
        # ReLU mask and bf16 operand
        dY = (dY32 * (Y > 0)).to(BF16)
        d_bias = torch.zeros((D,), dtype=F32, device=dev)
        _chk(lib.vlb_colsum_bf16(_p(dY), D, _p(d_bias), B * R, D, st))
        d_w = torch.zeros((D, 2048 + Fd), dtype=F32, device=dev)
        d_w._vlb_accumulate = True
        gemm(2, dY, A, d_w, split_k=max(1, min(16, (B * R) // 256)))
        # gradient wrt the feature half of boxes (the coordinate half is not propagated: the reference's boxes are data)
        if not ctx.needs_input_grad[0]:
            return None, d_w, d_bias, None, None, None
        d_boxes = torch.zeros((B * R, C), dtype=F32, device=dev)
        d_feat = torch.empty((B * R, Fd), dtype=BF16, device=dev)
        gemm(1, dY, w16[:, 2048:], d_feat, M=B * R, N=Fd, K=D)
        if ctx.drop is not None and ctx.drop.p > 0:      # the features entered the GEMM through the dropout mask
            d_feat = dropout_2d(d_feat, ctx.drop, col_offset=2048, total_cols=2048 + Fd)
        d_boxes[:, 4:] = d_feat.float()
        return d_boxes.view(B, R, C), d_w, d_bias, None, None, None


class RoIAlignFn(torch.autograd.Function):
    """_ROIAlign (common/lib/roi_pooling/roi_align.py:11-43) on vlb_roi_align_forward/backward."""

    @staticmethod
    def forward(ctx, input, rois, output_size, spatial_scale, sampling_ratio):
        ctx.save_for_backward(rois)
        ctx.cfg = (tuple(output_size), float(spatial_scale), int(sampling_ratio), tuple(input.shape))
        return roi_align_forward(input, rois, spatial_scale, output_size[0], output_size[1], sampling_ratio)

    @staticmethod
    def backward(ctx, grad):
        (rois,) = ctx.saved_tensors
        (ph, pw), scale, sr, (N, C, H, W) = ctx.cfg
        return roi_align_backward(grad, rois, scale, ph, pw, N, C, H, W, sr), None, None, None, None


def roi_align_forward(input, rois, spatial_scale, pooled_h, pooled_w, sampling_ratio):
    """C_ROIPooling.roi_align_forward (common/lib/roi_pooling/ROIAlign.h:11-25)."""
    _require_cuda(input, rois)
    inp = input.contiguous().float()
    r = rois.contiguous().float()
    N, C, H, W = inp.shape
    K = r.shape[0]
    out = torch.empty((K, C, pooled_h, pooled_w), dtype=F32, device=inp.device)
    _chk(_lib.lib().vlb_roi_align_forward(_p(inp), _p(r), _p(out), K, C, H, W, pooled_h, pooled_w, float(spatial_scale),
                                          int(sampling_ratio), _stream()))
    return out


def roi_align_backward(grad, rois, spatial_scale, pooled_h, pooled_w, batch_size, channels, height, width, sampling_ratio):
    """C_ROIPooling.roi_align_backward (common/lib/roi_pooling/ROIAlign.h:27-45)."""
    _require_cuda(grad, rois)
    g = grad.contiguous().float()
    r = rois.contiguous().float()
    gin = torch.empty((batch_size, channels, height, width), dtype=F32, device=g.device)
    _chk(_lib.lib().vlb_roi_align_backward(_p(g), _p(r), _p(gin), r.shape[0], batch_size, channels, height, width, pooled_h,
                                           pooled_w, float(spatial_scale), int(sampling_ratio), _stream()))
    return gin


# ------------------------------------------------------------------------------------------------
# convolution front end (NHWC bf16): conv + frozen BatchNorm + ReLU (+ residual) on the tcgen05 GEMM
# ------------------------------------------------------------------------------------------------
def _conv_out(n, k, stride, pad, dil):
    return (n + 2 * pad - dil * (k - 1) - 1) // stride + 1


def weight_to_gemm(weight, Kp=None):
    """[Cout, Cin, kh, kw] fp32 -> bf16 [Cout, Kp] with columns ordered (r, s, c) like the im2col rows."""
    Cout = weight.shape[0]
    w = weight.detach().permute(0, 2, 3, 1).reshape(Cout, -1)
    K = w.shape[1]
    Kp = Kp or _align(K, 8)
    if Kp != K:
        w = torch.nn.functional.pad(w, (0, Kp - K))
    return w.to(BF16).contiguous()


def _im2col(x, kh, kw, stride, pad, dil, Ho, Wo, Kp):
    N, H, W, C = x.shape
    col = torch.empty((N * Ho * Wo, Kp), dtype=BF16, device=x.device)
    _chk(_lib.lib().vlb_im2col_nhwc(_p(x), _p(col), N, H, W, C, kh, kw, stride, pad, dil, Ho, Wo, Kp, _stream()))
    return col


# implicit GEMM (TMA im2col-mode operand) for every convolution whose input channels are a multiple of 64; the explicit
# im2col lowering remains for the stem (C = 3) and for the data gradient of strided convolutions.  VLB_IMPLICIT_CONV=0 disables.
IMPLICIT_CONV = os.environ.get("VLB_IMPLICIT_CONV", "1") != "0"


def _geom(N, H, W, C, Ho, Wo, kh, kw, stride, pad, dil):
    return _lib.ConvGeom(N, H, W, C, Ho, Wo, kh, kw, stride, pad, dil)


def weight_to_dgrad(w16, Cout, kh, kw, C):
    """bf16 [Cout, (r, s, c)] -> [C, (r', s', k)] with r' = kh-1-r, s' = kw-1-s: the filter of the convolution over dY that
    yields dX for a stride-1 convolution."""
    return w16[:, :kh * kw * C].view(Cout, kh, kw, C).flip(1, 2).permute(3, 1, 2, 0).reshape(C, kh * kw * Cout).contiguous()


class ConvBnActFn(torch.autograd.Function):
    """y = act(conv(x, weight) * scale + shift (+ resid)) in NHWC bf16.
    relu_mode: 0 none, 1 ReLU, 2 ReLU after the residual add (Bottleneck output, resnet.py:110-116).
    scale/shift are the constants of a frozen eval-mode BatchNorm (no gradient)."""

    @staticmethod
    def forward(ctx, x, weight, scale, shift, resid, stride, pad, dil, relu_mode, w16, bag=None, role=None):
        _require_cuda(x, weight, scale)
        ctx.bag, ctx.role = bag, role
        N, H, W, C = x.shape
        Cout, Cin, kh, kw = weight.shape
        assert Cin == C and x.dtype == BF16 and x.is_contiguous()
        Ho, Wo = _conv_out(H, kh, stride, pad, dil), _conv_out(W, kw, stride, pad, dil)
        K = kh * kw * C
        Kp = _align(K, 8)
        if w16 is None:
            w16 = weight_to_gemm(weight, Kp)
        direct = (kh == 1 and kw == 1 and stride == 1 and pad == 0)
        implicit = IMPLICIT_CONV and not direct and C % 64 == 0
        P = N * Ho * Wo
        y = torch.empty((N, Ho, Wo, Cout), dtype=BF16, device=x.device)
        r = None if resid is None else resid.contiguous()
        lib = _lib.lib()
        if implicit:
            g = _geom(N, H, W, C, Ho, Wo, kh, kw, stride, pad, dil)
            _chk(lib.vlb_conv_fprop(_p(x), ctypes.byref(g), _p(w16), w16.stride(0), _p(y), Cout, _p(scale), _p(shift), _p(r),
                                    int(relu_mode), _stream()))
        else:
            col = x.view(N * H * W, C) if direct else _im2col(x, kh, kw, stride, pad, dil, Ho, Wo, Kp)
            _chk(lib.vlb_conv_gemm(_p(col), col.stride(0), _p(w16), w16.stride(0), _p(y), P, Cout, Kp, _p(scale), _p(shift),
                                   _p(r), int(relu_mode), _stream()))
        ctx.save_for_backward(x, w16, y if relu_mode else None, scale)
        ctx.geom = (N, H, W, C, Cout, kh, kw, stride, pad, dil, Ho, Wo, Kp, direct, implicit, relu_mode, resid is not None)
        ctx.wshape = tuple(weight.shape)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w16, y, scale = ctx.saved_tensors
        N, H, W, C, Cout, kh, kw, stride, pad, dil, Ho, Wo, Kp, direct, implicit, relu_mode, has_resid = ctx.geom
        lib = _lib.lib()
        st = _stream()
        dev = x.device
        P = N * Ho * Wo
        dy = dy.contiguous()
        need_x, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        need_r = has_resid and ctx.needs_input_grad[4]
        d_pre = torch.empty_like(dy) if need_r else None
        d_conv = torch.empty_like(dy)
        _chk(lib.vlb_relu_bn_backward(_p(dy), None, _p(y) if relu_mode else None, _p(scale), _p(d_pre), _p(d_conv), P, Cout, st))
        dconv2 = d_conv.view(P, Cout)
        dx = dw = None
        # Bottleneck identity branch: instead of handing d_pre to autograd (which would add it to conv1's dX with a separate
        # elementwise kernel), conv3 ("produce") parks it and conv1 ("consume") adds it in its data-gradient GEMM epilogue
        extra = None
        if ctx.role == "produce" and d_pre is not None:
            ctx.bag["d_identity"] = d_pre
            d_pre = None
        elif ctx.role == "consume":
            extra = ctx.bag.pop("d_identity", None)
            assert direct
        if need_w:
            dwk = torch.zeros((Cout, Kp), dtype=F32, device=dev)
            tiles = ((Cout + 127) // 128) * ((Kp + 255) // 256)
            split = max(1, min(16, 148 // max(1, tiles), (P + 63) // 64))
            if implicit:
                g = _geom(N, H, W, C, Ho, Wo, kh, kw, stride, pad, dil)
                _chk(lib.vlb_conv_wgrad(_p(x), ctypes.byref(g), _p(dconv2), Cout, _p(dwk), Kp, split, st))
            else:
                col = x.view(P, C) if direct else _im2col(x, kh, kw, stride, pad, dil, Ho, Wo, Kp)
                dwk._vlb_accumulate = True
                gemm(2, dconv2, col, dwk, split_k=split)
            dw = dwk[:, :kh * kw * C].view(Cout, kh, kw, C).permute(0, 3, 1, 2).contiguous()
        if need_x:
            if implicit and stride == 1 and Cout % 64 == 0:
                # dX = conv(dY, flipped filter): same implicit GEMM, no dcol / col2im
                pad_t = dil * (kh - 1) - pad
                g = _geom(N, Ho, Wo, Cout, H, W, kh, kw, 1, pad_t, dil)
                wd = weight_to_dgrad(w16, Cout, kh, kw, C)
                dx = torch.empty((N, H, W, C), dtype=BF16, device=dev)
                _chk(lib.vlb_conv_fprop(_p(d_conv), ctypes.byref(g), _p(wd), wd.stride(0), _p(dx), C, None, None, None, 0, st))
            else:
                dcol = torch.empty((P, Kp), dtype=BF16, device=dev)
                gemm(1, dconv2, w16, dcol, resid=extra.view(P, Kp) if extra is not None else None)
                extra = None
                if direct:
                    dx = dcol.view(N, H, W, C)
                else:
                    dx = torch.empty((N, H, W, C), dtype=BF16, device=dev)
                    _chk(lib.vlb_col2im_nhwc(_p(dcol), None, _p(dx), N, H, W, C, kh, kw, stride, pad, dil, Ho, Wo, Kp, st))
        if extra is not None:   # x needs no gradient itself but the identity branch does: pass it through
            dx = extra if dx is None else dx + extra
        return dx, dw, None, None, d_pre, None, None, None, None, None, None, None


def conv_bn_act(x, weight, scale, shift, resid=None, stride=1, pad=0, dil=1, relu_mode=1, w16=None, bag=None, role=None):
    return ConvBnActFn.apply(x, weight, scale, shift, resid, stride, pad, dil, relu_mode, w16, bag, role)


def maxpool3x3s2(x):
    N, H, W, C = x.shape
    Ho, Wo = (H + 2 - 3) // 2 + 1, (W + 2 - 3) // 2 + 1
    y = torch.empty((N, Ho, Wo, C), dtype=BF16, device=x.device)
    _chk(_lib.lib().vlb_maxpool3x3s2_nhwc(_p(x), _p(y), N, H, W, C, _stream()))
    return y


def nchw_to_nhwc_bf16(x):
    N, C, H, W = x.shape
    y = torch.empty((N, H, W, C), dtype=BF16, device=x.device)
    _chk(_lib.lib().vlb_nchw_f32_to_nhwc_bf16(_p(x.contiguous().float()), _p(y), N, C, H, W, _stream()))
    return y


def nhwc_to_nchw_f32(x):
    N, H, W, C = x.shape
    y = torch.empty((N, C, H, W), dtype=F32, device=x.device)
    _chk(_lib.lib().vlb_nhwc_bf16_to_nchw_f32(_p(x.contiguous()), _p(y), N, C, H, W, _stream()))
    return y


class AvgPoolFn(torch.autograd.Function):
    """mean over the spatial positions: bf16 [K, h, w, C] -> f32 [K, C]  (AvgPool2d + Flattener, common/fast_rcnn.py:80-84)"""

    @staticmethod
    def forward(ctx, x):
        K, h, w, C = x.shape
        y = torch.empty((K, C), dtype=F32, device=x.device)
        _chk(_lib.lib().vlb_avgpool_forward(_p(x.contiguous()), _p(y), K, h * w, C, _stream()))
        ctx.shape = (K, h, w, C)
        return y

    @staticmethod
    def backward(ctx, dy):
        K, h, w, C = ctx.shape
        dx = torch.empty((K, h, w, C), dtype=BF16, device=dy.device)
        _chk(_lib.lib().vlb_avgpool_backward(_p(dy.contiguous().float()), _p(dx), K, h * w, C, _stream()))
        return dx


class RoIAlignNHWCFn(torch.autograd.Function):
    """RoIAlign on an NHWC bf16 feature map (same sampling rules as the reference op) -> bf16 [K, ph, pw, C]."""

    @staticmethod
    def forward(ctx, feat, rois, ph, pw, spatial_scale, sampling_ratio):
        N, H, W, C = feat.shape
        r = rois.contiguous().float()
        K = r.shape[0]
        out = torch.empty((K, ph, pw, C), dtype=BF16, device=feat.device)
        _chk(_lib.lib().vlb_roi_align_nhwc_forward(_p(feat.contiguous()), _p(r), _p(out), K, C, H, W, ph, pw, float(spatial_scale),
                                                   int(sampling_ratio), _stream()))
        ctx.save_for_backward(r)
        ctx.cfg = (N, H, W, C, ph, pw, float(spatial_scale), int(sampling_ratio))
        return out

    @staticmethod
    def backward(ctx, g):
        (r,) = ctx.saved_tensors
        N, H, W, C, ph, pw, scale, sr = ctx.cfg
        gf = torch.empty((N, H, W, C), dtype=F32, device=g.device)
        _chk(_lib.lib().vlb_roi_align_nhwc_backward(_p(g.contiguous()), _p(r), _p(gf), r.shape[0], N, C, H, W, ph, pw, scale, sr, _stream()))
        return gf.to(BF16), None, None, None, None, None
