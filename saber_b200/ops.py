"""Thin Python wrappers over the C-ABI kernels: torch owns device memory and the stream, every
arithmetic op on the hot path is one of our sm_100a kernels. No CPU / eager fallback.
"""
from __future__ import annotations

import math
import os
from typing import Optional

import torch

from . import lib as _lib

ACT_NONE, ACT_GELU, ACT_RELU, ACT_SIGMOID = 0, 1, 2, 3
_BF16, _F32 = torch.bfloat16, torch.float32

launch_count = 0  # kernels launched through this module (bench.py reports it as gpu_launches)
_gemm_profiler = None  # set by GemmProfiler: CUDA events around every GEMM launch (bench.py roofline leg)


class GemmProfiler:
    """Context manager: brackets every ``gemm`` launch with CUDA events on the launching stream and sums the
    algorithmic FLOPs (2*M*N*K); ``summary()`` gives launches, milliseconds and achieved TFLOP/s."""

    def __init__(self):
        self.records = []

    def __enter__(self):
        global _gemm_profiler
        _gemm_profiler = self
        return self

    def __exit__(self, *exc):
        global _gemm_profiler
        _gemm_profiler = None
        return False

    def summary(self):
        torch.cuda.synchronize()
        ms = sum(r[1].elapsed_time(r[2]) for r in self.records)
        flops = float(sum(r[0] for r in self.records))
        return {"launches": len(self.records), "ms": ms, "flops": flops,
                "tflops": (flops / (ms * 1e-3) / 1e12) if ms > 0 else 0.0}

    def by_shape(self, top: int = 25):
        """Aggregate (tag, launches, ms, TFLOP/s) per GEMM shape, sorted by time."""
        torch.cuda.synchronize()
        agg = {}
        for rec in self.records:
            f, a, b = rec[0], rec[1], rec[2]
            tag = rec[3] if len(rec) > 3 else "?"
            e = agg.setdefault(tag, [0, 0.0, 0.0])
            e[0] += 1
            e[1] += a.elapsed_time(b)
            e[2] += f
        rows = sorted(agg.items(), key=lambda kv: -kv[1][1])[:top]
        return [(t, n, ms, fl / (ms * 1e-3) / 1e12 if ms > 0 else 0.0) for t, (n, ms, fl) in rows]


def _stream() -> int:
    # the current stream of the calling thread's current device, which _chk_cuda has just made the operands' device
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _chk_cuda(*ts):
    """Every wrapper calls this first: all tensor operands must live on ONE CUDA device, and that device becomes the
    calling thread's current device, so the kernel launch (C side: current device, stream from ``_stream()``) runs
    where the data is. SABER's GPUPool drives several GPUs from the threads of one process (REF saber/utils/
    parallelization.py:139-155); the current device is per-thread state, so pool threads do not disturb each other."""
    dev = None
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("saber_b200 ops need CUDA tensors: there is no CPU fallback")
        idx = t.device.index
        if dev is None:
            dev = idx
        elif idx != dev:
            raise RuntimeError(f"saber_b200 ops: operands on different devices (cuda:{dev} and cuda:{idx})")
    if dev is not None and dev != torch.cuda.current_device():
        torch.cuda.set_device(dev)


def _count(n=1):
    global launch_count
    launch_count += n


def require_b200() -> None:
    if not torch.cuda.is_available():
        raise RuntimeError("saber_b200 needs a CUDA device (sm_100a); no CPU fallback exists")
    L = _lib.load()
    _lib.check(L.sb_require_sm100(), "sb_require_sm100")


# ---------------------------------------------------------------------------------------------
# fp32 validation mode (BASELINE north_star: "1e-4 in the fp32 validation mode"; csrc/validate.cu). While it is on,
# executors keep fp32 weights (`weight()`), activations stay fp32 between kernels, every GEMM runs as the 6-term
# bf16 split product on the PRODUCTION tcgen05 kernel (K' = 6 K, fp32 accumulation in TMEM) and Hiera's attention
# runs in fp32 on CUDA cores. Covers the image encoder (U1); the fused decoder / memory kernels exist in bf16 only.
# ---------------------------------------------------------------------------------------------
VALIDATE_FP32 = os.environ.get("SB_VALIDATE_FP32", "0") == "1"
_split_w_cache: dict = {}
_weight_ptrs: set = set()  # fp32 weights created by weight(): only their split operands are cached


class validate_fp32:
    """Context manager: `with ops.validate_fp32(): model = build_sam2(...); model.forward_image(x)`."""

    def __init__(self, on: bool = True):
        self.on = on

    def __enter__(self):
        global VALIDATE_FP32
        self.prev, VALIDATE_FP32 = VALIDATE_FP32, self.on
        return self

    def __exit__(self, *exc):
        global VALIDATE_FP32
        VALIDATE_FP32 = self.prev
        _split_w_cache.clear()
        _weight_ptrs.clear()


def weight(t: torch.Tensor, device) -> torch.Tensor:
    """GEMM weight as the executors store it: bf16, or fp32 in validation mode."""
    w = t.to(device, _F32 if VALIDATE_FP32 else _BF16).contiguous()
    if VALIDATE_FP32:
        _weight_ptrs.add(w.data_ptr())
    return w


def act_dtype():
    """dtype of the activations that feed GEMMs / attention: bf16, or fp32 in validation mode."""
    return _F32 if VALIDATE_FP32 else _BF16


def split3(x: torch.Tensor, role: int) -> torch.Tensor:
    """fp32 [M,K] -> bf16 [M,6K] operand of the 6-term split product (role 0 activation, 1 weight)."""
    _chk_cuda(x)
    assert x.dtype == _F32 and x.dim() == 2 and x.stride(1) == 1 and x.shape[1] % 8 == 0, (x.dtype, x.shape)
    M, K = x.shape
    out = torch.empty((M, 6 * K), dtype=_BF16, device=x.device)
    L = _lib.load()
    _lib.check(L.sb_split3_bf16(x.data_ptr(), x.stride(0), M, K, role, out.data_ptr(), out.stride(0), _stream()),
               "sb_split3_bf16")
    _count()
    return out


def gelu_exact_(x: torch.Tensor) -> torch.Tensor:
    """Exact erf GELU in place on an fp32 tensor (validation mode)."""
    _chk_cuda(x)
    assert x.dtype == _F32 and x.is_contiguous()
    L = _lib.load()
    _lib.check(L.sb_gelu_exact_f32(x.data_ptr(), x.numel(), _stream()), "sb_gelu_exact_f32")
    _count()
    return x


def _gemm_validate(a, w, bias, act, residual, res_mod, out, alpha, force_bn):
    assert a.dtype == _F32 and w.dtype == _F32, "validation mode: fp32 activations and weights"
    key = (w.data_ptr(), tuple(w.shape), w.stride(0))
    w6 = _split_w_cache.get(key)
    if w6 is None:
        w6 = split3(w, 1)
        if key[0] in _weight_ptrs:  # a model weight (constant); activation-valued "weights" (hyper vectors) are not cached
            _split_w_cache[key] = w6
    a6 = split3(a, 0)
    if act == ACT_GELU:  # exact erf GELU after the product (the fused MUFU.TANH form is accurate to 4e-4 only)
        assert residual is None
        # the GELU kernel runs over numel() contiguous elements: a strided `out` would have other elements rewritten
        assert out is None or out.is_contiguous(), "validation mode: GELU needs a contiguous out"
        y = gemm(a6, w6, bias, ACT_NONE, None, 0, _F32, out=out, alpha=alpha, force_bn=force_bn)
        L = _lib.load()
        _lib.check(L.sb_gelu_exact_f32(y.data_ptr(), y.numel(), _stream()), "sb_gelu_exact_f32")
        _count()
        return y
    return gemm(a6, w6, bias, act, residual, res_mod, _F32, out=out, alpha=alpha, force_bn=force_bn)


def gemm(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, act: int = ACT_NONE,
         residual: Optional[torch.Tensor] = None, res_mod: int = 0, out_dtype=_BF16,
         out: Optional[torch.Tensor] = None, alpha: float = 1.0, force_bn: int = 0) -> torch.Tensor:
    """out[M,N] = act(alpha * a[M,K] @ w[N,K]^T + bias[N]) + residual[M (mod res_mod), N].

    a, w: bf16 row-major (last dim contiguous, pitch multiple of 8). bias: fp32. residual: bf16 or
    fp32 2-D. out: bf16 or fp32.
    """
    _chk_cuda(a, w, bias, residual, out)
    if w.dtype == _F32:  # validation mode: fp32 operands through the split product (fp32 result)
        return _gemm_validate(a, w, bias, act, residual, res_mod, out, alpha, force_bn)
    assert a.dtype == _BF16 and w.dtype == _BF16, (a.dtype, w.dtype)
    assert a.dim() == 2 and w.dim() == 2 and a.stride(1) == 1 and w.stride(1) == 1
    M, K = a.shape
    N, K2 = w.shape
    assert K == K2, (a.shape, w.shape)
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=a.device)
    assert out.dim() == 2 and out.stride(1) == 1 and out.shape == (M, N)
    flags = (1 if out.dtype == _F32 else 0)
    ldr = 0
    if residual is not None:
        assert residual.dim() == 2 and residual.stride(1) == 1 and residual.shape[1] == N
        assert residual.dtype in (_BF16, _F32)
        flags |= 2 if residual.dtype == _F32 else 0
        ldr = residual.stride(0)
    if bias is not None:
        assert bias.dtype == _F32 and bias.numel() == N and bias.is_contiguous()
    L = _lib.load()
    prof = _gemm_profiler
    if prof is not None:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
    rc = L.sb_gemm_bf16(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), out.data_ptr(),
                        out.stride(0), M, N, K, _ptr(bias), act, _ptr(residual), ldr, res_mod,
                        flags, alpha, force_bn, _stream())
    if prof is not None:
        ev1.record()
        prof.records.append((2.0 * M * N * K, ev0, ev1, f"std M={M} N={N} K={K} {'f32' if out.dtype == _F32 else 'bf16'}"
                             f"{' +res' if residual is not None else ''}"))
    _lib.check(rc, "sb_gemm_bf16")
    _count()
    return out


def _prof_begin():
    if _gemm_profiler is None:
        return None
    ev0 = torch.cuda.Event(enable_timing=True)
    ev0.record()
    return ev0


def _prof_end(ev0, flops, tag="fused"):
    if ev0 is not None and _gemm_profiler is not None:
        ev1 = torch.cuda.Event(enable_timing=True)
        ev1.record()
        _gemm_profiler.records.append((flops, ev0, ev1, tag))


def gemm_ln(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], residual: Optional[torch.Tensor],
            gamma: torch.Tensor, beta: torch.Tensor, eps: float, res_mod: int = 0, out_dtype=_BF16) -> torch.Tensor:
    """out = LayerNorm(a @ w^T + bias + residual[m % res_mod or m]) * gamma + beta, fused in the GEMM epilogue."""
    _chk_cuda(a, w, bias, residual, gamma, beta)
    if w.dtype == _F32:  # validation mode: split-product GEMM, then the row LayerNorm kernel
        y = gemm(a, w, bias, ACT_NONE, residual, res_mod, _F32)
        return layernorm(y, gamma, beta, eps, _F32)
    assert a.dtype == _BF16 and w.dtype == _BF16 and a.stride(1) == 1 and w.stride(1) == 1
    M, K = a.shape
    N = w.shape[0]
    assert w.shape[1] == K and N <= 256 and N % 16 == 0
    out = torch.empty((M, N), dtype=out_dtype, device=a.device)
    flags = 1 if out_dtype == _F32 else 0
    ldr = 0
    if residual is not None:
        assert residual.dim() == 2 and residual.stride(1) == 1 and residual.shape[1] == N
        flags |= 2 if residual.dtype == _F32 else 0
        ldr = residual.stride(0)
    L = _lib.load()
    ev = _prof_begin()
    rc = L.sb_gemm_ln(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), out.data_ptr(), out.stride(0), M, N, K,
                      _ptr(bias), _ptr(residual), ldr, res_mod, flags, gamma.data_ptr(), beta.data_ptr(), eps, _stream())
    _prof_end(ev, 2.0 * M * N * K, f"ln M={M} N={N} K={K}")
    _lib.check(rc, "sb_gemm_ln")
    _count()
    return out


def iou_gate(ious4: torch.Tensor, thresh: float):
    """Prompts whose best predicted IoU exceeds `thresh` (ascending): (list int32 [B], count int32 [1]) on the device."""
    _chk_cuda(ious4)
    assert ious4.dtype == _F32 and ious4.is_contiguous() and ious4.dim() == 2 and ious4.shape[1] == 4
    B = ious4.shape[0]
    lst = torch.empty((B,), dtype=torch.int32, device=ious4.device)
    cnt = torch.empty((1,), dtype=torch.int32, device=ious4.device)
    L = _lib.load()
    _lib.check(L.sb_iou_gate(ious4.data_ptr(), B, float(thresh), lst.data_ptr(), cnt.data_ptr(), _stream()), "sb_iou_gate")
    _count()
    return lst, cnt


def gemm_upscale1(keys: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, feat_s1: torch.Tensor, s1_bstride: int,
                  gamma: torch.Tensor, beta: torch.Tensor, B: int, gh: int, gw: int, eps: float = 1e-6,
                  plist=None) -> torch.Tensor:
    """keys [B*gh*gw,256] bf16 -> u1 [B*2gh*2gw, 64] bf16 (transposed conv + skip + LayerNorm2d + GELU fused).
    plist = (list, count) from iou_gate: only those prompts are computed."""
    _chk_cuda(keys, w, bias, feat_s1, gamma, beta)
    assert keys.dtype == _BF16 and keys.shape == (B * gh * gw, 256) and keys.stride(1) == 1
    assert w.dtype == _BF16 and w.shape == (256, 256) and bias.numel() == 256 and feat_s1.dtype == _F32
    u1 = torch.empty((B * 4 * gh * gw, 64), dtype=_BF16, device=keys.device)
    L = _lib.load()
    ev = _prof_begin()
    rc = L.sb_gemm_upscale1(keys.data_ptr(), keys.stride(0), w.data_ptr(), w.stride(0), B, gh, gw, bias.data_ptr(),
                            feat_s1.data_ptr(), s1_bstride, gamma.data_ptr(), beta.data_ptr(), eps, u1.data_ptr(),
                            _ptr(plist[0]) if plist else None, _ptr(plist[1]) if plist else None, _stream())
    _prof_end(ev, 2.0 * B * gh * gw * 256 * 256, f"up1 M={B * gh * gw} N=256 K=256")
    _lib.check(rc, "sb_gemm_upscale1")
    _count()
    return u1


def gemm_upscale2(u1: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, feat_s0: torch.Tensor, s0_bstride: int,
                  hyper: torch.Tensor, B: int, gh: int, gw: int, plist=None, zero_fill: bool = False) -> torch.Tensor:
    """u1 [B*gh*gw,64] bf16 -> masks [B,4,2gh,2gw] fp32 (transposed conv + skip + GELU + hyper-network dot fused).
    plist = (list, count) from iou_gate: only those prompts' masks are written (the others are uninitialised, or zero
    with zero_fill)."""
    _chk_cuda(u1, w, bias, feat_s0, hyper)
    assert u1.dtype == _BF16 and u1.shape == (B * gh * gw, 64) and (gh * gw) % 128 == 0
    assert w.dtype == _BF16 and w.shape == (128, 64) and bias.numel() == 128 and feat_s0.dtype == _F32
    assert hyper.dtype == _F32 and hyper.is_contiguous() and hyper.shape == (B, 4, 32)
    masks = (torch.zeros if (plist and zero_fill) else torch.empty)((B, 4, 2 * gh, 2 * gw), dtype=_F32, device=u1.device)
    L = _lib.load()
    ev = _prof_begin()
    rc = L.sb_gemm_upscale2(u1.data_ptr(), u1.stride(0), w.data_ptr(), w.stride(0), B, gh, gw, bias.data_ptr(),
                            feat_s0.data_ptr(), s0_bstride, hyper.data_ptr(), masks.data_ptr(),
                            _ptr(plist[0]) if plist else None, _ptr(plist[1]) if plist else None, _stream())
    _prof_end(ev, 2.0 * B * gh * gw * 128 * 64, f"up2 M={B * gh * gw} N=128 K=64")
    _lib.check(rc, "sb_gemm_upscale2")
    _count()
    return masks


def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-6,
              out_dtype=_BF16, act: int = ACT_NONE, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """LayerNorm over the last dim of a 2-D row-major tensor (fp32 or bf16 in; bf16 or fp32 out)."""
    _chk_cuda(x, gamma, beta, out)
    assert x.dim() == 2 and x.stride(1) == 1 and x.dtype in (_BF16, _F32)
    M, Cc = x.shape
    if VALIDATE_FP32 and out is None:
        out_dtype = _F32
    if out is None:
        out = torch.empty((M, Cc), dtype=out_dtype, device=x.device)
    assert gamma.dtype == _F32 and beta.dtype == _F32
    L = _lib.load()
    rc = L.sb_layernorm(x.data_ptr(), x.stride(0), int(x.dtype == _F32), out.data_ptr(), out.stride(0),
                        int(out.dtype == _F32), gamma.data_ptr(), beta.data_ptr(), M, Cc, eps, act,
                        _stream())
    _lib.check(rc, "sb_layernorm")
    _count()
    return out


def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, batch: int, heads: int, nq: int,
              nk: int, scale: Optional[float] = None, out: Optional[torch.Tensor] = None,
              q_shared: bool = False, kv_shared: bool = False) -> torch.Tensor:
    """Plain batched MHA. q [batch*nq, heads*hd], k/v [batch*nk, heads*hd] (bf16, row views allowed).
    With q_shared / kv_shared the operand holds one batch entry ([nq|nk, C]) read by every batch element."""
    _chk_cuda(q, k, v, out)
    if q.dtype == _F32:  # validation mode
        return _attention_f32(q, k, None, v, batch, heads, nq, nk, scale, q_shared, kv_shared, out)
    assert q.dtype == _BF16 and k.dtype == _BF16 and v.dtype == _BF16
    Cc = q.shape[1]
    hd = Cc // heads
    assert q.shape[0] == (1 if q_shared else batch) * nq
    assert k.shape[0] == (1 if kv_shared else batch) * nk and v.shape[0] == k.shape[0]
    if scale is None:
        scale = 1.0 / math.sqrt(hd)
    if out is None:
        out = torch.empty((batch * nq, Cc), dtype=_BF16, device=q.device)
    L = _lib.load()
    rc = L.sb_attention(q.data_ptr(), q.stride(0), k.data_ptr(), k.stride(0), v.data_ptr(), v.stride(0),
                        out.data_ptr(), out.stride(0), batch, heads, hd, nq, nk, scale, int(q_shared),
                        int(kv_shared), _stream())
    _lib.check(rc, "sb_attention")
    _count()
    return out


def _attention_f32(q, k, k_add, v, batch, heads, nq, nk, scale, q_shared, kv_shared, out):
    assert q.dtype == _F32 and k.dtype == _F32 and v.dtype == _F32 and (k_add is None or k_add.dtype == _F32)
    assert q.stride(1) == 1 and k.stride(1) == 1 and v.stride(1) == 1
    Cc = q.shape[1]
    hd = Cc // heads
    if scale is None:
        scale = 1.0 / math.sqrt(hd)
    if out is None:
        out = torch.empty((batch * nq, Cc), dtype=_F32, device=q.device)
    L = _lib.load()
    _lib.check(L.sb_attention_f32(q.data_ptr(), q.stride(0), k.data_ptr(), k.stride(0), _ptr(k_add),
                                  k_add.stride(0) if k_add is not None else 0, v.data_ptr(), v.stride(0), out.data_ptr(),
                                  out.stride(0), batch, heads, hd, nq, nk, scale, int(q_shared), int(kv_shared), _stream()),
               "sb_attention_f32")
    _count()
    return out


def attention_kadd(q: torch.Tensor, k: torch.Tensor, k_add: torch.Tensor, v: torch.Tensor, batch: int, heads: int, nq: int,
                   nk: int, kv_shared: bool = False, scale: Optional[float] = None) -> torch.Tensor:
    """attention() with scores = q (k[b] + k_add)^T; k_add [nk, heads*hd] bf16 is shared by all batch entries."""
    _chk_cuda(q, k, k_add, v)
    if q.dtype == _F32:  # validation mode
        return _attention_f32(q, k, k_add, v, batch, heads, nq, nk, scale, False, kv_shared, None)
    assert q.dtype == _BF16 and k.dtype == _BF16 and v.dtype == _BF16 and k_add.dtype == _BF16
    Cc = q.shape[1]
    hd = Cc // heads
    assert q.shape[0] == batch * nq and k.shape[0] == (1 if kv_shared else batch) * nk and v.shape[0] == k.shape[0]
    assert k_add.shape == (nk, Cc) and k_add.stride(1) == 1
    if scale is None:
        scale = 1.0 / math.sqrt(hd)
    out = torch.empty((batch * nq, Cc), dtype=_BF16, device=q.device)
    L = _lib.load()
    _lib.check(L.sb_attention_kadd(q.data_ptr(), q.stride(0), k.data_ptr(), k.stride(0), k_add.data_ptr(), k_add.stride(0),
                                   v.data_ptr(), v.stride(0), out.data_ptr(), out.stride(0), batch, heads, hd, nq, nk,
                                   scale, int(kv_shared), _stream()), "sb_attention_kadd")
    _count()
    return out


def attention_few_keys(q: torch.Tensor, q_add: Optional[torch.Tensor], k: torch.Tensor, v: torch.Tensor, batch: int,
                       nq: int, nk: int, q_shared: bool = False, scale: Optional[float] = None) -> torch.Tensor:
    """Image -> token attention of the mask decoder (8 heads x 16, nk <= 16): out[b, i] = softmax((q[b,i] + q_add[i]) k_b^T)
    v_b. q [batch*nq (nq when q_shared), 128] bf16 (row views allowed), q_add [nq,128] fp32 or None."""
    _chk_cuda(q, q_add, k, v)
    assert q.dtype == _BF16 and k.dtype == _BF16 and v.dtype == _BF16 and q.shape[1] == 128 and q.stride(1) == 1
    assert q.shape[0] == (1 if q_shared else batch) * nq and k.shape == (batch * nk, 128) and v.shape == k.shape
    assert q_add is None or (q_add.dtype == _F32 and q_add.is_contiguous() and q_add.shape == (nq, 128))
    if scale is None:
        scale = 0.25
    out = torch.empty((batch * nq, 128), dtype=_BF16, device=q.device)
    L = _lib.load()
    _lib.check(L.sb_attention_few_keys(q.data_ptr(), q.stride(0), _ptr(q_add), k.data_ptr(), k.stride(0), v.data_ptr(),
                                       v.stride(0), out.data_ptr(), out.stride(0), batch, nq, nk, scale, int(q_shared),
                                       _stream()), "sb_attention_few_keys")
    _count()
    return out


def i2t_fold(kt: torch.Tensor, vt: torch.Tensor, wq: torch.Tensor, wo: torch.Tensor, batch: int, nt: int,
             bo: torch.Tensor, scale: float = 0.25):
    """Per-prompt folded operands of ``i2t_block_tc`` (TwoWayAttentionBlock step 4 with <= 8 tokens per prompt):
    kt / vt [batch*nt, 128] bf16 (row views allowed), wq [128,256] / wo [256,128] bf16, bo [256] fp32 (the out-projection
    bias, folded into w2t) -> (w1t [B,64,256], w2t [B,256,64], kts [B,8,128]) bf16."""
    _chk_cuda(kt, vt, wq, wo, bo)
    assert kt.dtype == _BF16 and vt.dtype == _BF16 and wq.dtype == _BF16 and wo.dtype == _BF16
    assert kt.shape == (batch * nt, 128) and vt.shape == kt.shape and kt.stride(1) == 1 and vt.stride(1) == 1
    assert wq.shape == (128, 256) and wq.is_contiguous() and wo.shape == (256, 128) and wo.is_contiguous()
    assert bo.dtype == _F32 and bo.is_contiguous() and bo.numel() == 256
    dev = kt.device
    w1t = torch.empty((batch, 64, 256), dtype=_BF16, device=dev)
    w2t = torch.empty((batch, 256, 64), dtype=_BF16, device=dev)
    kts = torch.empty((batch, 8, 128), dtype=_BF16, device=dev)
    L = _lib.load()
    _lib.check(L.sb_i2t_fold(kt.data_ptr(), kt.stride(0), vt.data_ptr(), vt.stride(0), wq.data_ptr(), wo.data_ptr(),
                             bo.data_ptr(), w1t.data_ptr(), w2t.data_ptr(), kts.data_ptr(), batch, nt, scale, _stream()),
               "sb_i2t_fold")
    _count()
    return w1t, w2t, kts


def i2t_block_tc(x: torch.Tensor, qres: torch.Tensor, w1t: torch.Tensor, w2t: torch.Tensor, kts: torch.Tensor,
                 gamma: torch.Tensor, beta: torch.Tensor, eps: float, batch: int, nq: int, nt: int,
                 out: Optional[torch.Tensor] = None, x_shared: bool = False) -> torch.Tensor:
    """keys_new = LN(keys + out_proj(attn(keys -> tokens))) in one pass over the image stream on tcgen05 / TMEM / TMA
    (csrc/decoder_i2t_tc.cu). x [batch*nq (nq when x_shared), 256] bf16, qres [nq,128] bf16 (= image_pe Wq^T + bq),
    w1t / w2t / kts from ``i2t_fold``; ``out`` may be ``x`` itself for a per-prompt stream."""
    _chk_cuda(x, qres, w1t, w2t, kts, gamma, beta)
    assert x.dtype == _BF16 and x.is_contiguous() and x.shape == ((1 if x_shared else batch) * nq, 256)
    assert qres.dtype == _BF16 and qres.is_contiguous() and qres.shape == (nq, 128)
    assert w1t.dtype == _BF16 and w1t.is_contiguous() and w1t.shape == (batch, 64, 256)
    assert w2t.dtype == _BF16 and w2t.is_contiguous() and w2t.shape == (batch, 256, 64)
    assert kts.dtype == _BF16 and kts.is_contiguous() and kts.shape == (batch, 8, 128)
    for v in (gamma, beta):
        assert v.dtype == _F32 and v.is_contiguous() and v.numel() == 256
    if out is None:
        out = torch.empty((batch * nq, 256), dtype=_BF16, device=x.device)
    assert out.dtype == _BF16 and out.is_contiguous() and out.shape == (batch * nq, 256)
    L = _lib.load()
    _lib.check(L.sb_i2t_block_tc(x.data_ptr(), int(x_shared), qres.data_ptr(), w1t.data_ptr(), w2t.data_ptr(), kts.data_ptr(),
                                 gamma.data_ptr(), beta.data_ptr(), eps, out.data_ptr(), batch, nq, nt, _stream()),
               "sb_i2t_block_tc")
    _count()
    return out


def t2i_fold_attention(q: torch.Tensor, x: torch.Tensor, kadd: torch.Tensor, wk: torch.Tensor, wv: torch.Tensor,
                       bv: torch.Tensor, batch: int, nt: int, nk: int, x_shared: bool = False,
                       scale: float = 0.25) -> torch.Tensor:
    """Mask-decoder token -> image attention on the raw image stream (k / v projections folded onto the <= 8 tokens of a
    prompt; both GEMMs on tcgen05, csrc/decoder_t2i_tc.cu). q [batch*nt,128] bf16, x [batch*nk (nk when shared),256]
    bf16, kadd [nk,128] bf16, wk / wv [128,256] bf16 (row views of a stacked weight allowed), bv [128] fp32
    -> [batch*nt,128] bf16."""
    _chk_cuda(q, x, kadd, wk, wv, bv)
    assert q.dtype == _BF16 and q.shape == (batch * nt, 128) and q.stride(1) == 1
    assert x.dtype == _BF16 and x.is_contiguous() and x.shape == ((1 if x_shared else batch) * nk, 256)
    assert kadd.dtype == _BF16 and kadd.is_contiguous() and kadd.shape == (nk, 128)
    for w_ in (wk, wv):
        assert w_.dtype == _BF16 and w_.shape == (128, 256) and w_.is_contiguous()
    assert bv.dtype == _F32 and bv.is_contiguous() and bv.numel() == 128
    L = _lib.load()
    ns = L.sb_t2i_tc_splits(batch, nk)
    dev = q.device
    qf = torch.empty((batch, 64, 384), dtype=_BF16, device=dev)
    qs = torch.empty((batch, 8, 128), dtype=_BF16, device=dev)
    opart = torch.empty((batch, ns, 64, 256), dtype=_F32, device=dev)
    ml = torch.empty((batch, ns, 2, 64), dtype=_F32, device=dev)
    out = torch.empty((batch * nt, 128), dtype=_BF16, device=dev)
    _lib.check(L.sb_t2i_fold_attention_tc(q.data_ptr(), q.stride(0), x.data_ptr(), int(x_shared), kadd.data_ptr(),
                                          wk.data_ptr(), wv.data_ptr(), bv.data_ptr(), qf.data_ptr(), qs.data_ptr(),
                                          opart.data_ptr(), ml.data_ptr(), out.data_ptr(), out.stride(0), batch, nt, nk,
                                          scale, _stream()), "sb_t2i_fold_attention_tc")
    _count(3)
    return out


def mask_embed_keys(ds: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, image_embed: torch.Tensor) -> torch.Tensor:
    """Per-prompt image stream of the m2m pass: bf16(image_embed[t] + bias + ds @ w^T); ds [B*T,16] bf16, w [256,16] fp32.
    The kernel rounds ``w`` to bf16 (the product is one bf16 tensor-core step per 16 tokens) and accumulates in fp32 from
    ``image_embed + bias``, so the result is that of the bf16-rounded ``w``, not of the fp32 one."""
    _chk_cuda(ds, w, bias, image_embed)
    assert ds.dtype == _BF16 and ds.is_contiguous() and ds.shape[1] == 16 and w.dtype == _F32 and w.shape == (256, 16)
    assert image_embed.dtype == _F32 and image_embed.is_contiguous() and image_embed.shape[1] == 256
    T = image_embed.shape[0]
    assert ds.shape[0] % T == 0
    keys = torch.empty((ds.shape[0], 256), dtype=_BF16, device=ds.device)
    L = _lib.load()
    _lib.check(L.sb_mask_embed_keys(ds.data_ptr(), w.data_ptr(), bias.data_ptr(), image_embed.data_ptr(), T, ds.shape[0],
                                    keys.data_ptr(), _stream()), "sb_mask_embed_keys")
    _count()
    return keys


def window_attention(qkv: torch.Tensor, qkv_bias: Optional[torch.Tensor], batch: int, H: int, W: int,
                     heads: int, ws: int, pool: int = 1, scale: Optional[float] = None) -> torch.Tensor:
    """Hiera (windowed / global, optionally q-pooled) attention over a fused qkv [B*H*W, 3*C] buffer."""
    _chk_cuda(qkv, qkv_bias)
    if qkv.dtype == _F32:  # validation mode
        return _window_attention_f32(qkv, qkv_bias, batch, H, W, heads, ws, pool, scale)
    assert qkv.dtype == _BF16 and qkv.is_contiguous() and qkv.shape[0] == batch * H * W
    C3 = qkv.shape[1]
    Cc = C3 // 3
    hd = Cc // heads
    if scale is None:
        scale = 1.0 / math.sqrt(hd)
    if ws <= 0 or ws >= max(H, W):
        ws = max(H, W)
    Ho, Wo = H // pool, W // pool
    out = torch.empty((batch * Ho * Wo, Cc), dtype=_BF16, device=qkv.device)
    L = _lib.load()
    rc = L.sb_window_attention(qkv.data_ptr(), _ptr(qkv_bias), out.data_ptr(), batch, H, W, heads, hd,
                               ws, pool, scale, _stream())
    _lib.check(rc, "sb_window_attention")
    _count()
    return out


def _window_attention_f32(qkv, qkv_bias, batch, H, W, heads, ws, pool, scale):
    assert qkv.is_contiguous() and qkv.shape[0] == batch * H * W
    Cc = qkv.shape[1] // 3
    hd = Cc // heads
    if scale is None:
        scale = 1.0 / math.sqrt(hd)
    if ws <= 0 or ws >= max(H, W):
        ws = max(H, W)
    out = torch.empty((batch * (H // pool) * (W // pool), Cc), dtype=_F32, device=qkv.device)
    L = _lib.load()
    _lib.check(L.sb_window_attention_f32(qkv.data_ptr(), _ptr(qkv_bias), out.data_ptr(), batch, H, W, heads, hd, ws, pool,
                                         scale, _stream()), "sb_window_attention_f32")
    _count()
    return out


def hiera_attention_tc(qkv: torch.Tensor, batch: int, H: int, W: int, heads: int, ws: int,
                       scale: Optional[float] = None) -> torch.Tensor:
    """The tcgen05 Hiera attention (head_dim 72, no q-pooling) called directly; raises for unsupported windows."""
    _chk_cuda(qkv)
    assert qkv.dtype == _BF16 and qkv.is_contiguous() and qkv.shape == (batch * H * W, 3 * heads * 72)
    if scale is None:
        scale = 1.0 / math.sqrt(72)
    out = torch.empty((batch * H * W, heads * 72), dtype=_BF16, device=qkv.device)
    L = _lib.load()
    _lib.check(L.sb_hiera_attention_tc(qkv.data_ptr(), out.data_ptr(), batch, H, W, heads, ws, scale, _stream()),
               "sb_hiera_attention_tc")
    _count()
    return out


def im2col_k7s4(img: torch.Tensor, kp: int) -> torch.Tensor:
    """[B,Cin,S,S] fp32 -> [B*(S/4)^2, kp] bf16 patches for the 7x7 stride-4 pad-3 patch embedding."""
    _chk_cuda(img)
    assert img.dtype == _F32 and img.is_contiguous() and img.dim() == 4 and img.shape[2] == img.shape[3]
    B, Cin, S, _ = img.shape
    cols = torch.empty((B * (S // 4) ** 2, kp), dtype=act_dtype(), device=img.device)
    L = _lib.load()
    fn = L.sb_im2col_k7s4_f32 if VALIDATE_FP32 else L.sb_im2col_k7s4
    _lib.check(fn(img.data_ptr(), cols.data_ptr(), B, Cin, S, kp, _stream()), "sb_im2col_k7s4")
    _count()
    return cols


def maxpool2x2(x: torch.Tensor, B: int, H: int, W: int) -> torch.Tensor:
    """Token-major [B*H*W, C] -> [B*(H/2)*(W/2), C]."""
    _chk_cuda(x)
    assert x.is_contiguous() and x.dtype in (_BF16, _F32)
    Cc = x.shape[1]
    out = torch.empty((B * (H // 2) * (W // 2), Cc), dtype=x.dtype, device=x.device)
    L = _lib.load()
    _lib.check(L.sb_maxpool2x2(x.data_ptr(), out.data_ptr(), int(x.dtype == _F32), B, H, W, Cc, _stream()),
               "sb_maxpool2x2")
    _count()
    return out


def add_upsample2x_(dst: torch.Tensor, src: torch.Tensor, B: int, H: int, W: int) -> torch.Tensor:
    """dst[B*H*W, C] += nearest-2x(src[B*(H/2)*(W/2), C]) — both fp32 token-major."""
    _chk_cuda(dst, src)
    assert dst.dtype == _F32 and src.dtype == _F32 and dst.is_contiguous() and src.is_contiguous()
    L = _lib.load()
    _lib.check(L.sb_add_upsample2x(dst.data_ptr(), src.data_ptr(), B, H, W, dst.shape[1], _stream()),
               "sb_add_upsample2x")
    _count()
    return dst


def nhwc_to_nchw(x: torch.Tensor, B: int, HW: int, out_dtype=_F32,
                 chan_add: Optional[torch.Tensor] = None) -> torch.Tensor:
    """[B*HW, C] token-major -> [B, C, HW] (optionally adding a per-channel fp32 vector)."""
    _chk_cuda(x, chan_add)
    assert x.is_contiguous() and x.shape[0] == B * HW
    Cc = x.shape[1]
    out = torch.empty((B, Cc, HW), dtype=out_dtype, device=x.device)
    L = _lib.load()
    _lib.check(L.sb_nhwc_to_nchw(x.data_ptr(), int(x.dtype == _F32), out.data_ptr(), int(out_dtype == _F32),
                                 B, HW, Cc, _ptr(chan_add), _stream()), "sb_nhwc_to_nchw")
    _count()
    return out


def nchw_to_nhwc(x: torch.Tensor, out_dtype=_BF16) -> torch.Tensor:
    """[B, C, ...spatial] -> [B*HW, C] token-major."""
    _chk_cuda(x)
    assert x.is_contiguous()
    B, Cc = x.shape[0], x.shape[1]
    HW = x.numel() // (B * Cc)
    out = torch.empty((B * HW, Cc), dtype=out_dtype, device=x.device)
    L = _lib.load()
    _lib.check(L.sb_nchw_to_nhwc(x.data_ptr(), int(x.dtype == _F32), out.data_ptr(), int(out_dtype == _F32),
                                 B, HW, Cc, _stream()), "sb_nchw_to_nhwc")
    _count()
    return out


def add_cast(a: torch.Tensor, b: Optional[torch.Tensor] = None, out_dtype=_BF16) -> torch.Tensor:
    """out = a + b (b fp32, broadcast by flat index modulo b.numel()), converted to out_dtype."""
    _chk_cuda(a, b)
    assert a.is_contiguous() and a.dtype in (_BF16, _F32)
    if VALIDATE_FP32 and out_dtype == _BF16:
        out_dtype = _F32
    out = torch.empty(a.shape, dtype=out_dtype, device=a.device)
    b_mod = 0
    if b is not None:
        assert b.dtype == _F32 and b.is_contiguous()
        b_mod = b.numel() if b.numel() != a.numel() else 0
    L = _lib.load()
    _lib.check(L.sb_add_cast(a.data_ptr(), int(a.dtype == _F32), _ptr(b), b_mod, out.data_ptr(),
                             int(out_dtype == _F32), a.numel(), _stream()), "sb_add_cast")
    _count()
    return out


def prompt_tokens(coords: torch.Tensor, labels: torch.Tensor, gauss: torch.Tensor, point_emb: torch.Tensor,
                  not_a_point: torch.Tensor, out_tokens: torch.Tensor, image_size: int, pad: bool = True) -> torch.Tensor:
    """Decoder token matrix [B, 6 + Np (+1 pad), 256] fp32: output tokens + point-prompt embeddings."""
    _chk_cuda(coords, labels, gauss, point_emb, not_a_point, out_tokens)
    assert coords.dtype == _F32 and coords.is_contiguous() and coords.dim() == 3 and coords.shape[2] == 2
    assert labels.dtype == torch.int32 and labels.is_contiguous() and labels.shape == coords.shape[:2]
    B, Np = coords.shape[0], coords.shape[1]
    Nt = 6 + Np + (1 if pad else 0)
    tokens = torch.empty((B, Nt, 256), dtype=_F32, device=coords.device)
    L = _lib.load()
    _lib.check(L.sb_prompt_tokens(coords.data_ptr(), labels.data_ptr(), B, Np, int(pad), gauss.data_ptr(),
                                  point_emb.data_ptr(), not_a_point.data_ptr(), out_tokens.data_ptr(), image_size,
                                  tokens.data_ptr(), _stream()), "sb_prompt_tokens")
    _count()
    return tokens


def mask_downscale(mask: torch.Tensor, w, clamp: float = 0.0) -> torch.Tensor:
    """Mask prompts -> [B*(S/4)^2, 16] bf16 (mask_downscaling convs 0..5 fused). ``mask`` is [B, S, S] fp32,
    or a decoder output [P, 4, S, S] whose multimask tokens 1..3 become B = 3P prompts (AMG m2m pass).
    clamp > 0 clamps the input to +-clamp first."""
    _chk_cuda(mask)
    assert mask.dtype == _F32 and mask.is_contiguous() and mask.dim() in (3, 4)
    if mask.dim() == 4:
        assert mask.shape[1] == 4
        B, S, cpp = mask.shape[0] * 3, mask.shape[2], 3
    else:
        B, S, cpp = mask.shape[0], mask.shape[1], 1
    out = torch.empty((B * (S // 4) ** 2, 16), dtype=_BF16, device=mask.device)
    L = _lib.load()
    _lib.check(L.sb_mask_downscale(mask.data_ptr(), B, S, cpp, clamp, *[t.data_ptr() for t in w], out.data_ptr(),
                                   _stream()), "sb_mask_downscale")
    _count()
    return out


def select_mask(masks: torch.Tensor, ious: torch.Tensor, delta: float, thresh: float):
    """dynamic_multimask_via_stability: returns (sel_idx int32 [B], sel_iou fp32 [B])."""
    _chk_cuda(masks, ious)
    assert masks.dtype == _F32 and masks.is_contiguous() and masks.dim() == 4 and masks.shape[1] == 4
    assert ious.dtype == _F32 and ious.is_contiguous() and ious.shape == (masks.shape[0], 4)
    B = masks.shape[0]
    idx = torch.empty((B,), dtype=torch.int32, device=masks.device)
    iou = torch.empty((B,), dtype=_F32, device=masks.device)
    L = _lib.load()
    _lib.check(L.sb_select_mask(masks.data_ptr(), ious.data_ptr(), B, masks.shape[2] * masks.shape[3], delta, thresh,
                                idx.data_ptr(), iou.data_ptr(), _stream()), "sb_select_mask")
    _count()
    return idx, iou


# ---------------------------------------------------------------------------------------------
# AMG post-processing (integer / indexing stages) and image-side bandwidth kernels
# ---------------------------------------------------------------------------------------------
_I32, _U8 = torch.int32, torch.uint8


def amg_mask_post(planes: torch.Tensor, ious4: torch.Tensor, sel: Optional[torch.Tensor], cpp: int, n: int,
                  crop_hw, crop_xy, frame_hw, pred_iou_thresh: float, mask_thresh: float, stab_offset: float,
                  stab_thresh: float, keep: torch.Tensor, stability: torch.Tensor, iou_out: torch.Tensor,
                  bbox: torch.Tensor, area: torch.Tensor, bits: torch.Tensor, base: int,
                  geom_dev: Optional[torch.Tensor] = None) -> None:
    """Stability score / threshold / bbox / near-edge test / bit-packing for ``n`` candidates whose low-res
    logits are ``planes`` [B,4,S,S]; results land in slots ``base .. base+n`` of the per-image arrays. With
    ``geom_dev`` (device int32 [5] = Hc, Wc, x0, y0, base) the geometry and slot base are read on the device instead
    (crop_hw / crop_xy / base arguments are ignored) — used under CUDA-graph replay."""
    _chk_cuda(planes, ious4, sel, keep, stability, iou_out, bbox, area, bits)
    assert planes.dtype == _F32 and planes.is_contiguous() and planes.dim() == 4 and planes.shape[1] == 4
    assert ious4.dtype == _F32 and ious4.is_contiguous() and ious4.shape == planes.shape[:2]
    assert sel is None or (sel.dtype == _I32 and sel.is_contiguous())
    assert keep.dtype == _U8 and bbox.dtype == _I32 and area.dtype == _I32 and bits.dtype == _I32
    S = planes.shape[2]
    (Hc, Wc), (x0, y0), (H, W) = crop_hw, crop_xy, frame_hw
    WW = (W + 31) // 32
    assert bits.shape[1:] == (H, WW) and base + n <= bits.shape[0] and n <= planes.shape[0] * cpp
    if geom_dev is not None:
        assert geom_dev.dtype == _I32 and geom_dev.numel() >= 5 and geom_dev.is_cuda
        base = 0
    L = _lib.load()
    rc = L.sb_amg_mask_post(planes.data_ptr(), ious4.data_ptr(), _ptr(sel), cpp, n, S, Hc, Wc, x0, y0, H, W,
                            pred_iou_thresh, mask_thresh, stab_offset, stab_thresh,
                            keep.data_ptr() + base, stability.data_ptr() + 4 * base, iou_out.data_ptr() + 4 * base,
                            bbox.data_ptr() + 16 * base, area.data_ptr() + 4 * base,
                            bits.data_ptr() + 4 * base * H * WW, _ptr(geom_dev), _stream())
    _lib.check(rc, "sb_amg_mask_post")
    _count()


def compact_keep(keep: torch.Tensor, base: int, n: int, cand: torch.Tensor, count: torch.Tensor) -> None:
    _chk_cuda(keep, cand, count)
    assert keep.dtype == _U8 and cand.dtype == _I32 and count.dtype == _I32 and cand.numel() >= n
    L = _lib.load()
    _lib.check(L.sb_compact_keep(keep.data_ptr(), base, n, cand.data_ptr(), count.data_ptr(), _stream()),
               "sb_compact_keep")
    _count()


def nms_dev(bbox: torch.Tensor, scores: torch.Tensor, cand: torch.Tensor, n_ptr: torch.Tensor, n_cap: int,
            iou_thresh: float, order_ws: torch.Tensor, mask_ws: torch.Tensor, out_list: torch.Tensor,
            out_count: torch.Tensor) -> None:
    """torchvision-semantics greedy NMS over candidate slots; appends kept slots to out_list (device counts)."""
    _chk_cuda(bbox, scores, cand, n_ptr, order_ws, mask_ws, out_list, out_count)
    assert bbox.dtype == _I32 and scores.dtype == _F32 and cand.dtype == _I32 and n_ptr.dtype == _I32
    cb = (n_cap + 63) // 64
    assert order_ws.numel() >= n_cap and mask_ws.numel() * mask_ws.element_size() >= n_cap * cb * 8
    L = _lib.load()
    _lib.check(L.sb_nms_dev(bbox.data_ptr(), scores.data_ptr(), cand.data_ptr(), n_ptr.data_ptr(), n_cap, iou_thresh,
                            order_ws.data_ptr(), mask_ws.data_ptr(), out_list.data_ptr(), out_count.data_ptr(),
                            _stream()), "sb_nms_dev")
    _count(3)


def pair_intersections(bits: torch.Tensor, bbox: torch.Tensor, area: torch.Tensor, W: int,
                       area_ratio_thresh: float) -> torch.Tensor:
    """inter[i,j] (i<j) = |mask_i & mask_j| or -1 when the area ratio is below the threshold."""
    _chk_cuda(bits, bbox, area)
    m, H, WW = bits.shape
    assert bits.dtype == _I32 and bits.is_contiguous() and WW == (W + 31) // 32
    assert bbox.dtype == _I32 and bbox.is_contiguous() and bbox.shape == (m, 4)
    assert area.dtype == _I32 and area.is_contiguous() and area.shape == (m,)
    inter = torch.full((m, m), -1, dtype=_I32, device=bits.device)
    L = _lib.load()
    _lib.check(L.sb_pair_intersections(bits.data_ptr(), bbox.data_ptr(), area.data_ptr(), m, H, W,
                                       float(area_ratio_thresh), inter.data_ptr(), _stream()), "sb_pair_intersections")
    _count()
    return inter


def unpack_bits(bits: torch.Tensor, sel: Optional[torch.Tensor], m: int, W: int) -> torch.Tensor:
    """Packed masks [*, H, ceil(W/32)] -> bool [m, H, W] for rows sel[0..m) (or the first m rows)."""
    _chk_cuda(bits, sel)
    H = bits.shape[1]
    out = torch.empty((m, H, W), dtype=torch.bool, device=bits.device)
    if m == 0:
        return out
    L = _lib.load()
    _lib.check(L.sb_unpack_bits(bits.data_ptr(), _ptr(sel), m, H, W, out.data_ptr(), _stream()), "sb_unpack_bits")
    _count()
    return out


def gather_rows(src: torch.Tensor, sel: torch.Tensor, m: int) -> torch.Tensor:
    """dst[k] = src[sel[k]] for 4-byte-element rows (mask bit planes, records)."""
    _chk_cuda(src, sel)
    assert src.is_contiguous() and src.element_size() == 4 and sel.dtype == _I32
    row_words = src[0].numel()
    dst = torch.empty((m,) + tuple(src.shape[1:]), dtype=src.dtype, device=src.device)
    if m == 0:
        return dst
    L = _lib.load()
    _lib.check(L.sb_gather_rows(src.data_ptr(), sel.data_ptr(), m, row_words, dst.data_ptr(), _stream()),
               "sb_gather_rows")
    _count()
    return dst


_SM_COUNT = 148  # B200: the persistent clean-up kernels run at most one CTA per SM


def amg_fill_lowres(planes: torch.Tensor, ious4: torch.Tensor, sel: Optional[torch.Tensor], cpp: int, n: int,
                    pred_iou_thresh: float, mask_threshold: float, max_hole_area: float,
                    max_sprinkle_area: float) -> torch.Tensor:
    """SAM2Transforms.postprocess_masks hole / sprinkle fill of the low-res planes ``n`` candidates use (candidate
    indexing and IoU gate as in ``amg_mask_post``). Returns a new [B,4,S,S] tensor in which only those planes are
    written: components with area <= floor(max_*_area) of (plane <= t) become t + 10, of (plane > t) t - 10."""
    _chk_cuda(planes, ious4, sel)
    assert planes.dtype == _F32 and planes.is_contiguous() and planes.dim() == 4 and planes.shape[1] == 4
    assert ious4.dtype == _F32 and ious4.is_contiguous() and ious4.shape == planes.shape[:2]
    assert sel is None or (sel.dtype == _I32 and sel.is_contiguous())
    assert 0 < n <= planes.shape[0] * cpp
    S = planes.shape[2]
    hole = int(math.floor(max_hole_area)) if max_hole_area > 0 else 0
    sprinkle = int(math.floor(max_sprinkle_area)) if max_sprinkle_area > 0 else 0
    out = torch.empty_like(planes)
    ctas = min(n, _SM_COUNT)
    ws = torch.empty((ctas * S * S,), dtype=_I32, device=planes.device)
    L = _lib.load()
    # the fill values are float32(t +/- 10.0) evaluated in double, as torch.where casts the Python scalar
    _lib.check(L.sb_amg_fill_lowres(planes.data_ptr(), ious4.data_ptr(), _ptr(sel), cpp, n, S, pred_iou_thresh,
                                    mask_threshold, hole, sprinkle, float(mask_threshold) + 10.0,
                                    float(mask_threshold) - 10.0, out.data_ptr(), ws.data_ptr(), ctas, _stream()),
               "sb_amg_fill_lowres")
    _count()
    return out


def small_regions_workspace(H: int, W: int, device, budget_bytes: int = 256 << 20) -> torch.Tensor:
    """Workspace of ``amg_small_regions`` for (H, W) frames: 32 H ceil(W/32) int32 per CTA, as many CTAs (at most one
    per SM) as fit the budget. Its size does not depend on the number of masks."""
    per_cta = 32 * H * ((W + 31) // 32)
    ctas = max(1, min(_SM_COUNT, budget_bytes // (4 * per_cta)))
    return torch.empty((ctas * per_cta,), dtype=_I32, device=device)


def amg_small_regions(bits: torch.Tensor, rows: Optional[torch.Tensor], m: int, W: int, min_area: float,
                      box: torch.Tensor, area: torch.Tensor, score: torch.Tensor, box_changed: Optional[torch.Tensor],
                      ws: torch.Tensor) -> None:
    """Upstream remove_small_regions("holes") then ("islands") with ``min_area`` on the packed masks rows[0..m) (or the
    first m) of ``bits`` [*, H, ceil(W/32)], in place. Per mask row: box (xyxy, zero when empty), area and score
    (1.0 unchanged / 0.0 changed); box_changed receives the box of changed masks only."""
    _chk_cuda(bits, rows, box, area, score, box_changed, ws)
    H, WW = bits.shape[1], bits.shape[2]
    assert bits.dtype == _I32 and bits.is_contiguous() and WW == (W + 31) // 32
    assert rows is None or (rows.dtype == _I32 and rows.numel() >= m)
    assert box.dtype == _I32 and area.dtype == _I32 and score.dtype == _F32 and ws.dtype == _I32
    assert box_changed is None or box_changed.dtype == _I32
    assert min_area > 0 and m > 0
    per_cta = 32 * H * WW
    assert ws.numel() >= per_cta
    L = _lib.load()
    _lib.check(L.sb_amg_small_regions(bits.data_ptr(), _ptr(rows), m, H, W, int(math.ceil(min_area)) - 1,
                                      box.data_ptr(), area.data_ptr(), score.data_ptr(), _ptr(box_changed),
                                      ws.data_ptr(), ws.numel() // per_cta, _stream()), "sb_amg_small_regions")
    _count()


def masks_to_rle(bits: torch.Tensor, sel: Optional[torch.Tensor], m: int, W: int, coco: bool = False):
    """Run-length encoding of the packed masks [*, H, ceil(W/32)] rows sel[0..m) (or the first m), on the device.
    Returns (data, offsets) with offsets [m+1] int64: the encoding of mask k is data[offsets[k]:offsets[k+1]], int32
    counts of upstream's mask_to_rle_pytorch, or with ``coco`` the uint8 characters of pycocotools' rleToString.
    Reads each total back with one host synchronisation."""
    _chk_cuda(bits, sel)
    H, WW = bits.shape[1], bits.shape[2]
    assert bits.dtype == _I32 and bits.is_contiguous() and WW == (W + 31) // 32
    assert sel is None or (sel.dtype == _I32 and sel.is_contiguous() and sel.numel() >= m)
    assert sel is not None or bits.shape[0] >= m
    dev = bits.device
    offsets = torch.zeros((m + 1,), dtype=torch.int64, device=dev)
    if m == 0:
        return torch.empty((0,), dtype=torch.uint8 if coco else _I32, device=dev), offsets
    L = _lib.load()
    ws = torch.empty((2 * m * W,), dtype=_I32, device=dev)
    _lib.check(L.sb_masks_rle_size(bits.data_ptr(), _ptr(sel), m, H, W, ws.data_ptr(), offsets.data_ptr(), _stream()),
               "sb_masks_rle_size")
    counts = torch.empty((int(offsets[m].item()),), dtype=_I32, device=dev)
    _lib.check(L.sb_masks_rle_counts(bits.data_ptr(), _ptr(sel), m, H, W, ws.data_ptr(), offsets.data_ptr(),
                                     counts.data_ptr(), _stream()), "sb_masks_rle_counts")
    _count(4)
    if not coco:
        return counts, offsets
    coff = torch.zeros((m + 1,), dtype=torch.int64, device=dev)
    _lib.check(L.sb_masks_rle_coco_size(counts.data_ptr(), offsets.data_ptr(), m, coff.data_ptr(), _stream()),
               "sb_masks_rle_coco_size")
    chars = torch.empty((int(coff[m].item()),), dtype=torch.uint8, device=dev)
    _lib.check(L.sb_masks_rle_coco(counts.data_ptr(), offsets.data_ptr(), m, coff.data_ptr(), chars.data_ptr(),
                                   _stream()), "sb_masks_rle_coco")
    _count(3)
    return chars, coff


def prepare_slice(img: torch.Tensor, box: int = 500, cutoff: float = 3.0) -> torch.Tensor:
    """REF saber/utils/preprocessing.py:67-81 ``prepare`` on one [H, W] fp32 slice -> [H, W] fp32 in [0,1]
    (the three RGB channels SABER feeds SAM2 are identical copies of it)."""
    _chk_cuda(img)
    assert img.dtype == _F32 and img.is_contiguous() and img.dim() == 2
    H, W = img.shape
    L = _lib.load()
    t0 = torch.empty_like(img)
    mean = torch.empty_like(img)
    sq = torch.empty_like(img)
    s = _stream()
    _lib.check(L.sb_box_filter(img.data_ptr(), t0.data_ptr(), H, W, 0, box, 0, s), "sb_box_filter")
    _lib.check(L.sb_box_filter(t0.data_ptr(), mean.data_ptr(), H, W, 1, box, 0, s), "sb_box_filter")
    _lib.check(L.sb_box_filter(img.data_ptr(), t0.data_ptr(), H, W, 0, box, 1, s), "sb_box_filter")
    _lib.check(L.sb_box_filter(t0.data_ptr(), sq.data_ptr(), H, W, 1, box, 0, s), "sb_box_filter")
    partials = torch.empty((2048,), dtype=_F32, device=img.device)
    _lib.check(L.sb_contrast_normalize(img.data_ptr(), mean.data_ptr(), sq.data_ptr(), t0.data_ptr(), img.numel(),
                                       cutoff, partials.data_ptr(), s), "sb_contrast_normalize")
    _count(6)
    return t0


def prepare_rgb(img: torch.Tensor, channel_mix, box: int = 500, cutoff: float = 3.0) -> torch.Tensor:
    """``prepare`` on an (H,W,3) fp32 image as the reference computes it for 3-D input (REF saber/utils/preprocessing.py:
    4-37,67-81): box filter over ALL three axes (the channel axis = the constant 3x3 ``channel_mix``), z-score, clip,
    global min-max. -> (H,W,3) fp32 in [0,1]."""
    _chk_cuda(img)
    assert img.dtype == _F32 and img.is_contiguous() and img.dim() == 3 and img.shape[2] == 3
    H, W, _ = img.shape
    n = H * W
    dev = img.device
    L = _lib.load()
    s = _stream()
    mix = torch.as_tensor(channel_mix, dtype=_F32).reshape(9).to(dev)
    eye = torch.eye(3, dtype=_F32).reshape(9).to(dev)
    planar = torch.empty((3, H, W), dtype=_F32, device=dev)
    m0 = torch.empty_like(planar)
    t0 = torch.empty((H, W), dtype=_F32, device=dev)
    mean = torch.empty_like(planar)
    sq = torch.empty_like(planar)
    _lib.check(L.sb_rgb_mix_planar(img.data_ptr(), eye.data_ptr(), 0, n, planar.data_ptr(), s), "sb_rgb_mix_planar")
    for square, dst in ((0, mean), (1, sq)):
        _lib.check(L.sb_rgb_mix_planar(img.data_ptr(), mix.data_ptr(), square, n, m0.data_ptr(), s), "sb_rgb_mix_planar")
        for c in range(3):
            _lib.check(L.sb_box_filter(m0[c].data_ptr(), t0.data_ptr(), H, W, 0, box, 0, s), "sb_box_filter")
            _lib.check(L.sb_box_filter(t0.data_ptr(), dst[c].data_ptr(), H, W, 1, box, 0, s), "sb_box_filter")
    partials = torch.empty((2048,), dtype=_F32, device=dev)
    _lib.check(L.sb_contrast_normalize(planar.data_ptr(), mean.data_ptr(), sq.data_ptr(), m0.data_ptr(), 3 * n, cutoff,
                                       partials.data_ptr(), s), "sb_contrast_normalize")
    out = torch.empty_like(img)
    _lib.check(L.sb_planar_to_hwc3(m0.data_ptr(), n, out.data_ptr(), s), "sb_planar_to_hwc3")
    _count(18)
    return out


_MEAN3 = (0.485, 0.456, 0.406)
_STD3 = (0.229, 0.224, 0.225)


def resize_normalize(img: torch.Tensor, crops: torch.Tensor, S: int = 1024, mean=_MEAN3, std=_STD3) -> torch.Tensor:
    """img [H,W] or [H,W,3] fp32, crops int32 [n,4] (x0,y0,x1,y1) -> [n,3,S,S] fp32 (SAM2Transforms)."""
    _chk_cuda(img, crops)
    assert img.dtype == _F32 and img.is_contiguous() and img.dim() in (2, 3)
    assert crops.dtype == _I32 and crops.is_contiguous() and crops.dim() == 2 and crops.shape[1] == 4
    H, W = img.shape[:2]
    Cc = 1 if img.dim() == 2 else img.shape[2]
    n = crops.shape[0]
    out = torch.empty((n, 3, S, S), dtype=_F32, device=img.device)
    import ctypes as _C
    m3 = (_C.c_float * 3)(*mean)
    s3 = (_C.c_float * 3)(*std)
    L = _lib.load()
    _lib.check(L.sb_resize_normalize(img.data_ptr(), H, W, Cc, crops.data_ptr(), n, S, m3, s3, out.data_ptr(),
                                     _stream()), "sb_resize_normalize")
    _count()
    return out


def stitch_labels(bits: torch.Tensor, order: Optional[torch.Tensor], m: int, W: int,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """labels[y,x] = 1 + max{k : mask order[k] covers (y,x)} (uint16; 0 = background)."""
    _chk_cuda(bits, order, out)
    H = bits.shape[1]
    if out is None:
        out = torch.empty((H, W), dtype=torch.int16, device=bits.device)  # uint16 payload in int16 storage
    assert out.dtype in (torch.int16, torch.uint16) and out.is_contiguous() and out.shape == (H, W)
    L = _lib.load()
    _lib.check(L.sb_stitch_labels(bits.data_ptr(), _ptr(order), m, H, W, out.data_ptr(), _stream()),
               "sb_stitch_labels")
    _count()
    return out


def ccl3d_26(vol: torch.Tensor, min_vol: int):
    """26-connected components of vol != 0 with components < min_vol voxels dropped and compact raster-order
    labels (REF saber/segmenters/utils.py:88-131). Returns (labels int32-as-uint32 [Z,Y,X], n_components tensor)."""
    _chk_cuda(vol)
    assert vol.is_contiguous() and vol.dim() == 3 and vol.element_size() in (1, 2, 4)
    Z, Y, X = vol.shape
    n = vol.numel()
    labels = torch.empty((Z, Y, X), dtype=_I32, device=vol.device)
    aux = torch.empty((n,), dtype=_I32, device=vol.device)
    nchunks = (n + 2047) // 2048
    chunk_ws = torch.empty((nchunks + 1,), dtype=_I32, device=vol.device)
    L = _lib.load()
    _lib.check(L.sb_ccl3d_26(vol.data_ptr(), vol.element_size(), Z, Y, X, int(min_vol), labels.data_ptr(),
                             aux.data_ptr(), chunk_ws.data_ptr(), _stream()), "sb_ccl3d_26")
    _count(7)
    return labels, chunk_ws[nchunks:]


def ccl3d(vol: torch.Tensor, min_vol: int = 1, conn: int = 6, with_sizes: bool = False):
    """Connected components of vol != 0 with connectivity 6 (scipy.ndimage.label's default) or 26, components with fewer
    than min_vol voxels dropped, compact labels in raster order of their first voxel. Returns (labels int32 [Z,Y,X],
    count tensor [1], sizes int32 [capacity] or None — sizes[id - 1] = voxels of component id)."""
    _chk_cuda(vol)
    assert vol.is_contiguous() and vol.dim() == 3 and vol.element_size() in (1, 2, 4)
    Z, Y, X = vol.shape
    n = vol.numel()
    labels = torch.empty((Z, Y, X), dtype=_I32, device=vol.device)
    aux = torch.empty((n,), dtype=_I32, device=vol.device)
    nchunks = (n + 2047) // 2048
    chunk_ws = torch.empty((nchunks + 1,), dtype=_I32, device=vol.device)
    sizes = torch.zeros((n // max(1, int(min_vol)) + 1,), dtype=_I32, device=vol.device) if with_sizes else None
    L = _lib.load()
    _lib.check(L.sb_ccl3d(vol.data_ptr(), vol.element_size(), Z, Y, X, int(min_vol), int(conn), labels.data_ptr(),
                          aux.data_ptr(), chunk_ws.data_ptr(), _ptr(sizes), _stream()), "sb_ccl3d")
    _count(7)
    return labels, chunk_ws[nchunks:], sizes


def upsample_bilinear(x: torch.Tensor, Ho: int, Wo: int) -> torch.Tensor:
    """[..., Hi, Wi] fp32 -> [..., Ho, Wo] fp32 (F.interpolate bilinear, align_corners=False)."""
    _chk_cuda(x)
    assert x.dtype == _F32 and x.is_contiguous() and x.dim() >= 2
    Hi, Wi = x.shape[-2:]
    N = x.numel() // (Hi * Wi)
    out = torch.empty(tuple(x.shape[:-2]) + (Ho, Wo), dtype=_F32, device=x.device)
    L = _lib.load()
    _lib.check(L.sb_upsample_bilinear(x.data_ptr(), N, Hi, Wi, Ho, Wo, out.data_ptr(), _stream()),
               "sb_upsample_bilinear")
    _count()
    return out


def upsample_select(planes: torch.Tensor, sel: Optional[torch.Tensor], cpp: int, Ho: int, Wo: int,
                    threshold: float = 0.0, logits: bool = False) -> torch.Tensor:
    """Decoder planes [P,4,S,S] -> [P, cpp, Ho, Wo] in one kernel: the selected planes (tokens 1..3 for cpp = 3, else the
    ``sel`` choice or token 0) up-sampled bit-identically to ``upsample_bilinear``, as fp32 logits or as bool
    ``value > threshold`` masks."""
    _chk_cuda(planes, sel)
    assert planes.dtype == _F32 and planes.is_contiguous() and planes.dim() == 4 and planes.shape[1] == 4
    assert sel is None or (sel.dtype == _I32 and sel.is_contiguous() and sel.numel() == planes.shape[0])
    assert cpp in (1, 3) and not (cpp == 3 and sel is not None)
    P, S = planes.shape[0], planes.shape[2]
    out = torch.empty((P, cpp, Ho, Wo), dtype=_F32 if logits else torch.bool, device=planes.device)
    L = _lib.load()
    _lib.check(L.sb_upsample_select(planes.data_ptr(), P, S, _ptr(sel), cpp, Ho, Wo, float(threshold), int(logits),
                                    out.data_ptr(), _stream()), "sb_upsample_select")
    _count()
    return out


_frame_coeff_cache: dict = {}


def pillow_bicubic_coeffs(n_in: int, n_out: int):
    """Pillow's 8-bit BICUBIC coefficients (libImaging/Resample.c precompute_coeffs + normalize_coeffs_8bpc) in float64
    with Pillow's order of operations -> (bounds int32 [n_out, 2] = (xmin, n), weights int32 [n_out, ksize])."""
    import numpy as np
    scale = n_in / n_out
    fs = max(scale, 1.0)
    support = 2.0 * fs
    ksize = int(math.ceil(support)) * 2 + 1
    center = (np.arange(n_out, dtype=np.float64) + 0.5) * scale
    xmin = np.maximum((center - support + 0.5).astype(np.int64), 0)  # C (int) truncates toward zero, as astype does
    n = np.minimum((center + support + 0.5).astype(np.int64), n_in) - xmin
    k = np.arange(ksize)
    t = np.abs((k[None, :] + xmin[:, None] - center[:, None] + 0.5) * (1.0 / fs))
    a = -0.5
    w = np.where(t < 1.0, ((a + 2.0) * t - (a + 3.0)) * t * t + 1,
                 np.where(t < 2.0, (((t - 5) * t + 8) * t - 4) * a, 0.0))
    w = np.where(k[None, :] < n[:, None], w, 0.0)
    ww = np.zeros(n_out)
    for j in range(ksize):  # Pillow sums the taps in order (numpy's pairwise sum would round differently)
        ww = ww + w[:, j]
    w = np.where(ww[:, None] != 0.0, w / np.where(ww == 0.0, 1.0, ww)[:, None], w)
    fixed = np.where(w < 0, -0.5 + w * (1 << 22), 0.5 + w * (1 << 22)).astype(np.int64)
    return np.stack([xmin, n], 1).astype(np.int32), fixed.astype(np.int32)


def _frame_coeffs(n_in: int, n_out: int, device):
    """Device coefficient tables of one axis, cached per (n_in, n_out, device): (bounds, weights, ksize, first, last),
    with [first, last) the source range the taps reach. n_in == n_out gives the one-tap identity (pass skipped)."""
    key = (n_in, n_out, str(device))
    c = _frame_coeff_cache.get(key)
    if c is None:
        import numpy as np
        if n_in == n_out:
            b = np.stack([np.arange(n_out), np.ones(n_out, np.int64)], 1).astype(np.int32)
            w = np.full((n_out, 1), 1 << 22, np.int32)
        else:
            b, w = pillow_bicubic_coeffs(n_in, n_out)
        c = (torch.from_numpy(b).to(device), torch.from_numpy(np.ascontiguousarray(w)).to(device), w.shape[1],
             int(b[0, 0]), int(b[-1, 0] + b[-1, 1]))
        _frame_coeff_cache[key] = c
    return c


def resample_frames_u8(frames: torch.Tensor, S: int, lut: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """uint8 RGB frames [N, H, W, 3] of one size -> fp32 [N, 3, S, S]: Pillow's ``Image.resize((S, S))`` (bicubic,
    8-bit fixed point) bit for bit, then ``lut[c, byte]`` ([3, 256] fp32). ``out``: optional contiguous destination."""
    _chk_cuda(frames, lut, out)
    assert frames.dtype == torch.uint8 and frames.is_contiguous() and frames.dim() == 4 and frames.shape[3] == 3
    assert lut.dtype == _F32 and lut.is_contiguous() and lut.numel() == 3 * 256
    N, H, W, _ = frames.shape
    if out is None:
        out = torch.empty((N, 3, S, S), dtype=_F32, device=frames.device)
    assert out.dtype == _F32 and out.is_contiguous() and tuple(out.shape) == (N, 3, S, S)
    yb, yw, yk, y0, y1 = _frame_coeffs(H, S, frames.device)
    xb = xw = tmp = None
    xk = 0
    if W != S:
        xb, xw, xk, _, _ = _frame_coeffs(W, S, frames.device)
        tmp = torch.empty((N, y1 - y0, S, 3), dtype=torch.uint8, device=frames.device)
    L = _lib.load()
    _lib.check(L.sb_resample_frames_u8(frames.data_ptr(), N, H, W, S, _ptr(xb), _ptr(xw), xk, yb.data_ptr(), yw.data_ptr(),
                                       yk, y0, y1 - y0, _ptr(tmp), lut.data_ptr(), out.data_ptr(), _stream()),
               "sb_resample_frames_u8")
    _count(2 if tmp is not None else 1)
    return out


# ---------------------------------------------------------------------------------------------
# z-axis propagation: memory attention / memory encoder / tracking glue (csrc/memory.cu)
# ---------------------------------------------------------------------------------------------
def rope_apply(x: torch.Tensor, cos_sin: torch.Tensor, rows_per_batch: int, n_rope: Optional[int] = None,
               out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Axial RoPE on a projected q / k matrix [batch*rows_per_batch, C] (fp32 or bf16 view) -> bf16. Rows
    r < n_rope of each batch entry use token r % ntok's frequencies; the rest are copied. cos_sin [ntok, C/2, 2] fp32."""
    _chk_cuda(x, cos_sin, out)
    assert x.dim() == 2 and x.stride(1) == 1 and x.dtype in (_BF16, _F32)
    rows, Cc = x.shape
    assert cos_sin.dtype == _F32 and cos_sin.is_contiguous() and cos_sin.shape[1:] == (Cc // 2, 2)
    if n_rope is None:
        n_rope = rows_per_batch
    if VALIDATE_FP32 and out is None:
        assert x.dtype == _F32
        out = torch.empty((rows, Cc), dtype=_F32, device=x.device)
        L = _lib.load()
        _lib.check(L.sb_rope_apply_f32(x.data_ptr(), x.stride(0), out.data_ptr(), out.stride(0), rows, Cc, rows_per_batch,
                                       n_rope, cos_sin.shape[0], cos_sin.data_ptr(), _stream()), "sb_rope_apply_f32")
        _count()
        return out
    if out is None:
        out = torch.empty((rows, Cc), dtype=_BF16, device=x.device)
    L = _lib.load()
    _lib.check(L.sb_rope_apply(x.data_ptr(), x.stride(0), int(x.dtype == _F32), out.data_ptr(), out.stride(0), rows, Cc,
                               rows_per_batch, n_rope, cos_sin.shape[0], cos_sin.data_ptr(), _stream()), "sb_rope_apply")
    _count()
    return out


def conv3x3s2_ln_gelu(x: torch.Tensor, stage: int, w, bias, gamma, beta, eps: float = 1e-6, in_xf: int = 0,
                      xf_scale: float = 20.0, xf_bias: float = -10.0) -> torch.Tensor:
    """One MaskDownSampler stage on NHWC input [B, H, W, Cin] -> bf16 [B, H/2, W/2, Cout]."""
    _chk_cuda(x, w, bias, gamma, beta)
    cin, cout = ((1, 4), (4, 16), (16, 64))[stage]
    assert x.is_contiguous() and x.dim() == 4 and x.shape[3] == cin and x.dtype == (_F32 if stage == 0 else _BF16)
    assert w.dtype == _F32 and w.is_contiguous() and w.numel() == cout * cin * 9
    B, H, W = x.shape[:3]
    out = torch.empty((B, (H + 1) // 2, (W + 1) // 2, cout), dtype=_BF16, device=x.device)
    L = _lib.load()
    _lib.check(L.sb_conv3x3s2_ln_gelu(x.data_ptr(), stage, B, H, W, w.data_ptr(), bias.data_ptr(), gamma.data_ptr(),
                                      beta.data_ptr(), eps, in_xf, xf_scale, xf_bias, out.data_ptr(), _stream()),
               "sb_conv3x3s2_ln_gelu")
    _count()
    return out


def im2col_3x3s2(x: torch.Tensor) -> torch.Tensor:
    """NHWC bf16 [B, H, W, C] -> [B*(H/2)*(W/2), 9*C] patches of a 3x3 stride-2 pad-1 conv (column = (ky*3+kx)*C + c)."""
    _chk_cuda(x)
    assert x.dtype == _BF16 and x.is_contiguous() and x.dim() == 4
    B, H, W, Cc = x.shape
    cols = torch.empty((B * ((H + 1) // 2) * ((W + 1) // 2), 9 * Cc), dtype=_BF16, device=x.device)
    L = _lib.load()
    _lib.check(L.sb_im2col_3x3s2(x.data_ptr(), B, H, W, Cc, cols.data_ptr(), _stream()), "sb_im2col_3x3s2")
    _count()
    return cols


def dwconv7_ln(x: torch.Tensor, B: int, H: int, W: int, w, bias, gamma, beta, eps: float = 1e-6) -> torch.Tensor:
    """CXBlock front half on token-major fp32 [B*H*W, 256] -> bf16."""
    _chk_cuda(x, w, bias, gamma, beta)
    assert x.dtype == _F32 and x.is_contiguous() and x.shape == (B * H * W, 256)
    out = torch.empty((B * H * W, 256), dtype=_BF16, device=x.device)
    L = _lib.load()
    _lib.check(L.sb_dwconv7_ln(x.data_ptr(), B, H, W, 256, w.data_ptr(), bias.data_ptr(), gamma.data_ptr(),
                               beta.data_ptr(), eps, out.data_ptr(), _stream()), "sb_dwconv7_ln")
    _count()
    return out


def add_vec_cond(x: torch.Tensor, score: torch.Tensor, vec: torch.Tensor, B: int) -> torch.Tensor:
    """bf16(x[b] + (score[b] <= 0) * vec) for x fp32 [B*rows, C]."""
    _chk_cuda(x, score, vec)
    assert x.dtype == _F32 and x.is_contiguous() and score.dtype == _F32 and score.numel() == B
    rows = x.shape[0] // B
    out = torch.empty(x.shape, dtype=_BF16, device=x.device)
    L = _lib.load()
    _lib.check(L.sb_add_vec_cond(x.data_ptr(), score.data_ptr(), vec.data_ptr(), B, rows, x.shape[1], out.data_ptr(),
                                 _stream()), "sb_add_vec_cond")
    _count()
    return out


def track_select(masks: torch.Tensor, ious: torch.Tensor, obj: torch.Tensor, hs: torch.Tensor,
                 sel: Optional[torch.Tensor], multimask: bool):
    """-> (low_res [B,S,S] fp32 gated by the object score, token [B,256] fp32, plane index int32 [B])."""
    _chk_cuda(masks, ious, obj, hs, sel)
    B, _, S, _ = masks.shape
    Nt = hs.shape[1]
    assert masks.dtype == _F32 and masks.is_contiguous() and ious.is_contiguous() and hs.is_contiguous() and hs.dtype == _F32
    low = torch.empty((B, S, S), dtype=_F32, device=masks.device)
    tok = torch.empty((B, 256), dtype=_F32, device=masks.device)
    best = torch.empty((B,), dtype=_I32, device=masks.device)
    L = _lib.load()
    _lib.check(L.sb_track_select(masks.data_ptr(), ious.data_ptr(), obj.data_ptr(), hs.data_ptr(), _ptr(sel),
                                 int(multimask), B, Nt, S, low.data_ptr(), tok.data_ptr(), best.data_ptr(), _stream()),
               "sb_track_select")
    _count()
    return low, tok, best


def objptr_mix_(ptr: torch.Tensor, cond: torch.Tensor, no_obj_ptr: torch.Tensor) -> torch.Tensor:
    _chk_cuda(ptr, cond, no_obj_ptr)
    assert ptr.dtype == _F32 and ptr.is_contiguous() and cond.dtype == _F32
    L = _lib.load()
    _lib.check(L.sb_objptr_mix(ptr.data_ptr(), cond.data_ptr(), no_obj_ptr.data_ptr(), ptr.shape[0], ptr.shape[1],
                               _stream()), "sb_objptr_mix")
    _count()
    return ptr


def fill_holes(masks: torch.Tensor, max_area: int) -> torch.Tensor:
    """[B, S, S] fp32 mask scores -> holes (8-connected background components, area <= max_area) set to 0.1."""
    _chk_cuda(masks)
    assert masks.dtype == _F32 and masks.is_contiguous() and masks.dim() == 3 and masks.shape[1] == masks.shape[2]
    B, S, _ = masks.shape
    out = torch.empty_like(masks)
    ws = torch.empty((B * 2 * S * S,), dtype=_I32, device=masks.device)
    L = _lib.load()
    _lib.check(L.sb_fill_holes(masks.data_ptr(), out.data_ptr(), B, S, int(max_area), ws.data_ptr(), _stream()),
               "sb_fill_holes")
    _count()
    return out


def threshold_affine(x: torch.Tensor, thr: float, scale: float, bias: float) -> torch.Tensor:
    _chk_cuda(x)
    assert x.dtype == _F32 and x.is_contiguous()
    out = torch.empty_like(x)
    L = _lib.load()
    _lib.check(L.sb_threshold_affine(x.data_ptr(), thr, scale, bias, x.numel(), out.data_ptr(), _stream()),
               "sb_threshold_affine")
    _count()
    return out


def conv4x4s4(x: torch.Tensor, w: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """SAM2Base.mask_downsample on [B, S, S] fp32 -> [B, S/4, S/4]."""
    _chk_cuda(x, w, bias)
    assert x.dtype == _F32 and x.is_contiguous() and x.dim() == 3
    B, S, _ = x.shape
    out = torch.empty((B, S // 4, S // 4), dtype=_F32, device=x.device)
    L = _lib.load()
    _lib.check(L.sb_conv4x4s4(x.data_ptr(), B, S, w.data_ptr(), bias.data_ptr(), out.data_ptr(), _stream()), "sb_conv4x4s4")
    _count()
    return out


def stitch_objects_(logits: torch.Tensor, ids: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
    """labels (uint16-in-int16 [H, W], in place) <- ids[i] where object i's video-resolution logits are > 0."""
    _chk_cuda(logits, ids, labels)
    assert logits.dtype == _F32 and logits.is_contiguous() and logits.dim() == 3 and logits.shape[1] == logits.shape[2]
    assert ids.dtype == _I32 and ids.numel() == logits.shape[0] and labels.is_contiguous() and labels.element_size() == 2
    H, W = labels.shape
    L = _lib.load()
    _lib.check(L.sb_stitch_objects(logits.data_ptr(), ids.data_ptr(), logits.shape[0], logits.shape[1], H, W,
                                   labels.data_ptr(), _stream()), "sb_stitch_objects")
    _count()
    return labels


def slice_any(vol: torch.Tensor) -> torch.Tensor:
    _chk_cuda(vol)
    assert vol.is_contiguous() and vol.element_size() == 2 and vol.dim() == 3
    out = torch.empty((vol.shape[0],), dtype=_U8, device=vol.device)
    L = _lib.load()
    _lib.check(L.sb_slice_any(vol.data_ptr(), vol.shape[0], vol.shape[1] * vol.shape[2], out.data_ptr(), _stream()),
               "sb_slice_any")
    _count()
    return out


def erase_label_(labels: torch.Tensor, obj_id: int) -> None:
    _chk_cuda(labels)
    assert labels.is_contiguous() and labels.element_size() == 2
    L = _lib.load()
    _lib.check(L.sb_erase_label(labels.data_ptr(), labels.numel(), int(obj_id), _stream()), "sb_erase_label")
    _count()


# ---------------------------------------------------------------------------------------------
# whole-tomogram bandwidth kernels of the 3-D path (csrc/volume.cu)
# ---------------------------------------------------------------------------------------------
def minmax(x: torch.Tensor) -> torch.Tensor:
    """-> device fp32 [2] = (min, max) of x (no host synchronisation)."""
    _chk_cuda(x)
    assert x.dtype == _F32 and x.is_contiguous()
    mm = torch.empty((2,), dtype=_F32, device=x.device)
    partials = torch.empty((2048,), dtype=_F32, device=x.device)
    L = _lib.load()
    _lib.check(L.sb_minmax(x.data_ptr(), x.numel(), mm.data_ptr(), partials.data_ptr(), _stream()), "sb_minmax")
    _count(2)
    return mm


def minmax_affine(x: torch.Tensor, mm: torch.Tensor, eps: float, a: float, b: float) -> torch.Tensor:
    """((x - mm[0]) / ((mm[1] - mm[0]) + eps)) * a + b with mm on the device."""
    _chk_cuda(x, mm)
    assert x.dtype == _F32 and x.is_contiguous() and mm.dtype == _F32 and mm.numel() == 2
    out = torch.empty_like(x)
    L = _lib.load()
    _lib.check(L.sb_minmax_affine(x.data_ptr(), x.numel(), mm.data_ptr(), eps, a, b, out.data_ptr(), _stream()),
               "sb_minmax_affine")
    _count()
    return out


def skimage_resize_stack(vol: torch.Tensor, S: int, a: float = 1.0, b: float = 0.0) -> torch.Tensor:
    """skimage.transform.resize(slice, (S, S), anti_aliasing=True) for every slice of vol [Z,H,W] fp32, then a*v + b."""
    _chk_cuda(vol)
    assert vol.dtype == _F32 and vol.is_contiguous() and vol.dim() == 3
    Z, H, W = vol.shape
    L = _lib.load()
    src = vol
    for axis, n in ((1, H), (2, W)):  # scipy.ndimage.gaussian_filter filters axis 0 of the slice first, then axis 1
        sigma = max(0.0, (n / S - 1) / 2)
        if sigma > 0:
            r = int(4.0 * sigma + 0.5)
            xs = torch.arange(-r, r + 1, dtype=torch.float64)
            w = torch.exp(-0.5 / (sigma * sigma) * xs ** 2)
            w = (w / w.sum()).to(vol.device)
            dst = torch.empty_like(src)
            _lib.check(L.sb_gauss1d_mirror(src.data_ptr(), Z, H, W, axis, w.data_ptr(), r, dst.data_ptr(), _stream()),
                       "sb_gauss1d_mirror")
            _count()
            src = dst
    out = torch.empty((Z, S, S), dtype=_F32, device=vol.device)
    _lib.check(L.sb_zoom_linear_mirror(src.data_ptr(), Z, H, W, S, S, a, b, out.data_ptr(), _stream()),
               "sb_zoom_linear_mirror")
    _count()
    return out


def gaussian_z(vol: torch.Tensor, weights: torch.Tensor) -> torch.Tensor:
    """Zero-padded 1-D correlation along z of vol [Z,Y,X] fp32 with `weights` (odd length, fp32, device)."""
    _chk_cuda(vol, weights)
    assert vol.dtype == _F32 and vol.is_contiguous() and vol.dim() == 3 and weights.dtype == _F32
    out = torch.empty_like(vol)
    L = _lib.load()
    _lib.check(L.sb_gaussian_z(vol.data_ptr(), vol.shape[0], vol.shape[1] * vol.shape[2], weights.data_ptr(),
                               weights.numel(), out.data_ptr(), _stream()), "sb_gaussian_z")
    _count()
    return out


def mean_z(vol: torch.Tensor, z0: int, z1: int) -> torch.Tensor:
    _chk_cuda(vol)
    assert vol.dtype == _F32 and vol.is_contiguous() and vol.dim() == 3 and 0 <= z0 < z1 <= vol.shape[0]
    out = torch.empty(vol.shape[1:], dtype=_F32, device=vol.device)
    L = _lib.load()
    _lib.check(L.sb_mean_z(vol.data_ptr(), vol.shape[1] * vol.shape[2], z0, z1, out.data_ptr(), _stream()), "sb_mean_z")
    _count()
    return out


# ---------------------------------------------------------------------------------------------
# expert classifier kernels (csrc/classifier.cu)
# ---------------------------------------------------------------------------------------------
def standardize(x: torch.Tensor) -> torch.Tensor:
    """monai NormalizeIntensity(): (x - mean) / std (population std; no division when std == 0)."""
    _chk_cuda(x)
    assert x.dtype == _F32 and x.is_contiguous()
    ms = torch.empty((2,), dtype=_F32, device=x.device)
    ws = torch.empty((2048,), dtype=torch.float64, device=x.device)
    out = torch.empty_like(x)
    L = _lib.load()
    _lib.check(L.sb_mean_std(x.data_ptr(), x.numel(), ms.data_ptr(), ws.data_ptr(), _stream()), "sb_mean_std")
    _lib.check(L.sb_standardize(x.data_ptr(), x.numel(), ms.data_ptr(), out.data_ptr(), _stream()), "sb_standardize")
    _count(3)
    return out


def mask_bbox(masks: torch.Tensor) -> torch.Tensor:
    """masks uint8 [N,H,W] -> int32 [N,4] (y_min, y_max, x_min, x_max), -1 for empty masks."""
    _chk_cuda(masks)
    assert masks.dtype == _U8 and masks.is_contiguous() and masks.dim() == 3
    N, H, W = masks.shape
    out = torch.empty((N, 4), dtype=_I32, device=masks.device)
    L = _lib.load()
    _lib.check(L.sb_mask_bbox(masks.data_ptr(), N, H, W, out.data_ptr(), _stream()), "sb_mask_bbox")
    _count()
    return out


def crop_resize(img: torch.Tensor, masks: torch.Tensor, geom: torch.Tensor, S: int):
    """-> (images fp32 [N,S,S], masks uint8 [N,S,S], areas int32 [N]) for crops geom[n] = (top, left, h, w)."""
    _chk_cuda(img, masks, geom)
    assert img.dtype == _F32 and img.is_contiguous() and img.dim() == 2 and masks.dtype == _U8 and masks.is_contiguous()
    assert geom.dtype == _I32 and geom.is_contiguous() and geom.shape == (masks.shape[0], 4)
    N, H, W = masks.shape
    oi = torch.empty((N, S, S), dtype=_F32, device=img.device)
    om = torch.empty((N, S, S), dtype=_U8, device=img.device)
    area = torch.zeros((N,), dtype=_I32, device=img.device)
    L = _lib.load()
    _lib.check(L.sb_crop_resize(img.data_ptr(), masks.data_ptr(), geom.data_ptr(), N, H, W, S, oi.data_ptr(),
                                om.data_ptr(), area.data_ptr(), _stream()), "sb_crop_resize")
    _count()
    return oi, om, area


def mask_features(feat: torch.Tensor, mask: torch.Tensor, B: int, G: int = 64) -> torch.Tensor:
    """feat fp32 [B*G*G, C] token-major, mask uint8 [B,S,S] -> bf16 [B*G*G, 2C] = [feat*m | feat*(1-m)]."""
    _chk_cuda(feat, mask)
    assert feat.dtype == _F32 and feat.is_contiguous() and mask.dtype == _U8 and mask.is_contiguous()
    Cc = feat.shape[1]
    out = torch.empty((feat.shape[0], 2 * Cc), dtype=_BF16, device=feat.device)
    L = _lib.load()
    _lib.check(L.sb_mask_features(feat.data_ptr(), mask.data_ptr(), B, G, mask.shape[1], Cc, out.data_ptr(), _stream()),
               "sb_mask_features")
    _count()
    return out


def prelu(x: torch.Tensor, slope: float) -> torch.Tensor:
    _chk_cuda(x)
    assert x.is_contiguous() and x.dtype in (_BF16, _F32)
    out = torch.empty(x.shape, dtype=_BF16, device=x.device)
    L = _lib.load()
    _lib.check(L.sb_prelu(x.data_ptr(), int(x.dtype == _F32), x.numel(), float(slope), out.data_ptr(), _stream()), "sb_prelu")
    _count()
    return out


def im2col_3x3s1(x: torch.Tensor) -> torch.Tensor:
    """NHWC bf16 [B,H,W,C] -> [B*H*W, 9*C] patches of a 3x3 stride-1 pad-1 conv."""
    _chk_cuda(x)
    assert x.dtype == _BF16 and x.is_contiguous() and x.dim() == 4
    B, H, W, Cc = x.shape
    cols = torch.empty((B * H * W, 9 * Cc), dtype=_BF16, device=x.device)
    L = _lib.load()
    _lib.check(L.sb_im2col_3x3s1(x.data_ptr(), B, H, W, Cc, cols.data_ptr(), _stream()), "sb_im2col_3x3s1")
    _count()
    return cols


def mean_tokens(x: torch.Tensor, B: int) -> torch.Tensor:
    _chk_cuda(x)
    assert x.dtype == _BF16 and x.is_contiguous() and x.shape[0] % B == 0
    out = torch.empty((B, x.shape[1]), dtype=_F32, device=x.device)
    L = _lib.load()
    _lib.check(L.sb_mean_tokens(x.data_ptr(), B, x.shape[0] // B, x.shape[1], out.data_ptr(), _stream()), "sb_mean_tokens")
    _count()
    return out


def softmax_rows(x: torch.Tensor) -> torch.Tensor:
    _chk_cuda(x)
    assert x.dtype == _F32 and x.is_contiguous() and x.dim() == 2
    out = torch.empty_like(x)
    L = _lib.load()
    _lib.check(L.sb_softmax_rows(x.data_ptr(), x.shape[0], x.shape[1], out.data_ptr(), _stream()), "sb_softmax_rows")
    _count()
    return out


def label_equals(vol: torch.Tensor, label: int):
    """-> ((vol == label) as fp32, device uint64-in-int64 [1] count of matches)."""
    _chk_cuda(vol)
    assert vol.is_contiguous() and vol.element_size() in (1, 2, 4)
    out = torch.empty(vol.shape, dtype=_F32, device=vol.device)
    count = torch.zeros((1,), dtype=torch.int64, device=vol.device)
    L = _lib.load()
    _lib.check(L.sb_label_equals(vol.data_ptr(), vol.element_size(), vol.numel(), int(label), out.data_ptr(),
                                 count.data_ptr(), _stream()), "sb_label_equals")
    _count()
    return out, count


def corr1d_zero(vol: torch.Tensor, weights: torch.Tensor, axis: int) -> torch.Tensor:
    _chk_cuda(vol, weights)
    assert vol.dtype == _F32 and vol.is_contiguous() and vol.dim() == 3 and weights.dtype == _F32 and weights.is_contiguous()
    out = torch.empty_like(vol)
    L = _lib.load()
    _lib.check(L.sb_corr1d_zero(vol.data_ptr(), vol.shape[0], vol.shape[1], vol.shape[2], axis, weights.data_ptr(),
                                weights.numel(), out.data_ptr(), _stream()), "sb_corr1d_zero")
    _count()
    return out


def threshold_label_(sm: torch.Tensor, thr: float, label: int, result: torch.Tensor) -> None:
    _chk_cuda(sm, result)
    assert sm.dtype == _F32 and sm.is_contiguous() and result.dtype == _U8 and result.is_contiguous()
    L = _lib.load()
    _lib.check(L.sb_threshold_label(sm.data_ptr(), sm.numel(), thr, int(label) & 0xFF, result.data_ptr(), _stream()),
               "sb_threshold_label")
    _count()


def morph_ball(x: torch.Tensor, radius: int, op: int) -> torch.Tensor:
    """Binary erosion (op 0) / dilation (op 1) of a uint8 {0,1} [Z,Y,X] volume with a radius-r ball, zero padding."""
    _chk_cuda(x)
    assert x.dtype == _U8 and x.is_contiguous() and x.dim() == 3
    out = torch.empty_like(x)
    L = _lib.load()
    _lib.check(L.sb_morph_ball(x.data_ptr(), x.shape[0], x.shape[1], x.shape[2], int(radius), int(op), out.data_ptr(),
                               _stream()), "sb_morph_ball")
    _count()
    return out


def morph_cube(x: torch.Tensor, radius: int, op: int) -> torch.Tensor:
    """morph_ball with the full (2r+1)^3 cube as the structuring element (scipy binary_erosion(structure=ones(3,3,3)))."""
    _chk_cuda(x)
    assert x.dtype == _U8 and x.is_contiguous() and x.dim() == 3
    out = torch.empty_like(x)
    L = _lib.load()
    _lib.check(L.sb_morph_cube(x.data_ptr(), x.shape[0], x.shape[1], x.shape[2], int(radius), int(op), out.data_ptr(),
                               _stream()), "sb_morph_cube")
    _count()
    return out


# ---- organelle / membrane refinement workflow (csrc/refine.cu; REF saber/analysis/refine_membranes.py:120-548) ----------
_DT_CODE = {torch.uint8: 0, torch.int16: 1, torch.uint16: 2, torch.int32: 3, torch.int64: 4, torch.float32: 5}


def _dt_code(t: torch.Tensor) -> int:
    if t.dtype not in _DT_CODE:
        raise TypeError(f"label / mask volumes must be one of {sorted(str(k) for k in _DT_CODE)}, got {t.dtype}")
    return _DT_CODE[t.dtype]


def trim_binarize(vol: torch.Tensor, z_trim: int, xy_trim: int) -> torch.Tensor:
    """uint8 (vol != 0) inside the trimmed box, 0 outside (REF _trim_edges incl. its empty-slice quirks)."""
    _chk_cuda(vol)
    assert vol.is_contiguous() and vol.dim() == 3
    out = torch.empty(vol.shape, dtype=_U8, device=vol.device)
    L = _lib.load()
    _lib.check(L.sb_trim_binarize(vol.data_ptr(), _dt_code(vol), *vol.shape, int(z_trim), int(xy_trim), out.data_ptr(),
                                  _stream()), "sb_trim_binarize")
    _count()
    return out


def z_any(vol: torch.Tensor) -> torch.Tensor:
    """uint8 [Z]: slice z of a uint8 [Z,Y,X] volume has a set voxel."""
    _chk_cuda(vol)
    assert vol.dtype == _U8 and vol.is_contiguous() and vol.dim() == 3
    out = torch.empty((vol.shape[0],), dtype=_U8, device=vol.device)
    L = _lib.load()
    _lib.check(L.sb_z_any(vol.data_ptr(), vol.shape[0], vol.shape[1] * vol.shape[2], out.data_ptr(), _stream()), "sb_z_any")
    _count()
    return out


def label_bbox(vol: torch.Tensor, present: Optional[torch.Tensor], cap: int) -> torch.Tensor:
    """int32 [cap + 1, 8] = (min z, y, x, max z, y, x, voxel count, -) per label value, restricted to slices with
    present[z]; entry [0, 7] is non-zero when a label above cap was met."""
    _chk_cuda(vol)
    assert vol.is_contiguous() and vol.dim() == 3
    table = torch.empty((int(cap) + 1, 8), dtype=_I32, device=vol.device)
    L = _lib.load()
    _lib.check(L.sb_label_bbox(vol.data_ptr(), _dt_code(vol), *vol.shape, _ptr(present), int(cap), table.data_ptr(),
                               _stream()), "sb_label_bbox")
    _count(2)
    return table


def roi_binarize(vol: torch.Tensor, roi, label: int = -1, present: Optional[torch.Tensor] = None) -> torch.Tensor:
    """uint8 crop vol[z0:z1, y0:y1, x0:x1] == label (label < 0: != 0), zeroed on slices without present[z]."""
    _chk_cuda(vol)
    assert vol.is_contiguous() and vol.dim() == 3
    z0, y0, x0, z1, y1, x1 = (int(v) for v in roi)
    out = torch.empty((z1 - z0, y1 - y0, x1 - x0), dtype=_U8, device=vol.device)
    L = _lib.load()
    _lib.check(L.sb_roi_binarize(vol.data_ptr(), _dt_code(vol), *vol.shape, z0, y0, x0, z1 - z0, y1 - y0, x1 - x0, int(label),
                                 _ptr(present), out.data_ptr(), _stream()), "sb_roi_binarize")
    _count()
    return out


def roi_paste(vol: torch.Tensor, roi, mask: torch.Tensor, value: int) -> None:
    """vol[z0:z1, y0:y1, x0:x1][mask != 0] = value, in place."""
    _chk_cuda(vol, mask)
    assert vol.is_contiguous() and vol.dim() == 3 and mask.dtype == _U8 and mask.is_contiguous()
    z0, y0, x0, z1, y1, x1 = (int(v) for v in roi)
    assert tuple(mask.shape) == (z1 - z0, y1 - y0, x1 - x0)
    L = _lib.load()
    _lib.check(L.sb_roi_paste(vol.data_ptr(), _dt_code(vol), *vol.shape, z0, y0, x0, z1 - z0, y1 - y0, x1 - x0, mask.data_ptr(),
                              int(value), _stream()), "sb_roi_paste")
    _count()


def mask_logic(a: torch.Tensor, b: torch.Tensor, op: str) -> torch.Tensor:
    """'and' / 'or' / 'andnot' of two uint8 {0,1} volumes."""
    _chk_cuda(a, b)
    assert a.dtype == _U8 and b.dtype == _U8 and a.is_contiguous() and b.is_contiguous() and a.shape == b.shape
    out = torch.empty_like(a)
    L = _lib.load()
    _lib.check(L.sb_mask_logic(a.data_ptr(), b.data_ptr(), a.numel(), {"and": 0, "or": 1, "andnot": 2}[op], out.data_ptr(),
                               _stream()), "sb_mask_logic")
    _count()
    return out


def label_select(labels: torch.Tensor, sizes: Optional[torch.Tensor] = None, count: Optional[torch.Tensor] = None,
                 largest: bool = False) -> torch.Tensor:
    """uint8 mask of the voxels with a label (largest=False) or of the largest component, the first among equals."""
    _chk_cuda(labels)
    assert labels.dtype == _I32 and labels.is_contiguous()
    out = torch.empty(labels.shape, dtype=_U8, device=labels.device)
    which = torch.empty((1,), dtype=_I32, device=labels.device) if largest else None
    L = _lib.load()
    _lib.check(L.sb_label_select(labels.data_ptr(), labels.numel(), _ptr(sizes), _ptr(count), 1 if largest else 0, _ptr(which),
                                 out.data_ptr(), _stream()), "sb_label_select")
    _count(2 if largest else 1)
    return out


def label_keep_ratio(labels: torch.Tensor, mask: torch.Tensor, sizes: torch.Tensor, ratio: float) -> torch.Tensor:
    """uint8 mask of the components whose overlap with `mask` exceeds ratio x their voxel count."""
    _chk_cuda(labels, mask, sizes)
    assert labels.dtype == _I32 and labels.is_contiguous() and mask.dtype == _U8 and mask.is_contiguous()
    out = torch.empty(labels.shape, dtype=_U8, device=labels.device)
    overlap = torch.empty_like(sizes)
    L = _lib.load()
    _lib.check(L.sb_label_keep_ratio(labels.data_ptr(), mask.data_ptr(), labels.numel(), sizes.data_ptr(), overlap.data_ptr(),
                                     sizes.numel(), float(ratio), out.data_ptr(), _stream()), "sb_label_keep_ratio")
    _count(2)
    return out


def overlay_nonzero(dst: torch.Tensor, src: torch.Tensor) -> None:
    """dst[src > 0] = src[src > 0], in place (one step of convert_to_3d_labels)."""
    _chk_cuda(dst, src)
    assert dst.dtype == src.dtype and dst.shape == src.shape and dst.is_contiguous() and src.is_contiguous()
    L = _lib.load()
    _lib.check(L.sb_overlay_nonzero(dst.data_ptr(), src.data_ptr(), _dt_code(dst), dst.numel(), _stream()), "sb_overlay_nonzero")
    _count()


# ---- Fourier-space rescale / band-pass (csrc/fft.cu; REF saber/filters/downsample.py, saber/filters/tomograms.py) ----------
_C64 = torch.complex64
_fft_tw_cache: dict = {}


def fft_twiddles(n: int, device) -> torch.Tensor:
    """complex64 [n]: exp(-2 pi i k / n), evaluated in double precision on the device; cached per (device, n)."""
    dev = torch.device(device)
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), int(n))
    tw = _fft_tw_cache.get(key)
    if tw is None:
        tw = torch.empty((int(n),), dtype=_C64, device=dev)
        L = _lib.load()
        _lib.check(L.sb_fft_twiddles(int(n), tw.data_ptr(), _stream()), "sb_fft_twiddles")
        _count()
        _fft_tw_cache[key] = tw
    return tw


def fft_lines(x: torch.Tensor, axis: int, inverse: bool = False, crop: Optional[tuple] = None, out_mode: str = "complex",
              scale: float = 1.0, bandpass=None) -> torch.Tensor:
    """One line pass of a complex FFT along `axis` of a 2-D / 3-D float32 (real) or complex64 array, out of place.
    crop=(start, m): store the m-wide centre crop of the fftshift-ed spectrum (un-shifted again) instead of all n values.
    out_mode 'complex' | 'real' | 'abs'; scale multiplies the stored values; bandpass = 8 floats (see sb_fft_lines),
    only on the first axis of a 3-D spectrum."""
    import ctypes as _C
    _chk_cuda(x)
    assert x.is_contiguous() and x.dim() in (2, 3) and x.dtype in (_F32, _C64)
    axis = axis % x.dim()
    shape = list(x.shape)
    n = shape[axis]
    start, m = crop if crop is not None else (0, n)
    oshape = list(shape)
    oshape[axis] = m
    out = torch.empty(oshape, dtype=_C64 if out_mode == "complex" else _F32, device=x.device)
    if axis == x.dim() - 1:
        rows_mode, lines, batch = 1, x.numel() // n, 1
    else:
        rows_mode = 0
        lines = 1
        for s in shape[axis + 1:]:
            lines *= s
        batch = 1
        for s in shape[:axis]:
            batch *= s
    bp = None
    D = H = W = 0
    if bandpass is not None:
        assert x.dim() == 3 and axis == 0 and crop is None
        bp = (_C.c_float * 8)(*[float(v) for v in bandpass])
        D, H, W = shape
    L = _lib.load()
    _lib.check(L.sb_fft_lines(x.data_ptr(), out.data_ptr(), fft_twiddles(n, x.device).data_ptr(), n, m, rows_mode, lines, batch,
                              1 if x.dtype == _F32 else 0, {"complex": 0, "real": 1, "abs": 2}[out_mode], 1 if inverse else 0,
                              float(scale), 0 if crop is None else 1, int(start), bp, D, H, W, _stream()), "sb_fft_lines")
    _count()
    return out


def bandpass_volume(shape, bandpass) -> torch.Tensor:
    """float32 [D,H,W]: the fftshift-ed cosine band-pass volume (REF Filter3D.filter)."""
    import ctypes as _C
    D, H, W = (int(v) for v in shape)
    out = torch.empty((D, H, W), dtype=_F32, device="cuda")
    bp = (_C.c_float * 8)(*[float(v) for v in bandpass])
    L = _lib.load()
    _lib.check(L.sb_bandpass_volume(D, H, W, bp, out.data_ptr(), _stream()), "sb_bandpass_volume")
    _count()
    return out
