"""Every attention kernel against an fp64 reference, with bars tight enough to see one dropped key.

The kernel-level tests in test_gpu_kernels.py compare with a max-error bar of 2e-2 / 3e-2 on outputs whose rms is
0.02-0.03 at 4096-8196 keys (softmax over random scores averages ~n/e keys), so an output scaled by 0.9 or a dropped
ragged tail passes them. Here every case is checked against two bars:

  * relative L2 ||out - ref|| / ||ref||            <= 5e-3   (bf16 routes), 1e-5 (fp32 validation routes)
  * max |out - ref| / rms(ref)                     <= 0.08   (bf16 routes), 2e-4 (fp32 validation routes)

The reference is exact SDPA in float64 on the bf16 (or fp32) operands the kernel receives; the same helpers with
mode="bf16" give the emulated floor, the rounding a correct bf16 flash kernel must have (fp32 scores, exponentials relative to the row maximum, P rounded to bf16 before
P V, fp32 row sums, bf16 output); every case also asserts that this floor is within half of each bar, so no bar asks
for more than bf16 arithmetic allows. The CPU tests at the end pin that the bars catch the defects they exist for.

Inputs make every key count: besides random q / k / v ("flat") and q x 3 ("peaked"), a "beacon" key sits ~8 nats above
all others for a group of query rows (output ~ that key's v row) at key 0, nk - 1 and both sides of each tile or split
edge of the route; "beacon2" puts two equal beacons in different tiles (output = the mean of their v rows); "ramp"
scores rise by 9 (or 5) log2 units per key tile so the online softmax rescales on every (every other) tile; "distinct"
scales and shifts each batch entry differently; "poison" makes the keys that follow a batch entry's last key
(the next entry's first keys, or extra rows after the last entry) ~30 nats hotter than anything that entry may see;
"cold" puts every real score ~6 nats below 0, so a zero key row counted in the softmax takes over; row-view operands sit in wider buffers whose unused columns hold finite +-3e4 sentinels.
"""
import math

import pytest
import torch
import torch.nn.functional as F

BF16, F32, F64 = torch.bfloat16, torch.float32, torch.float64

# Bars (relative L2, max |err| / rms(ref)), measured on a B200 (1000 W power limit) over this file's cases.
# bf16: the emulated floor is 1.5e-4-2.4e-3 relative L2 and 0.001-0.039 x rms. The kernels sit on it (flash, window,
# kadd, few-keys, d256 tc: <= 2.4e-3 and <= 0.032) except two routes, both inside the bars: the t2i fold kernels reach
# 4.0e-3 / 0.068 because they round the folded query (scale log2(e) Wk_h^T q_h) to bf16, an extra rounding the floor
# does not have (modelled on the CPU, that rounding alone gives 3.4e-3 / 0.058 on the B3 nt7 case, as the kernel does);
# the tcgen05 Hiera kernel reaches 0.055 x rms max error (floor 0.030) on peaked global attention, 2.2e-3 rel L2.
# fp32 validation routes: 3e-7-2e-6 relative L2 for kernel and floor alike; the max bar is 2e-4 x rms because plain fp32
# arithmetic already reaches 6.1e-5 x rms on the pooled, padded 14x14 windows (the validation mode's "1e-4" is relative
# to the worst element, max |ref|, which is several times the rms).
BF16_BARS = (5e-3, 0.08)
F32_BARS = (1e-5, 2e-4)

BEACON_GAP = 12.0   # beacon score in nats over the mean score: ~8 nats above the maximum of 4096-8196 random scores
POISON_GAP = 30.0   # poisoned keys over the entry's own scores


# ------------------------------------------------------------------------------------------------------------------
# Reference and emulated floor
# ------------------------------------------------------------------------------------------------------------------
def _sdpa(q, k, v, scale, mode):
    """q [N, h, nq, d], k / v [N, h, nk, d] (expanded views allowed) -> [N, h, nq, dv].

    mode "exact": float64 softmax(q k^T scale) v. mode "bf16": a correct bf16 flash kernel (fp32 scores, exponentials
    relative to the row maximum, P rounded to bf16 for P V, fp32 row sums, bf16 output). mode "f32": the same in fp32
    without any bf16 rounding (the fp32 validation kernels). Chunked over N and queries so memory stays bounded."""
    dt = F64 if mode == "exact" else F32
    N, h, nq, _ = q.shape
    nk, dv = k.shape[2], v.shape[3]
    out = torch.empty(N, h, nq, dv, dtype=dt, device=q.device)
    budget = 1 << 24
    qc = max(1, min(nq, budget // max(1, h * nk)))
    nc = max(1, min(N, budget // max(1, h * nk * nq))) if qc == nq else 1
    for n0 in range(0, N, nc):
        kk = k[n0:n0 + nc].to(dt)
        vv = v[n0:n0 + nc].to(dt)
        for i0 in range(0, nq, qc):
            s = (q[n0:n0 + nc, :, i0:i0 + qc].to(dt) @ kk.transpose(-1, -2)) * scale
            if mode == "exact":
                o = torch.softmax(s, -1) @ vv
            else:
                p = torch.exp(s - s.amax(-1, keepdim=True))
                pv = p.to(BF16).to(dt) if mode == "bf16" else p
                o = (pv @ vv) / p.sum(-1, keepdim=True)
            out[n0:n0 + nc, :, i0:i0 + qc] = o.to(BF16).to(dt) if mode == "bf16" else o
    return out


def ref_attention(q, k, v, B, heads, nq, nk, q_shared=False, kv_shared=False, k_add=None, scale=None, mode="exact"):
    """Plain batched MHA on row-major operands: q [(1|B)*nq, C], k / v [(1|B)*nk, C], k_add [nk, C] added to every
    batch entry's keys. Returns [B*nq, C] (float64 for "exact")."""
    C = q.shape[1]
    hd = C // heads
    dt = F64 if mode == "exact" else F32
    scale = hd ** -0.5 if scale is None else scale

    def heads_major(x, n, shared):
        x = x.to(dt).reshape(-1, n, heads, hd).transpose(1, 2)
        return x.expand(B, -1, -1, -1) if shared else x

    kk = k.to(dt)
    if k_add is not None:
        kk = (kk.reshape(-1, nk, C) + k_add.to(dt)[None]).reshape(-1, C)
    o = _sdpa(heads_major(q, nq, q_shared), heads_major(kk, nk, kv_shared), heads_major(v, nk, kv_shared), scale, mode)
    return o.transpose(1, 2).reshape(B * nq, C)


def ref_window(qkv, bias, B, H, W, heads, hd, ws, pool, mode="exact"):
    """Hiera MultiScaleAttention on an already-projected qkv [B*H*W, 3C] (padding tokens carry ``bias`` [3C]; 2x2
    max-pooled queries for pool 2). The window logic of test_gpu_kernels._window_ref, in float64 and chunked."""
    dt = F64 if mode == "exact" else F32
    C = heads * hd
    x = qkv.to(dt).view(B, H, W, 3 * C)
    if ws > 0:
        ph, pw = (ws - H % ws) % ws, (ws - W % ws) % ws
        if ph or pw:
            b3 = bias.to(dt) if bias is not None else torch.zeros(3 * C, dtype=dt, device=qkv.device)
            pad = b3.view(1, 1, 1, 3 * C).expand(B, H + ph, W + pw, 3 * C).clone()
            pad[:, :H, :W] = x
            x = pad
        Hp, Wp = H + ph, W + pw
        x = x.view(B, Hp // ws, ws, Wp // ws, ws, 3 * C).permute(0, 1, 3, 2, 4, 5).reshape(-1, ws, ws, 3 * C)
    else:
        Hp, Wp = H, W
    nW, hh, ww = x.shape[0], x.shape[1], x.shape[2]
    q, k, v = x.reshape(nW, hh * ww, 3, heads, hd).unbind(2)
    if pool == 2:
        qq = F.max_pool2d(q.reshape(nW, hh, ww, C).permute(0, 3, 1, 2), 2, 2)
        hq, wq = qq.shape[2:]
        q = qq.permute(0, 2, 3, 1).reshape(nW, hq * wq, heads, hd)
    else:
        hq, wq = hh, ww
    o = _sdpa(q.transpose(1, 2), k.transpose(1, 2), v.transpose(1, 2), hd ** -0.5, mode)
    o = o.transpose(1, 2).reshape(nW, hq, wq, C)
    if nW != B:
        nwh, nww = Hp // hh, Wp // ww
        o = o.view(B, nwh, nww, hq, wq, C).permute(0, 1, 3, 2, 4, 5).reshape(B, nwh * hq, nww * wq, C)
    Ho, Wo = H // pool, W // pool
    return o[:, :Ho, :Wo].reshape(B * Ho * Wo, C)


def ref_t2i(q, x, kadd, wk, wv, bv, B, nt, nk, x_shared, mode="exact"):
    """Token -> image attention of the mask decoder: softmax(q (x Wk^T + kadd)^T / 4) (x Wv^T + bv), 8 heads x 16."""
    dt = F64 if mode == "exact" else F32
    xf = x.to(dt).view(-1, nk, 256).expand(B, nk, 256)
    k = (xf @ wk.to(dt).t() + kadd.to(dt)[None]).view(B, nk, 8, 16).transpose(1, 2)
    v = (xf @ wv.to(dt).t() + bv.to(dt)).view(B, nk, 8, 16).transpose(1, 2)
    qq = q.to(dt).view(B, nt, 8, 16).transpose(1, 2)
    return _sdpa(qq, k, v, 0.25, mode).transpose(1, 2).reshape(B * nt, 128)


def _errors(out, ref):
    d = out.to(F64) - ref.to(F64)
    rms = ref.to(F64).pow(2).mean().sqrt()
    return (d.norm() / ref.to(F64).norm()).item(), (d.abs().max() / rms).item()


def assert_close(out, ref, emu, case, fp32=False):
    """Both bars on the kernel output, and the emulated floor within half of each bar."""
    rel_bar, max_bar = F32_BARS if fp32 else BF16_BARS
    assert out.shape == ref.shape, (out.shape, ref.shape)
    assert torch.isfinite(out).all(), f"{case}: non-finite output"
    rel, mx = _errors(out, ref)
    frel, fmx = _errors(emu, ref)
    print(f"\n[bars] {case}: rel_l2 {rel:.2e} max/rms {mx:.2e} | floor rel_l2 {frel:.2e} max/rms {fmx:.2e}")
    assert frel <= rel_bar / 2 and fmx <= max_bar / 2, f"{case}: emulated floor {frel:.2e} / {fmx:.4f} above half the bar"
    assert rel <= rel_bar and mx <= max_bar, f"{case}: rel_l2 {rel:.3e} (bar {rel_bar}), max/rms {mx:.4f} (bar {max_bar})"


# ------------------------------------------------------------------------------------------------------------------
# Inputs
# ------------------------------------------------------------------------------------------------------------------
def _orthonormal(n, d, gen):
    qm, _ = torch.linalg.qr(torch.randn(d, n, generator=gen, dtype=F64))
    return qm.t().float()  # [n, d]


def _project_out(x, U):
    """Remove the components of x [..., d] along the orthonormal rows of U [n, d]."""
    return x - (x @ U.t()) @ U


def edge_positions(nk, tile, half=None, splits=None, limit=24):
    """Key 0, key nk - 1 and both sides of the first and last tile edges (and of the 32-key halves of a tc tile, and of
    every split boundary), without duplicates, in that order."""
    pos = [0, nk - 1]
    edges = [t * tile for t in range(1, (nk + tile - 1) // tile)]
    edges = edges[:3] + edges[-3:]
    if half:
        edges += [t * tile + half for t in (0, 1, (nk - 1) // tile) if t * tile + half < nk]
    if splits:
        kps = nk // splits
        edges += [s * kps for s in range(1, splits)]
    for e in sorted(set(edges)):
        pos += [e - 1, e]
    out = []
    for p in pos:
        if 0 <= p < nk and p not in out:
            out.append(p)
    return out[:limit]


def _pairs(pos, tile):
    """Disjoint pairs of positions in different tiles (for two equal beacons)."""
    lo, hi = pos[: len(pos) // 2], pos[len(pos) // 2:][::-1]
    return [(a, b) for a, b in zip(lo, hi) if a // tile != b // tile]


def _sentinels(rows, cols, gen):
    return torch.where(torch.rand(rows, cols, generator=gen) < 0.5, 3e4, -3e4)


def plain_case(kind, B, heads, hd, nq, nk, tile=64, half=None, q_shared=False, kv_shared=False, rowview=False,
               k_add=False, seed=0, device="cuda"):
    """bf16 operands of ops.attention(_kadd): dict(q, k, v, k_add) with q [(1|B)*nq, C], k / v [(1|B)*nk, C]."""
    gen = torch.Generator().manual_seed(seed)
    Bq, Bk = (1 if q_shared else B), (1 if kv_shared else B)
    s = hd ** -0.5
    q = torch.randn(Bq, nq, heads, hd, generator=gen)
    k = torch.randn(Bk, nk, heads, hd, generator=gen)
    v = torch.randn(Bk, nk, heads, hd, generator=gen)
    extra = None  # key rows after the last batch entry (inside the allocation, outside the operand)
    if kind == "peaked":
        q *= 3
    elif kind in ("beacon", "beacon2"):
        pos = edge_positions(nk, tile, half)
        groups = [(p,) for p in pos] if kind == "beacon" else _pairs(pos, tile)
        G = max(1, min(len(groups), hd // 2, nq))
        U = _orthonormal(G, hd, gen)
        a = math.sqrt(BEACON_GAP / s)
        q, k = _project_out(q, U), _project_out(k, U)
        q += a * U[torch.arange(nq) % G][None, :, None, :]
        for bk in range(Bk):
            for h in range(heads):
                for g in range(G):
                    for p in groups[(g + bk * heads + h) % len(groups)]:
                        k[bk, p, h] = a * U[g]
    elif kind == "cold":  # every real score ~6 nats below zero: a zero key row (score 0) counted in the softmax dominates
        U = _orthonormal(1, hd, gen)
        a = 4.0
        q, k = _project_out(q, U) + a * U[0], _project_out(k, U) - (6.0 / (s * a)) * U[0]
    elif kind in ("ramp9", "ramp5"):
        slope = 9.0 if kind == "ramp9" else 5.0  # log2 units per key tile
        U = _orthonormal(1, hd, gen)
        a = 4.0
        q, k = 0.1 * _project_out(q, U), _project_out(k, U)
        q += a * U[0]
        beta = slope * math.log(2.0) * torch.arange(nk, dtype=F32) / (tile * s * a)
        k += beta[None, :, None, None] * U[0]
    elif kind == "distinct":
        for b in range(B):
            if not q_shared:
                q[b] *= 0.6 + 0.4 * b
            if not kv_shared:
                k[b] *= 1.0 + 0.25 * b
                v[b] = v[b] * (1.0 + 0.5 * b) + 0.5 * b
    elif kind == "poison":
        assert not q_shared and not kv_shared and B <= hd
        npois = (tile - nk % tile) % tile
        U = _orthonormal(B, hd, gen)
        a = math.sqrt(POISON_GAP / s)
        q, k = _project_out(q, U), _project_out(k, U)
        for b in range(B):
            q[b] += a * U[b]
            if b + 1 < B:
                k[b + 1, :npois] += a * U[b]
        extra = a * U[B - 1].expand(npois, heads, hd).reshape(npois, heads * hd) + 0.0
    else:
        assert kind == "flat", kind
    C = heads * hd
    q, k, v = q.reshape(-1, C), k.reshape(-1, C), v.reshape(-1, C)
    nrows = k.shape[0] + (extra.shape[0] if extra is not None else 0)
    if rowview:
        qbuf = _sentinels(q.shape[0], 2 * C, gen)
        qbuf[:, C:] = q
        kvbuf = _sentinels(nrows, 3 * C, gen)
        kvbuf[: k.shape[0], :C] = k
        kvbuf[: k.shape[0], 2 * C:] = v
        if extra is not None:
            kvbuf[k.shape[0]:, :C] = extra
        qbuf, kvbuf = qbuf.to(BF16).to(device), kvbuf.to(BF16).to(device)
        out = dict(q=qbuf[:, C:], k=kvbuf[: k.shape[0], :C], v=kvbuf[: k.shape[0], 2 * C:], _keep=(qbuf, kvbuf))
    else:
        kbuf = torch.cat([k, extra]) if extra is not None else k
        vbuf = torch.cat([v, torch.randn(nrows - v.shape[0], C, generator=gen)]) if extra is not None else v
        kbuf, vbuf = kbuf.to(BF16).to(device), vbuf.to(BF16).to(device)
        out = dict(q=q.to(BF16).to(device), k=kbuf[: k.shape[0]], v=vbuf[: v.shape[0]], _keep=(kbuf, vbuf))
    out["k_add"] = (0.5 * torch.randn(nk, C, generator=gen)).to(BF16).to(device) if k_add else None
    return out


def window_case(kind, B, H, W, heads, hd, ws, pool, tile=64, bias=True, seed=0, device="cuda"):
    """qkv [B*H*W, 3C] bf16 (and the fp32 bias padding tokens carry). Beacons are per (batch entry, window, head),
    indexed by the key order inside the window (row-major over the window)."""
    gen = torch.Generator().manual_seed(seed)
    C = heads * hd
    s = hd ** -0.5
    x = torch.randn(B, H, W, 3, heads, hd, generator=gen)
    if ws <= 0 or ws >= max(H, W):
        wsy, wsx = H, W
    else:
        wsy = wsx = ws
    nwy, nwx = -(-H // wsy), -(-W // wsx)
    if kind == "peaked":
        x[:, :, :, 0] *= 3
    elif kind in ("beacon", "beacon2", "ramp9", "ramp5"):
        U = _orthonormal(1, hd, gen)
        x[:, :, :, :2] = _project_out(x[:, :, :, :2], U)
        if kind.startswith("ramp"):
            slope = 9.0 if kind == "ramp9" else 5.0
            a = 4.0
            x[:, :, :, 0] = 0.1 * x[:, :, :, 0] + a * U[0]
            yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
            j = ((yy % wsy) * wsx + (xx % wsx)).float()
            beta = slope * math.log(2.0) * j / (tile * s * a)
            x[:, :, :, 1] += beta[None, :, :, None, None] * U[0]
        else:
            a = math.sqrt(BEACON_GAP / s)
            x[:, :, :, 0] += a * U[0]
            pos = edge_positions(wsy * wsx, tile)
            groups = [(p,) for p in pos] if kind == "beacon" else _pairs(pos, tile)
            idx = 0
            for b in range(B):
                for wy in range(nwy):
                    for wx in range(nwx):
                        for h in range(heads):
                            for p in groups[idx % len(groups)]:
                                y, xq = wy * wsy + p // wsx, wx * wsx + p % wsx
                                if y >= H or xq >= W:  # padding position: use the window's last real key
                                    y, xq = min(y, H - 1), min(xq, W - 1)
                                x[b, y, xq, 1, h] = a * U[0]
                            idx += 1
    elif kind == "distinct":
        for b in range(B):
            x[b, :, :, 0] *= 0.6 + 0.4 * b
            x[b, :, :, 2] = x[b, :, :, 2] * (1.0 + 0.5 * b) + 0.5 * b
    else:
        assert kind == "flat", kind
    qkv = x.reshape(B * H * W, 3 * C).to(BF16).to(device)
    b3 = (torch.randn(3 * C, generator=gen) * 0.2).to(device) if bias else None
    return qkv, b3


# ------------------------------------------------------------------------------------------------------------------
# GPU: every route at its edges
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ops():
    from saber_b200 import ops as _ops
    _ops.require_b200()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return _ops


def _run_plain(ops, case, kind, B, heads, hd, nq, nk, tile, half=None, q_shared=False, kv_shared=False, rowview=False,
               kadd=False, seed=0):
    d = plain_case(kind, B, heads, hd, nq, nk, tile=tile, half=half, q_shared=q_shared, kv_shared=kv_shared,
                   rowview=rowview, k_add=kadd, seed=seed)
    if kadd:
        out = ops.attention_kadd(d["q"], d["k"], d["k_add"], d["v"], B, heads, nq, nk, kv_shared=kv_shared)
    else:
        out = ops.attention(d["q"], d["k"], d["v"], B, heads, nq, nk, q_shared=q_shared, kv_shared=kv_shared)
    args = (d["q"], d["k"], d["v"], B, heads, nq, nk, q_shared, kv_shared, d["k_add"])
    assert_close(out, ref_attention(*args), ref_attention(*args, mode="bf16"), case)


TC_SHAPES = [(3, 128, 64), (3, 128, 65), (1, 128, 96), (3, 128, 97), (1, 128, 127), (3, 128, 128), (3, 128, 129),
             (1, 4096, 4096), (3, 128, 4100), (3, 256, 8196), (1, 128, 8256), (1, 128, 7 * 4096 + 64)]
TC_CASES = ([("flat", *s, {}) for s in TC_SHAPES] + [("beacon", *s, {}) for s in TC_SHAPES] + [
    ("peaked", 3, 128, 4100, {}), ("beacon2", 3, 128, 4100, {}), ("beacon2", 1, 128, 129, {}),
    ("ramp9", 1, 128, 8196, {}), ("ramp5", 1, 128, 8196, {}), ("ramp9", 3, 128, 129, {}), ("ramp5", 1, 4096, 4096, {}),
    ("distinct", 3, 256, 8196, {}), ("poison", 3, 128, 65, {}), ("poison", 3, 128, 97, {}), ("poison", 3, 128, 127, {}),
    ("poison", 3, 256, 8196, {}), ("poison", 3, 128, 4100, {}), ("poison", 1, 128, 129, {}),
    ("cold", 1, 128, 65, {}), ("cold", 3, 128, 97, {}), ("cold", 1, 128, 4100, {}), ("cold", 3, 128, 8196, {}),
    ("beacon", 3, 128, 4100, dict(q_shared=True)), ("distinct", 3, 128, 4100, dict(kv_shared=True)),
    ("beacon", 3, 128, 97, dict(rowview=True)), ("poison", 3, 128, 8196, dict(rowview=True)),
    ("flat", 3, 4096, 8196, dict(rowview=True, q_shared=True))])


@pytest.mark.gpu
@pytest.mark.parametrize("kind,B,nq,nk,kw", TC_CASES,
                         ids=[f"{c[0]}-B{c[1]}-nq{c[2]}-nk{c[3]}" + "".join("-" + k for k in c[4]) for c in TC_CASES])
def test_attn_d256_tc(ops, kind, B, nq, nk, kw):
    """Route: attn_d256_tc_kernel (1 head x 256, nq % 128 == 0, nk >= 64; memory attention). 64-key tiles split in
    two 32-key halves per softmax thread; beacons at keys 0, nk - 1, 31/32 and 63/64 of the first tiles, 63/64 and
    127/128, the halves of the last tile and the last tile edges. Ragged nk: the tail mask (poison reads the next
    entry's first keys or rows past the operand); ramps fire the lazy rescale on every / every other tile."""
    _run_plain(ops, f"d256_tc {kind} B{B} nq{nq} nk{nk} {kw}", kind, B, 1, 256, nq, nk, 64, half=32, **kw)


FLASH256_CASES = [("flat", 2, 100, 31), ("flat", 2, 100, 32), ("flat", 1, 100, 33), ("flat", 2, 128, 33),
                  ("flat", 1, 4000, 4100), ("flat", 3, 100, 8196), ("beacon", 2, 100, 33), ("beacon", 2, 128, 33),
                  ("beacon", 1, 4000, 4100), ("beacon", 3, 100, 8196), ("beacon2", 2, 100, 8196),
                  ("ramp9", 1, 100, 4100), ("ramp5", 2, 100, 4100), ("distinct", 3, 100, 8196)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,B,nq,nk", FLASH256_CASES)
def test_flash_hd256(ops, kind, B, nq, nk):
    """Route: flash_attn_kernel<256, 4, 32> (1 head x 256 with nq % 128 != 0 or nk < 64): Q in shared memory, 32-key
    tiles; beacons at 0, nk - 1 and 31/32, 63/64, 95/96 and the last tile edges."""
    _run_plain(ops, f"flash256 {kind} B{B} nq{nq} nk{nk}", kind, B, 1, 256, nq, nk, 32)


FLASH_CASES = [
    # (B, heads, hd, nq, nk): 1-warp CTAs for nq <= 16, 4 warps otherwise; 64-key tiles
    (2, 8, 72, 4096, 4096), (3, 8, 16, 7, 4096), (3, 2, 32, 17, 4097), (2, 1, 64, 65, 4095), (1, 2, 96, 64, 63),
    (2, 1, 128, 1, 65), (3, 8, 64, 16, 17), (2, 2, 128, 4096, 64), (2, 8, 16, 4096, 15), (3, 2, 16, 1024, 4097), (3, 2, 32, 64, 4097)]
FLASH16_CASES = [(3, 2, 32, 16, 1), (2, 8, 72, 16, 8), (1, 1, 128, 7, 16), (3, 8, 16, 1, 16)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["flat", "beacon", "ramp9", "cold"])
@pytest.mark.parametrize("B,heads,hd,nq,nk", FLASH_CASES)
def test_flash(ops, kind, B, heads, hd, nq, nk):
    """Route: flash_attn_kernel<HDP, 1|4, 64> (head_dim <= 128): beacons at 0, nk - 1, 63/64, 127/128 and the last
    tile edges; ramps rescale O on every tile. (2, 8, 16, 4096, 15) stays on this kernel: 4-warp CTAs, heads x 16 at
    8 heads would take the few-keys kernel only with nq >= 1024 and no kv sharing — it has nq 4096 but kv_shared."""
    kw = dict(kv_shared=True) if (heads, hd, nk) == (8, 16, 15) else {}
    if kind != "flat" and nk == 1:
        pytest.skip("one key")
    _run_plain(ops, f"flash {kind} B{B} h{heads} hd{hd} nq{nq} nk{nk}", kind, B, heads, hd, nq, nk, 64, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["flat", "beacon", "distinct"])
@pytest.mark.parametrize("B,heads,hd,nq,nk", FLASH16_CASES)
def test_flash_16key_tiles(ops, kind, B, heads, hd, nq, nk):
    """Route: flash_attn_kernel<HDP, 1, 16> (1 warp: nq <= 16, nk <= 16, no k_add; Hiera 4x4 windows): one 16-key
    tile, beacons at every key in turn across (batch entry, head)."""
    if kind == "beacon" and nk == 1:
        pytest.skip("one key")
    _run_plain(ops, f"flash16 {kind} B{B} h{heads} hd{hd} nq{nq} nk{nk}", kind, B, heads, hd, nq, nk, 16)


@pytest.mark.gpu
@pytest.mark.parametrize("extra", [{}, dict(q_shared=True), dict(kv_shared=True), dict(rowview=True)])
def test_flash_operand_layouts(ops, extra):
    """Route: flash_attn_kernel<80, 4, 64>: shared q / kv operands and row views (pitch > width, +-3e4 sentinels in
    the unused columns) with distinct batch entries and with beacons."""
    for kind in ("distinct", "beacon"):
        _run_plain(ops, f"flash layout {kind} {extra}", kind, 3, 2, 72, 300, 1000, 64, **extra)


KADD_CASES = [(3, 8, 16, 8, 4096, True), (3, 8, 16, 8, 4096, False), (2, 2, 64, 8, 4096, True),
              (2, 1, 256, 8, 4096, True), (2, 1, 256, 100, 4100, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["flat", "beacon", "ramp5"])
@pytest.mark.parametrize("B,heads,hd,nq,nk,kv_shared", KADD_CASES)
def test_flash_kadd(ops, kind, B, heads, hd, nq, nk, kv_shared):
    """Route: flash_attn_kernel with k_add (ops.attention_kadd; the mask decoder's token -> image attention with the
    positional key term): 64-key tiles (32 at head_dim 256), beacons at tile edges, k_add in a third staging region."""
    tile = 32 if hd > 128 else 64
    _run_plain(ops, f"kadd {kind} B{B} h{heads} hd{hd} nq{nq} nk{nk} shared{kv_shared}", kind, B, heads, hd, nq, nk,
               tile, kv_shared=kv_shared, kadd=True)


FEWKEYS_CASES = [(1, 1024, False), (2, 1500, False), (8, 4096, False), (9, 4096, True), (16, 1500, True),
                 (16, 4096, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["flat", "beacon", "distinct"])
@pytest.mark.parametrize("nk,nq,q_shared", FEWKEYS_CASES)
def test_fewkeys(ops, kind, nk, nq, q_shared):
    """Route: fewkeys_attn_kernel through ops.attention (8 heads x 16, nk <= 16, nq >= 1024, kv per prompt): K / V of
    a prompt in shared memory as fp32, one thread per (query row, head); a beacon at every key in turn."""
    if kind == "beacon" and nk == 1:
        pytest.skip("one key")
    _run_plain(ops, f"fewkeys {kind} nk{nk} nq{nq} qs{q_shared}", kind, 3, 8, 16, nq, nk, 16, q_shared=q_shared)


@pytest.mark.gpu
@pytest.mark.parametrize("nk,q_shared", [(2, False), (8, True), (16, False)])
def test_fewkeys_query_term(ops, nk, q_shared):
    """Route: fewkeys_attn_kernel through ops.attention_few_keys (q_eff = bf16(q + q_add)), beacons per group."""
    B, nq = 3, 1500
    d = plain_case("beacon", B, 8, 16, nq, nk, tile=16, q_shared=q_shared, seed=4)
    qa = (0.3 * torch.randn(nq, 128, generator=torch.Generator().manual_seed(5))).cuda()
    out = ops.attention_few_keys(d["q"], qa, d["k"], d["v"], B, nq, nk, q_shared=q_shared)
    qe = (d["q"].float().view(-1, nq, 128) + qa[None]).to(BF16).reshape(-1, 128)
    args = (qe, d["k"], d["v"], B, 8, nq, nk, q_shared, False)
    assert_close(out, ref_attention(*args), ref_attention(*args, mode="bf16"), f"fewkeys q_add nk{nk} qs{q_shared}")


WINDOW_CASES = [
    # (B, H, W, heads, hd, ws, pool): none of these is taken by the tcgen05 Hiera kernel
    (2, 40, 40, 2, 72, 16, 1),   # 8-warp CTAs: 256-query windows, hd 72; W % ws != 0 -> padding tokens carry the bias
    (1, 64, 64, 4, 96, 8, 2),    # pooled 8x8 windows (16 queries, 1 warp)
    (1, 64, 64, 8, 96, 14, 2),   # pooled 14x14 windows, ragged: 64 = 4 x 14 + 8
    (1, 64, 64, 2, 96, 14, 1),   # 196-query windows, ragged
    (1, 62, 62, 2, 56, 4, 1),    # 4x4 windows (16-key tiles), ragged
    (2, 32, 32, 4, 72, 8, 2),    # hd 72 pooled
    (1, 32, 32, 2, 96, 0, 1),    # global, 1024 keys
]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["flat", "beacon", "ramp9", "distinct"])
@pytest.mark.parametrize("B,H,W,heads,hd,ws,pool", WINDOW_CASES)
def test_window_flash(ops, kind, B, H, W, heads, hd, ws, pool):
    """Route: window-mode flash_attn_kernel (sb_window_attention when the tcgen05 kernel does not apply): beacons per
    (batch entry, window, head) at the window's first / last key and the 63/64-key tile edges (window corners for small
    windows), q-pooling applied to queries that all carry the beacon direction."""
    wk = ws if 0 < ws < max(H, W) else max(H, W)
    tile = 16 if wk * wk <= 16 else 64
    qkv, bias = window_case(kind, B, H, W, heads, hd, ws, pool, tile=tile, seed=7)
    out = ops.window_attention(qkv, bias, B, H, W, heads, ws, pool)
    bb = bias.to(BF16)  # padding tokens carry the bias as the kernel stages it (bf16)
    args = (qkv, bb, B, H, W, heads, hd, ws, pool)
    assert_close(out, ref_window(*args), ref_window(*args, mode="bf16"), f"window {kind} {B, H, W, heads, hd, ws, pool}")


HIERA_CASES = [(1, 64, 64, 2, 16), (3, 64, 64, 8, 16), (1, 64, 64, 8, 0), (3, 64, 64, 2, 0), (1, 32, 64, 8, 0),
               (2, 32, 64, 2, 16)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["flat", "peaked", "beacon", "beacon2", "ramp9", "ramp5", "distinct"])
@pytest.mark.parametrize("B,H,W,heads,ws", HIERA_CASES)
def test_hiera_tc(ops, kind, B, H, W, heads, ws):
    """Route: hiera_attn_tc_kernel (head_dim 72, pool 1, 16x16 windows or global; persistent (crop, window, head,
    q-tile) items, P in TMEM): beacons per (crop, window, head) at the first / last key of the 128-key tiles (127/128,
    255/256, ... and the window's last key); ramps of 9 / 5 log2 units per 128-key tile."""
    qkv, _ = window_case(kind, B, H, W, heads, 72, ws, 1, tile=128, bias=False, seed=11)
    out = ops.hiera_attention_tc(qkv, B, H, W, heads, ws)
    args = (qkv, None, B, H, W, heads, 72, ws, 1)
    assert_close(out, ref_window(*args), ref_window(*args, mode="bf16"), f"hiera_tc {kind} {B, H, W, heads, ws}")


def t2i_case(kind, B, nt, nk, x_shared, splits, seed=12, device="cuda"):
    """Operands of ops.t2i_fold_attention. Beacons live in the positional key term kadd [nk, 128] (per head columns):
    group g of the (prompt, token) rows carries direction u_g in its queries, and kadd holds c u_g at key positions that
    differ per (group, head) and sit on the split boundaries; 'beacon2' gives each group two such keys."""
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn((1 if x_shared else B) * nk, 256, generator=gen)
    wk = torch.randn(128, 256, generator=gen) / 16
    wv = torch.randn(128, 256, generator=gen) / 16
    bv = torch.randn(128, generator=gen) * 0.02
    kadd = torch.randn(nk, 8, 16, generator=gen)
    q = torch.randn(B * nt, 8, 16, generator=gen) * 1.5
    if kind in ("beacon", "beacon2"):
        pos = edge_positions(nk, 32, splits=splits, limit=40)
        groups = [(p,) for p in pos] if kind == "beacon" else _pairs(pos, nk // splits)
        G = min(8, len(groups), B * nt)
        U = _orthonormal(G, 16, gen)
        a, c = 4.0, 60.0
        q = _project_out(q, U) + a * U[torch.arange(B * nt) % G][:, None, :]
        for h in range(8):
            for g in range(G):
                for p in groups[(g + h * G) % len(groups)]:
                    kadd[p, h] = c * U[g]
    else:
        assert kind == "flat", kind
    to = lambda t: t.to(BF16).to(device)  # noqa: E731
    return (to(q.reshape(B * nt, 128)), to(x), to(kadd.reshape(nk, 128)), to(wk), to(wv), bv.to(device))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["flat", "beacon", "beacon2"])
@pytest.mark.parametrize("B,nt,shared", [(1, 1, False), (3, 7, False), (3, 8, True), (100, 8, False), (100, 1, True)])
def test_t2i_fold(ops, kind, B, nt, shared):
    """Route: the tcgen05 fold kernel (64-key tiles) followed by t2i_unfold_kernel, which merges the key splits.
    Beacons at keys 0 / nk - 1, the first / last key of every split (sb_t2i_tc_splits) and the first tile edges."""
    from saber_b200 import lib
    nk = 4096
    L = lib.load()
    splits = L.sb_t2i_tc_splits(B, nk)
    q, x, kadd, wk, wv, bv = t2i_case(kind, B, nt, nk, shared, splits)
    out = ops.t2i_fold_attention(q, x, kadd, wk, wv, bv, B, nt, nk, x_shared=shared)
    args = (q, x, kadd, wk, wv, bv, B, nt, nk, shared)
    assert_close(out, ref_t2i(*args), ref_t2i(*args, mode="bf16"), f"t2i {kind} B{B} nt{nt} shared{shared} ns{splits}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["flat", "beacon"])
@pytest.mark.parametrize("B,heads,hd,nq,nk,kw", [(2, 2, 72, 33, 4097, {}), (3, 1, 256, 16, 8196, {}),
                                                 (3, 2, 64, 20, 1000, dict(q_shared=True)),
                                                 (3, 8, 16, 8, 4096, dict(kadd=True, kv_shared=True))])
def test_attention_f32(ops, kind, B, heads, hd, nq, nk, kw):
    """Route: sb_attention_f32 / its k_add form (fp32 validation mode: fp32 operands to ops.attention(_kadd));
    bars 1e-5 relative L2 and 2e-4 x rms, which back the validation mode's 1e-4 of the fp32 oracle."""
    kw = dict(kw)
    kadd = kw.pop("kadd", False)
    d = plain_case(kind, B, heads, hd, nq, nk, k_add=kadd, seed=21, **kw)
    q, k, v = d["q"].float(), d["k"].float(), d["v"].float()
    ka = d["k_add"].float() if kadd else None
    qs, kvs = kw.get("q_shared", False), kw.get("kv_shared", False)
    if kadd:
        out = ops.attention_kadd(q, k, ka, v, B, heads, nq, nk, kv_shared=kvs)
    else:
        out = ops.attention(q, k, v, B, heads, nq, nk, q_shared=qs, kv_shared=kvs)
    args = (q, k, v, B, heads, nq, nk, qs, kvs, ka)
    assert_close(out, ref_attention(*args), ref_attention(*args, mode="f32"), f"attn_f32 {kind} {B, heads, hd, nq, nk} {kw}",
                 fp32=True)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["flat", "beacon"])
@pytest.mark.parametrize("B,H,W,heads,hd,ws,pool", [(1, 40, 40, 2, 72, 16, 1), (1, 64, 64, 8, 96, 14, 2),
                                                    (2, 32, 32, 2, 72, 0, 1)])
def test_window_attention_f32(ops, kind, B, H, W, heads, hd, ws, pool):
    """Route: sb_window_attention_f32 (fp32 qkv to ops.window_attention): ragged windows whose padding carries the fp32
    bias, a pooled padded window, global attention."""
    qkv, bias = window_case(kind, B, H, W, heads, hd, ws, pool, seed=23)
    qkv = qkv.float()
    out = ops.window_attention(qkv, bias, B, H, W, heads, ws, pool)
    args = (qkv, bias, B, H, W, heads, hd, ws, pool)
    assert_close(out, ref_window(*args), ref_window(*args, mode="f32"), f"window_f32 {kind} {B, H, W, heads, hd, ws, pool}",
                 fp32=True)


# ------------------------------------------------------------------------------------------------------------------
# CPU: the bars are attainable and catch the defects they exist for (float64 model, no kernel involved)
# ------------------------------------------------------------------------------------------------------------------
CPU_SHAPES = [(72, 4096), (256, 8196), (16, 4096)]  # (head_dim, keys); 2 batch entries x 2 heads x 48 queries
CPU_KINDS = ["flat", "peaked", "beacon", "cold"]


def _cpu_instance(hd, nk, kind):
    B, heads, nq = 2, 2, 48
    d = plain_case(kind, B, heads, hd, nq, nk, tile=64, seed=hd + nk, device="cpu")
    return d["q"], d["k"], d["v"], B, heads, nq


def _defective(defect, q, k, v, B, heads, nq, nk):
    """The emulated bf16 kernel with one defect."""
    C = k.shape[1]
    kk = k.float().view(B, nk, C)
    vv = v.float().view(B, nk, C)
    post = None
    if defect == "scale_0.99":
        post = lambda o: o * 0.99  # noqa: E731
    elif defect == "swap_batch":
        post = lambda o: o.view(B, nq, C).flip(0).reshape(B * nq, C)  # noqa: E731
    elif defect == "pad60_counted":  # 60 zero keys (score 0) and zero values inside the softmax
        kk = torch.cat([kk, torch.zeros(B, 60, C)], 1)
        vv = torch.cat([vv, torch.zeros(B, 60, C)], 1)
    elif defect == "beacon_from_neighbour_tile":  # the rows at the beacon positions are read one tile further on
        kk, vv = kk.clone(), vv.clone()
        for p in edge_positions(nk, 64):
            src = p + 64 if p + 64 < nk else p - 64
            kk[:, p], vv[:, p] = kk[:, src], vv[:, src]
    else:
        keep = torch.ones(nk, dtype=torch.bool)
        keep[{"drop_last": slice(nk - 1, nk), "drop_first": slice(0, 1), "drop_last4": slice(nk - 4, nk),
              "drop_tile": slice(64, 128)}[defect]] = False
        kk, vv = kk[:, keep], vv[:, keep]
    n = kk.shape[1]
    o = ref_attention(q, kk.reshape(B * n, C), vv.reshape(B * n, C), B, heads, nq, n, mode="bf16")
    return post(o) if post else o


DEFECTS = ["scale_0.99", "drop_last", "drop_first", "drop_last4", "drop_tile", "pad60_counted",
           "beacon_from_neighbour_tile", "swap_batch"]
# Input kinds on which a defect can pass the bars. One key among 4096-8196 random keys moves the output by about as much
# as bf16 rounding does when its score is not above the others (peaked scores at head_dim 256: drop_last 2.4e-3, drop_first
# 2.6e-3 relative L2); the beacon input puts a hot key on those positions for some query rows and catches both. Zero-score
# padding keys weigh nothing once real scores are far above 0 (peaked, beacon) and about the rounding floor among 8196
# keys at head_dim 256 (flat: 5.0e-3); the cold input, whose real scores all sit ~6 nats below 0, catches it everywhere.
CPU_MISSES = {"drop_last": {"peaked"}, "drop_first": {"peaked"}, "pad60_counted": {"flat", "peaked", "beacon"}}


@pytest.mark.parametrize("hd,nk", CPU_SHAPES)
@pytest.mark.parametrize("kind", CPU_KINDS)
def test_cpu_emulated_floor_has_2x_margin(hd, nk, kind):
    q, k, v, B, heads, nq = _cpu_instance(hd, nk, kind)
    ref = ref_attention(q, k, v, B, heads, nq, nk)
    rel, mx = _errors(ref_attention(q, k, v, B, heads, nq, nk, mode="bf16"), ref)
    assert rel <= BF16_BARS[0] / 2 and mx <= BF16_BARS[1] / 2, (rel, mx)


@pytest.mark.parametrize("hd,nk", CPU_SHAPES)
@pytest.mark.parametrize("defect", DEFECTS)
def test_cpu_defect_fails_the_bar(defect, hd, nk):
    """Each modelled defect fails a bar on every input kind except the ones listed in CPU_MISSES, and on at least one
    structured kind (beacon or cold)."""
    caught = {}
    for kind in CPU_KINDS:
        q, k, v, B, heads, nq = _cpu_instance(hd, nk, kind)
        ref = ref_attention(q, k, v, B, heads, nq, nk)
        rel, mx = _errors(_defective(defect, q, k, v, B, heads, nq, nk), ref)
        caught[kind] = (rel > BF16_BARS[0] or mx > BF16_BARS[1], rel, mx)
    for kind, (ok, rel, mx) in caught.items():
        assert ok or kind in CPU_MISSES.get(defect, ()), f"{defect} passes the bars on {kind}: rel {rel:.2e}, max/rms {mx:.3f}"
    assert caught["beacon"][0] or caught["cold"][0]
