"""Fused tcgen05 attention (pixray_b200/csrc/attn_tc.cu) against a torch fp32 restatement of nn.MultiheadAttention's
core (SLIP/models.py:18-64 residual blocks call it with need_weights=False): S = q k^T / sqrt(d), P = softmax(S),
O = P v, and its backward.  Tolerances: fp16 operands / fp32 accumulate vs fp32 math on the same fp16 inputs."""
import ctypes as C

import pytest
import torch

from pixray_b200 import _lib

pytestmark = pytest.mark.gpu


def _run(qkv, d_o, B, T, H, repeat=1):
    lib = _lib.load()
    W = 64 * H
    o = torch.zeros(B * T, W, dtype=torch.half, device="cuda")
    lse = torch.zeros(B * H * T, dtype=torch.float32, device="cuda")
    gqkv = torch.zeros(B * T, 3 * W, dtype=torch.half, device="cuda") if d_o is not None else None
    err = C.create_string_buffer(512)
    rc = lib.pxr_test_attention(C.c_void_p(qkv.data_ptr()), C.c_void_p(o.data_ptr()), C.c_void_p(lse.data_ptr()),
                                C.c_void_p(d_o.data_ptr()) if d_o is not None else None,
                                C.c_void_p(gqkv.data_ptr()) if gqkv is not None else None, B, T, H, W,
                                C.c_float(0.125), repeat, err, 512)
    assert rc == 0, err.value.decode()
    torch.cuda.synchronize()
    return o, lse, gqkv


def _reference(qkv, d_o, B, T, H):
    W = 64 * H
    x = qkv.float().view(B, T, 3, H, 64).permute(2, 0, 3, 1, 4).contiguous().requires_grad_(True)  # [3,B,H,T,64]
    q, k, v = x[0], x[1], x[2]
    s = (q @ k.transpose(-1, -2)) * 0.125
    p = s.softmax(-1)
    o = p @ v  # [B,H,T,64]
    lse = torch.logsumexp(s, -1)  # [B,H,T]
    g = d_o.float().view(B, T, H, 64).permute(0, 2, 1, 3)
    (gx,) = torch.autograd.grad(o, x, g)
    o_flat = o.permute(0, 2, 1, 3).reshape(B * T, W)
    g_flat = gx.permute(1, 3, 0, 2, 4).reshape(B * T, 3 * W)  # [B,T,3,H,64]
    return o_flat.detach(), lse.reshape(-1).detach(), g_flat


def _report(name, got, ref):
    err = (got.float() - ref).abs()
    m = ref.abs().max().item()
    idx = err.argmax().item()
    shape = tuple(ref.shape)
    pos = [] if ref.dim() == 1 else [idx // shape[1], idx % shape[1]]
    line = f"{name}: max_abs_err {err.max().item():.4e} (max |ref| {m:.4e}) at {pos or idx} nan={torch.isnan(got.float()).sum().item()}"
    print(line)
    return err.max().item(), m


@pytest.mark.parametrize("B,T,H", [(2, 197, 12), (3, 50, 4), (1, 240, 2), (2, 130, 3), (5, 64, 2), (1, 16, 1), (150, 197, 1),
                                   # several (image, head) items per CTA at T <= 128 (ViT-B/32 with many cutouts)
                                   (40, 50, 12), (13, 128, 12)])
def test_attention_matches_torch(B, T, H):
    torch.manual_seed(B * 1000 + T)
    W = 64 * H
    qkv = (torch.randn(B * T, 3 * W, device="cuda") * 1.5).half()
    d_o = torch.randn(B * T, W, device="cuda").half()
    o, lse, gqkv = _run(qkv, d_o, B, T, H)
    ro, rl, rg = _reference(qkv, d_o, B, T, H)
    eo, mo = _report("o", o, ro)
    el, ml = _report("lse", lse, rl)
    edq, mdq = _report("dq", gqkv[:, :W], rg[:, :W])
    edk, mdk = _report("dk", gqkv[:, W:2 * W], rg[:, W:2 * W])
    edv, mdv = _report("dv", gqkv[:, 2 * W:], rg[:, 2 * W:])
    assert eo <= 4e-3 * max(mo, 1.0)
    assert el <= 2e-3 * max(ml, 1.0)
    assert edq <= 1e-2 * mdq and edk <= 1e-2 * mdk and edv <= 1e-2 * mdv


def test_attention_throughput_report():
    """Config-2 shape (64 images x 12 heads x 197 tokens): time per call, reported (not asserted)."""
    B, T, H = 64, 197, 12
    W = 64 * H
    qkv = torch.randn(B * T, 3 * W, device="cuda").half()
    d_o = torch.randn(B * T, W, device="cuda").half()
    _run(qkv, None, B, T, H, repeat=3)
    _run(qkv, d_o, B, T, H, repeat=3)
    lines = []
    for name, g in (("fwd", None), ("fwd+bwd", d_o)):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        _run(qkv, g, B, T, H, repeat=20)
        e1.record()
        torch.cuda.synchronize()
        lines.append(f"attention {name} B={B} T={T} H={H}: {e0.elapsed_time(e1) / 20 * 1e3:.1f} us per call")
    print("\n".join(lines))
