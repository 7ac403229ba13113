"""GPU parity of the tcgen05 attention (SURVEY section 8f row N1, csrc/attention.cu): against exact math (oracle/attention.py, fp64), against
the reference kernel's committed B200 outputs, and against what the reference kernel computed on a B200 with padded / masked keys at
FLUX head counts (tests/golden/make_ref_parity_golden.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import attention as AT
from oracle import svdq as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "ref_gpu_golden.npz")


def _run(q, k, v, out_dtype, scale=128 ** -0.5):
    from nunchaku_b200.ops.attention import attention_fp16

    B, H, T, _ = q.shape
    o = torch.full((B, T, H * 128), float("nan"), dtype=out_dtype, device="cuda")
    attention_fp16(q.cuda(), k.cuda(), v.cuda(), o, scale)
    torch.cuda.synchronize()
    return o.cpu()


@pytest.mark.parametrize("dtn", ["float16", "bfloat16"])
def test_attention_matches_reference_golden_and_exact_math(dtn):
    g = np.load(GOLD)
    dt = getattr(torch, dtn)
    qkv = torch.from_numpy(g["attn.qkv"].astype(np.int16)).view(torch.float16)
    q, k, v = AT.pack_qkv_rowmajor(qkv, heads=2, tokens_pad=512)
    o = _run(q, k, v, dt)
    exact = AT.attention_fp16(q, k, v, 128 ** -0.5)
    ref = torch.from_numpy(g[f"attn.ref_o_{dtn}"].astype(np.int16)).view(dt)
    ours_vs_exact, ref_vs_exact, ours_vs_ref = O.rel_fro(o, exact), O.rel_fro(ref, exact), O.rel_fro(o, ref)
    # fp32 accumulation: closer to exact math than the reference's fp16 accumulation, within the output rounding
    assert ours_vs_exact <= (6e-4 if dt == torch.float16 else 3e-3), (ours_vs_exact, ref_vs_exact)
    assert ours_vs_exact <= ref_vs_exact * 1.05 + 1e-5 and ours_vs_ref <= (2e-3 if dt == torch.float16 else 5e-3), (ours_vs_exact, ref_vs_exact, ours_vs_ref)


@pytest.mark.parametrize("T,Tpad,H,B", [(300, 512, 3, 1), (128, 128, 1, 2), (1000, 1024, 2, 1)])
def test_attention_masks_padded_keys(T, Tpad, H, B):
    g = torch.Generator().manual_seed(T)
    qs, ks, vs = [], [], []
    for _ in range(B):
        qkv = (torch.randn(T, 3 * H * 128, generator=g) * 0.7).to(torch.float16)
        q, k, v = AT.pack_qkv_rowmajor(qkv, heads=H, tokens_pad=Tpad)
        qs.append(q), ks.append(k), vs.append(v)
    q, k, v = torch.cat(qs), torch.cat(ks), torch.cat(vs)
    o = _run(q, k, v, torch.float16)
    exact = AT.attention_fp16(q, k, v, 128 ** -0.5)
    assert torch.isfinite(o[:, :T].float()).all()
    assert O.rel_fro(o[:, :T], exact[:, :T]) <= 6e-4
    # large scores: the running maximum moves late (rescale path) and probabilities span the fp16 range
    q2 = q * 6.0
    o2 = _run(q2, k, v, torch.float16)
    assert O.rel_fro(o2[:, :T], AT.attention_fp16(q2, k, v, 128 ** -0.5)[:, :T]) <= 1.5e-3


FLUX_T, FLUX_TPAD, FLUX_H = 4352, 4608, 24


def flux_qkv():
    """the projection both kernels read: [T, 3 * H * 128] fp16, followed in the generator by the pad rows the reference's run needs"""
    g = torch.Generator(device="cuda").manual_seed(3)
    return g, (torch.randn(FLUX_T, 3 * FLUX_H * 128, generator=g, device="cuda") * 0.5).to(torch.float16)


def test_attention_flux_size_vs_reference_kernel_live():
    """24 heads, 4352 valid of 4608 padded tokens: our kernel on the PackQKV-layout tensors vs what the reference kernel computed on a
    B200 on ITS packed layout of the same projection (produced by its own test_pack_qkv hook, pad keys masked)"""
    from gpu_util import ref_golden, sample

    T, Tpad, H = FLUX_T, FLUX_TPAD, FLUX_H
    _, qkv = flux_qkv()
    o_ref = ref_golden("attn_flux", qkv)["o"]
    q = torch.zeros(1, H, Tpad, 128, dtype=torch.float16, device="cuda")
    k = torch.full_like(q, float("nan"))
    v = torch.zeros_like(q)
    for t, i in ((q, 0), (k, 1), (v, 2)):
        t[0, :, :T] = qkv[:, i * H * 128:(i + 1) * H * 128].view(T, H, 128).transpose(0, 1)
    from nunchaku_b200.ops.attention import attention_fp16

    o = torch.empty(1, Tpad, H * 128, dtype=torch.float16, device="cuda")
    attention_fp16(q, k, v, o, 128 ** -0.5)
    torch.cuda.synchronize()
    assert torch.isfinite(o[:, :T].float()).all()
    rel = O.rel_fro(sample(o[:, :T], o_ref.numel()), o_ref)
    assert rel <= 2e-3, rel
    # and both against fp32 math on the GPU for a few heads
    sl = slice(0, 3)
    s = torch.einsum("hid,hjd->hij", q[0, sl, :T].float(), k[0, sl, :T].float()) * 128 ** -0.5
    want = (torch.softmax(s, -1) @ v[0, sl, :T].float()).transpose(0, 1).reshape(T, 3 * 128)
    assert O.rel_fro(o[0, :T, : 3 * 128].float().cpu(), want.cpu()) <= 6e-4
