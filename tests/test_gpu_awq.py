"""GPU parity of the AWQ W4A16 GEMV (SURVEY section 8f row N2): against the oracle (oracle/awq.py, bit-exact with the reference's kernel
on its golden vectors: tests/test_ref_gpu_golden.py), against the committed reference-on-B200 outputs themselves, at the FLUX AdaLN
sizes against the reference kernel's recorded outputs (tests/golden/make_ref_parity_golden.py), and -- when the seam library is
built -- through the reference's own host entry point."""
import os

import numpy as np
import pytest
import torch

from oracle import awq as A
from oracle import svdq as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "ref_gpu_golden.npz")


def _close(y, want, name):
    eq = float((y.cpu().view(torch.int16) == want.cpu().view(torch.int16)).double().mean())
    rel = O.rel_fro(y.cpu(), want.cpu())
    assert rel <= 2e-3 and eq >= 0.98, (name, rel, eq)   # same products, different fp32 summation order


@pytest.mark.parametrize("dtn", ["bfloat16", "float16"])
def test_gemv_awq_matches_reference_golden(dtn):
    from nunchaku_b200.ops.gemv import awq_gemv_w4a16_cuda

    g = np.load(GOLD)
    dt = getattr(torch, dtn)
    ht = lambda a: torch.from_numpy(a.astype(np.int16)).view(dt)  # noqa: E731
    qw = torch.from_numpy(g["awq.qweight"]).cuda()
    sc, ze = ht(g[f"awq_{dtn}.scales"]).cuda(), ht(g[f"awq_{dtn}.zeros"]).cuda()
    for m in (1, 3):
        x = ht(g[f"awq_{dtn}.x{m}"]).cuda()
        y = awq_gemv_w4a16_cuda(x, qw, sc, ze, m, 256, 3072, 64)
        torch.cuda.synchronize()
        _close(y, ht(g[f"awq_{dtn}.ref_y{m}"]), f"golden {dtn} m={m}")


@pytest.mark.parametrize("m", [1, 2, 8])
@pytest.mark.parametrize("hT", [torch.bfloat16, torch.float16])
def test_gemv_awq_vs_oracle_and_layer(m, hT):
    from nunchaku_b200.ops.gemv import AWQW4A16Linear

    g = torch.Generator().manual_seed(m)
    OC, IC = 512, 1024
    codes = torch.randint(0, 16, (OC, IC), generator=g, dtype=torch.uint8)
    layer = AWQW4A16Linear(IC, OC, bias=True, torch_dtype=hT, device="cuda")
    sc = (torch.rand(IC // 64, OC, generator=g) * 0.02 + 0.005).to(hT)
    ze = (-(torch.rand(IC // 64, OC, generator=g) * 0.1 + 0.03)).to(hT)
    bias = torch.randn(OC, generator=g).to(hT)
    x = torch.randn(m, IC, generator=g).to(hT)
    layer.load_state_dict({"qweight": A.pack_awq_qweight(codes), "wscales": sc, "wzeros": ze, "bias": bias})
    y = layer(x.cuda())
    torch.cuda.synchronize()
    want = (A.gemv_awq(x, A.pack_awq_qweight(codes), sc, ze).double() + bias.double()).to(hT)   # output.add_(bias): one more hT rounding
    _close(y, want, f"oracle {hT} m={m}")


def adaln_case():
    """-> (qweight, [(dtype, scales, zeros, x)]) in the order they are drawn"""
    g = torch.Generator(device="cuda").manual_seed(5)
    OC, IC = 18432, 3072
    qw = torch.randint(-2 ** 31, 2 ** 31 - 1, (OC // 4, IC // 2), generator=g, device="cuda", dtype=torch.int64).to(torch.int32)
    per = []
    for hT in (torch.bfloat16, torch.float16):
        sc = (torch.rand(IC // 64, OC, generator=g, device="cuda") * 0.02 + 0.005).to(hT)
        ze = (-(torch.rand(IC // 64, OC, generator=g, device="cuda") * 0.1 + 0.03)).to(hT)
        x = torch.randn(1, IC, generator=g, device="cuda").to(hT)
        per.append((hT, sc, ze, x))
    return qw, per


def test_gemv_awq_flux_adaln_size_vs_reference_kernel_live():
    """FLUX AdaLN: 3072 -> 18432 (6 x dim), batch 1: our kernel vs what the reference's kernel computed on a B200 from the same
    checkpoint bytes"""
    from gpu_util import ref_golden, sample
    from nunchaku_b200.ops.gemv import awq_gemv_w4a16_cuda

    qw, per = adaln_case()
    OC, IC = qw.shape[0] * 4, qw.shape[1] * 2
    gold = ref_golden("awq_adaln", qw, *[t for _, sc, ze, x in per for t in (sc, ze, x)])
    for hT, sc, ze, x in per:
        y = awq_gemv_w4a16_cuda(x, qw, sc, ze, 1, OC, IC, 64)
        torch.cuda.synchronize()
        want = gold[str(hT).split(".")[-1]]
        _close(sample(y, want.numel()), want, f"live {hT}")


def test_gemv_awq_through_the_cpp_seam_and_the_pybind_surface():
    """the reference's host entry point `gemv_awq(Tensor...)` (src/kernels/awq/gemv_awq.h) defined on our kernel (csrc/seam/awq_b200.cpp):
    through the seam library's C shim and through `nunchaku._C.ops.gemv_awq` -- bit-identical to the Python operator"""
    import importlib.util

    from oracle import refgpu as R

    if not R.available("seam"):
        pytest.skip("oracle/_ref/libnunchaku_seam.so not built")
    from nunchaku_b200.ops.gemv import awq_gemv_w4a16_cuda

    g = torch.Generator(device="cuda").manual_seed(9)
    OC, IC, m = 1024, 3072, 2
    qw = torch.randint(-2 ** 31, 2 ** 31 - 1, (OC // 4, IC // 2), generator=g, device="cuda", dtype=torch.int64).to(torch.int32)
    sc = (torch.rand(IC // 64, OC, generator=g, device="cuda") * 0.02 + 0.005).to(torch.bfloat16)
    ze = (-(torch.rand(IC // 64, OC, generator=g, device="cuda") * 0.1 + 0.03)).to(torch.bfloat16)
    x = torch.randn(m, IC, generator=g, device="cuda").to(torch.bfloat16)
    y = awq_gemv_w4a16_cuda(x, qw, sc, ze, m, OC, IC, 64)
    assert torch.equal(R.gemv_awq(x, qw, sc, ze, m, OC, IC, 64, lib="seam"), y)
    so = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "pyseam", "_C.so")
    if os.path.exists(so):
        spec = importlib.util.spec_from_file_location("_C", so)
        C = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(C)
        assert torch.equal(C.ops.gemv_awq(x, qw, sc, ze, m, OC, IC, 64), y)


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16])
def test_gemv_fused_silu_bias_equals_three_launches(dt):
    """silu -> gemv -> + bias as one launch (nb200_gemv_awq_fused, SURVEY row N2) == the three separate launches, bit for bit"""
    from nunchaku_b200.ops import glue
    from nunchaku_b200.ops.gemv import awq_gemv_w4a16_cuda

    g = torch.Generator(device="cuda").manual_seed(11)
    IC, OC = 3072, 18432
    x = torch.randn(1, IC, generator=g, device="cuda").to(dt)
    qw = torch.randint(-2 ** 31, 2 ** 31 - 1, (OC // 4, IC // 2), generator=g, device="cuda", dtype=torch.int64).to(torch.int32)
    sc = (0.01 + 0.01 * torch.rand(IC // 64, OC, generator=g, device="cuda")).to(dt)
    zr = (-0.08 * torch.rand(IC // 64, OC, generator=g, device="cuda")).to(dt)
    bias = (0.1 * torch.randn(OC, generator=g, device="cuda")).to(dt)
    want = awq_gemv_w4a16_cuda(glue.silu(x), qw, sc, zr, 1, OC, IC).add_(bias)
    got = awq_gemv_w4a16_cuda(x, qw, sc, zr, 1, OC, IC, bias=bias, fuse_silu=True)
    torch.cuda.synchronize()
    assert torch.equal(got.view(torch.int16), want.view(torch.int16))
