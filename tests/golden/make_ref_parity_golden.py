"""Record what the UNMODIFIED reference kernels compute for the full-size parity tests, so that those tests compare with the
reference on any B200 without its library:

    tests/test_gpu_vs_reference.py   linear / fused MLP / QKV+RMSNorm+RoPE through the reference's GEMM_W4A4, glue kernels
    tests/test_gpu_awq.py            gemv_awq at the FLUX AdaLN size
    tests/test_gpu_attention.py      test_pack_qkv -> attention_fp16 at 24 heads, 4352 of 4608 tokens

Needs a B200 and oracle/_ref/libnunchaku_ref.so (oracle/ref_build/build_ref.sh):

    python tests/golden/make_ref_parity_golden.py OUT_DIR      # writes OUT_DIR/ref_parity_golden.npz, then copy it to tests/golden/

Each case is built by the test's own input function from its seeds.  Per case the file keeps a fingerprint of the inputs
(gpu_util.fingerprint), a fixed sample of the reference's output (gpu_util.sample) and, for the linears, the reference's
distance from exact math over the WHOLE output.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

TESTS = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.dirname(TESTS), TESTS]

import test_gpu_attention as AT  # noqa: E402
import test_gpu_awq as AW  # noqa: E402
import test_gpu_vs_reference as VR  # noqa: E402
from gpu_util import fingerprint, sample  # noqa: E402
from oracle import refgpu as R  # noqa: E402
from oracle import svdq as O  # noqa: E402


def main(out_dir: str) -> None:
    assert R.available("ref"), "oracle/_ref/libnunchaku_ref.so missing: run oracle/ref_build/build_ref.sh where the reference's sources are"
    out = {}

    def put(case, inputs, **arrays):
        out[case + ".inputs"] = fingerprint(*inputs)
        for k, v in arrays.items():
            if isinstance(v, torch.Tensor) and v.dtype in (torch.bfloat16, torch.float16):
                out[f"{case}.{k}@{VR.dtype_name(v.dtype)}"] = v.view(torch.int16).numpy()
            else:
                out[f"{case}.{k}"] = v.numpy() if isinstance(v, torch.Tensor) else np.asarray(v)
        print(case, {k: (tuple(v.shape) if isinstance(v, torch.Tensor) else v) for k, v in arrays.items()}, flush=True)

    for M, K, N, hT in VR.linear_cases():
        key, layer, ck, x, inputs = VR.linear_case(M, K, N, hT)
        y = VR.ref_module(layer, ck, "ref").forward(x)
        torch.cuda.synchronize()
        put(key, inputs, ref=sample(y), ref_vs_exact=O.rel_fro(y.cpu(), VR.exact_linear(layer, x).cpu()))
    for M in (256, 4352):
        key, l1, l2, c1, c2, x, inputs = VR.mlp_case(M)
        y = VR.ref_module(l1, c1, "ref").forward_mlp(VR.ref_module(l2, c2, "ref"), x)
        torch.cuda.synchronize()
        put(key, inputs, ref=sample(y))
    for hT in (torch.bfloat16, torch.float16):
        key, layer, ck, x, norm_q, norm_k, rot, inputs = VR.qkv_case(hT)
        y = VR.ref_module(layer, ck, "ref").forward_qkv(x, norm_q, norm_k, rot)
        torch.cuda.synchronize()
        put(key, inputs, ref=sample(y))
    for hT, t in VR.glue_case():
        res = {}
        for name, fn in VR.glue_ops("ref", **t).items():
            r = fn()
            torch.cuda.synchronize()
            if name == "split_mod":
                res.update({f"split_mod{i}": sample(o) for i, o in enumerate(r)})
            else:
                res[name] = sample(r)
        put(f"glue_{VR.dtype_name(hT)}", t.values(), **res)

    qw, per = AW.adaln_case()
    OC, IC = qw.shape[0] * 4, qw.shape[1] * 2
    ys = {VR.dtype_name(hT): sample(R.gemv_awq(x, qw, sc, ze, 1, OC, IC, 64)) for hT, sc, ze, x in per}
    put("awq_adaln", [qw] + [t for _, sc, ze, x in per for t in (sc, ze, x)], **ys)

    T, Tpad, H = AT.FLUX_T, AT.FLUX_TPAD, AT.FLUX_H
    g, qkv = AT.flux_qkv()
    rq = torch.zeros(1, H, Tpad, 128, dtype=torch.float16, device="cuda")
    rk, rv = torch.zeros_like(rq), torch.zeros_like(rq)
    qkv_pad = torch.cat([qkv, torch.randn(Tpad - T, 3 * H * 128, generator=g, device="cuda").to(torch.float16)])   # the GEMM computes pad rows too;
    R.test_pack_qkv(qkv_pad, rq, rk, rv, T)                                                                         # the epilogue masks them (0 / NaN / 0)
    assert torch.isnan(rk.view(-1)[-1:]).all() or torch.isnan(rk).any()
    o_ref = torch.empty(1, Tpad, H * 128, dtype=torch.float16, device="cuda")
    R.attention_fp16(rq, rk, rv, o_ref, 128 ** -0.5)
    torch.cuda.synchronize()
    assert torch.isfinite(o_ref[:, :T].float()).all()
    put("attn_flux", [qkv], o=sample(o_ref[:, :T], 8192))

    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "ref_parity_golden.npz")
    np.savez_compressed(path, device=np.asarray(torch.cuda.get_device_name(0)), **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main(sys.argv[1])
