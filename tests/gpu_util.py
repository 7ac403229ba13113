"""Helpers shared by the -m gpu tests: build reference-layout parameters from a logical
synthetic layer (oracle), error diagnostics, and the recorded outputs of the reference's kernels
(tests/golden/ref_parity_golden.npz, written by tests/golden/make_ref_parity_golden.py)."""
from __future__ import annotations

import os

import numpy as np
import torch

from oracle import formats as F
from oracle import svdq as O


def ref_layout_params(layer: O.SynthLayer, device="cuda") -> dict:
    """Logical synthetic layer -> the reference's packed checkpoint tensors on ``device``."""
    N, K = layer.qw.shape
    p = {}
    p["qweight"] = F.pack_qweight(layer.qw).to(device)
    if layer.fp4:
        p["wscales"] = F.pack_micro_scales(layer.wscales).view(torch.float8_e4m3fn).to(device)
    else:
        p["wscales"] = F.pack_group_scales(layer.wscales).to(device)
    p["bias"] = F.pack_channel_vector(layer.bias).to(device)
    p["smooth"] = F.pack_channel_vector(layer.smooth).to(device)
    p["proj_up"] = F.pack_lowrank(layer.lora_up, down=False).to(device)
    p["proj_down"] = F.pack_lowrank(layer.lora_down, down=True).to(device)
    p["wcscales"] = None if layer.wcscales is None else F.pack_channel_vector(layer.wcscales).to(device)
    return p


def diag(name: str, test: torch.Tensor, ref: torch.Tensor, blk: int = 32) -> str:
    """Human-readable mismatch report (printed on failure so one GPU run is enough to debug)."""
    t, r = test.detach().double().cpu(), ref.detach().double().cpu()
    lines = [f"[{name}] shape {tuple(t.shape)} rel_fro {O.rel_fro(t, r):.4e} max_abs {float((t - r).abs().max()):.4e} "
             f"ref_absmax {float(r.abs().max()):.4e} nan {int(torch.isnan(t).sum())}"]
    if t.dim() == 2:
        M, N = t.shape
        e = (t - r).abs()
        bm, bn = min(blk, M), min(blk, N)
        eb = e[: M // bm * bm, : N // bn * bn].reshape(M // bm, bm, N // bn, bn).amax(dim=(1, 3))
        rb = r.abs()[: M // bm * bm, : N // bn * bn].reshape(M // bm, bm, N // bn, bn).amax(dim=(1, 3)) + 1e-30
        bad = (eb / rb > 0.05)
        lines.append(f"  bad {bm}x{bn} blocks: {int(bad.sum())}/{bad.numel()}  rows-with-bad {bad.any(1).nonzero().flatten()[:16].tolist()} "
                     f"cols-with-bad {bad.any(0).nonzero().flatten()[:16].tolist()}")
        lines.append(f"  test[0,:8] {t[0, :8].tolist()}")
        lines.append(f"  ref [0,:8] {r[0, :8].tolist()}")
        lines.append(f"  test[-1,-8:] {t[-1, -8:].tolist()}")
        lines.append(f"  ref [-1,-8:] {r[-1, -8:].tolist()}")
    return "\n".join(lines)


REF_PARITY_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_parity_golden.npz")


def sample_index(numel: int, n: int) -> torch.Tensor:
    """``min(n, numel)`` distinct flat indices spread over ``[0, numel)``: i * p mod numel with p prime and larger than any
    tensor here, so the selection is fixed by the shape alone"""
    return torch.arange(min(n, numel), dtype=torch.int64) * 2654435761 % numel


def sample(t: torch.Tensor, n: int = 4096) -> torch.Tensor:
    """the elements of ``t`` at ``sample_index``, on the CPU: what the golden file keeps of a full-size output"""
    flat = t.detach().reshape(-1)
    return flat[sample_index(flat.numel(), n).to(flat.device)].cpu()


def fingerprint(*inputs: torch.Tensor) -> np.ndarray:
    """64 sampled elements of each input, exactly (float64 holds every int32 / 16-bit value)"""
    return torch.cat([sample(t, 64).double() for t in inputs]).numpy()


def ref_golden(case: str, *inputs: torch.Tensor) -> dict:
    """The reference kernels' recorded results for ``case`` ({name: tensor}; 16-bit floats are stored as their bits under
    "<name>@<dtype>"), after checking that ``inputs`` are the tensors they were recorded on: the tests rebuild their inputs
    from seeds, and a changed random stream must fail here instead of comparing unrelated numbers."""
    g = np.load(REF_PARITY_GOLDEN)
    assert np.array_equal(fingerprint(*inputs), g[case + ".inputs"]), f"{case}: inputs differ from those the reference outputs were recorded on"
    out = {}
    for k in g.files:
        if k.startswith(case + "."):
            name, _, dt = k[len(case) + 1:].partition("@")
            out[name] = torch.from_numpy(g[k]).view(getattr(torch, dt)) if dt else torch.from_numpy(g[k])
    return out
