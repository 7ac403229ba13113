#!/usr/bin/env python
"""bench.py -- FLUX.1-schnell 1024x1024 4-step: the SVDQuant W4A4 + low-rank hot path of every transformer block on B200.

A "step" is one denoising step's worth of the hot path (SURVEY.md section 8), CHAINED the way the model chains it:

    joint block (x19), image stream (4096 tokens) and text stream (256 tokens) each:
        LayerNorm -> QKV projection with RMSNorm(Q,K) + RoPE in the GEMM epilogue -> [attention: NOT run, out of scope]
        -> out projection -> LayerNorm -> fc1 -> GELU -> fc2 (fc2's 4-bit input produced by fc1's epilogue / the split route) -> add
    single block (x38), 4352 tokens: LayerNorm -> QKV(+RMSNorm+RoPE) -> out projection ; fc1 -> GELU -> fc2 ; add

= 304 fused W4A4 GEMM launches + the activation quantizers + the LayerNorm / add glue kernels (row a14), at the model's
exact shapes, rank 32, random-init 4-bit weights in the reference's checkpoint layout (no checkpoints offline).  Every layer
reads its predecessor's output; the out projection reads the first M x 3072 elements of the QKV result as the stand-in for
the attention output.  Attention itself and the AdaLN modulation GEMVs are outside the hot path and not run.
An image is 4 steps.  value = images/s of this stack, whole job over all ranks (replicas, no collective in the timed path).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--precision nvfp4|int4] [--impl reference] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step returned (the hidden states after the 57 blocks, [4352, 3072]) as
DIR/hidden_states.npy in float32 (53 MB).  Inputs and weights come from fixed seeds, so two builds run with the same arguments
can be compared output for output.

One JSON line on stdout (driver contract + roofline, cpu_baseline, e2e, clocks, gpu_launches, reference_gpu, cublas_bf16).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DIM, MLP, RANK, HEADS = 3072, 12288, 32, 24
IMG_TOKENS, TXT_TOKENS = 4096, 256
N_JOINT, N_SINGLE = 19, 38
STEPS_PER_IMAGE = 4
METRIC = "FLUX.1-schnell 1024px 4-step images/sec (SVDQuant W4A4+LR linear stack)"

# (name, K, N)
BLOCK_LINEARS = [("qkv", DIM, 3 * DIM), ("out", DIM, DIM), ("fc1", DIM, MLP), ("fc2", MLP, DIM)]


def block_list():
    """[(tag, M)] stream-blocks of one denoising step in execution order; each runs the four linears of BLOCK_LINEARS."""
    blocks = []
    for b in range(N_JOINT):
        blocks.append((f"joint{b}.img", IMG_TOKENS))
        blocks.append((f"joint{b}.txt", TXT_TOKENS))
    for b in range(N_SINGLE):
        blocks.append((f"single{b}", IMG_TOKENS + TXT_TOKENS))
    return blocks


def layer_list():
    """[(tag, M, K, N)] for one denoising step, in execution order (304 linears)."""
    return [(f"{tag}.{name}", M, K, N) for tag, M in block_list() for name, K, N in BLOCK_LINEARS]


def step_flops():
    f_main = f_lr = 0
    for _, M, K, N in layer_list():
        f_main += 2 * M * K * N
        f_lr += 2 * M * RANK * (K + N)
    return f_main, f_lr


def gemm_bytes(M, K, N, R, fp4):
    """algorithmic bytes of one fused GEMM launch (SURVEY section 8d)"""
    G, s = (16, 1) if fp4 else (64, 2)
    Mp = (M + 255) // 256 * 256
    return Mp * K // 2 + (K // G) * Mp * s + N * K // 2 + (K // G) * N * s + 4 * Mp * R + 2 * N * R + 4 * N + 2 * M * N


def host_threads() -> int:
    """threads this process may actually use: the affinity mask, capped by the cgroup CPU quota when one is set (a box whose mask shows 128 CPUs
    behind a quota of a few cores runs 128 OpenMP threads SLOWER than 8 -- r01: the same sample took 41 ms on one box and 651 ms on another)"""
    try:
        n = max(1, len(os.sched_getaffinity(0)))
    except AttributeError:  # pragma: no cover
        n = os.cpu_count() or 1
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:      # cgroup v2: "<quota|max> <period>"
            q, per = f.read().split()[:2]
            if q != "max":
                quota = int(q) / int(per)
    except (OSError, ValueError):
        try:                                            # cgroup v1
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f1, open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f2:
                q, per = int(f1.read()), int(f2.read())
                if q > 0 and per > 0:
                    quota = q / per
        except (OSError, ValueError):
            pass
    if quota is not None:
        n = max(1, min(n, int(quota + 0.999)))
    return n


# --------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# --------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self._stop = threading.Event()
        self._t = None

    def _run_nvml(self) -> bool:
        """NVML polled every 20 ms (the timed region of a default run is ~0.2 s; nvidia-smi alone takes ~0.1 s per query)."""
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        except Exception:
            return False
        bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        while not self._stop.is_set():
            try:
                r = int(reasons(h))
                self.samples.append([str(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), str(mx), str(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)] +
                                    [("Active" if r & bits[n] else "Not Active") for n in ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")])
            except Exception:
                pass
            self._stop.wait(0.02)
        return True

    def _run(self):
        if self._run_nvml():
            return
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm = sorted(int(float(s[0])) for s in self.samples if s and s[0].replace(".", "").isdigit())
        mx = [int(float(s[1])) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for i, n in enumerate(names):
                if len(s) > 3 + i and s[3 + i].lower().startswith("active"):
                    reasons.add(n)
        pw = sorted(float(s[2]) for s in self.samples if len(s) > 2 and s[2].replace(".", "").isdigit())
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_median": pw[len(pw) // 2] if pw else None, "power_w_max": pw[-1] if pw else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------
# the FLUX.1-schnell block stack on the GPU (reference-layout random parameters)
# --------------------------------------------------------------------------------------------
def make_linear(torch, K, N, precision, dtype, device, g, act_unsigned=False):
    from nunchaku_b200.models.linear import SVDQW4A4Linear

    fp4 = precision == "nvfp4"
    m = SVDQW4A4Linear(K, N, rank=RANK, bias=True, precision=precision, torch_dtype=dtype, device=device, act_unsigned=act_unsigned)
    with torch.no_grad():
        # the packed layouts are permutations: random bytes in the reference layout ARE random weights
        m.qweight.copy_(torch.randint(-128, 128, m.qweight.shape, generator=g, device=device, dtype=torch.int8))
        if fp4:
            m.wscales.copy_(torch.randint(0x30, 0x38, m.wscales.shape, generator=g, device=device, dtype=torch.uint8).view(torch.float8_e4m3fn))  # 0.5 .. 0.94
            m.wtscale = 1.0 / (2.6 * 0.72 * K ** 0.5)
            m.wcscales.copy_((1.0 + 0.05 * torch.randn(N, generator=g, device=device)).to(dtype))
        else:
            m.wscales.copy_(((0.75 + 0.5 * torch.rand(m.wscales.shape, generator=g, device=device)) / (4.6 * K ** 0.5)).to(dtype))
        m.bias.copy_((0.1 * torch.randn(N, generator=g, device=device)).to(dtype))
        m.smooth_factor.copy_((0.75 + 0.5 * torch.rand(K, generator=g, device=device)).to(dtype))
        m.proj_down.copy_((torch.randn(K, RANK, generator=g, device=device) / K ** 0.5).to(dtype))
        m.proj_up.copy_((0.1 * torch.randn(N, RANK, generator=g, device=device) / RANK ** 0.5).to(dtype))
    m.invalidate()
    return m


class Block:
    def __init__(self, torch, tag, M, precision, dtype, device, g):
        fp4 = precision == "nvfp4"
        self.tag, self.M = tag, M
        self.qkv = make_linear(torch, DIM, 3 * DIM, precision, dtype, device, g)
        self.out = make_linear(torch, DIM, DIM, precision, dtype, device, g)
        self.fc1 = make_linear(torch, DIM, MLP, precision, dtype, device, g)
        # fc2 consumes the fused fc1 epilogue's UNSIGNED (shifted GELU) INT4 activations (attention.py:98-99)
        self.fc2 = make_linear(torch, MLP, DIM, precision, dtype, device, g, act_unsigned=not fp4)
        self.norm_q = (1.0 + 0.1 * torch.randn(128, generator=g, device=device)).to(dtype)
        self.norm_k = (1.0 + 0.1 * torch.randn(128, generator=g, device=device)).to(dtype)

    def linears(self):
        return [self.qkv, self.out, self.fc1, self.fc2]


class StackRunner:
    """One denoising step of the hot path through the package's public module / ops API."""

    def __init__(self, torch, precision, dtype, device):
        from nunchaku_b200.ops import fused, glue
        from nunchaku_b200.utils import pack_rotemb

        from nunchaku_b200._C import lib

        self.torch, self.glue, self.fused, self.lib = torch, glue, fused, lib
        self.precision, self.dtype, self.device = precision, dtype, device
        g = torch.Generator(device=device).manual_seed(1234)
        self.blocks = [Block(torch, tag, M, precision, dtype, device, g) for tag, M in block_list()]
        for b in self.blocks:   # convert once, then drop the checkpoint-layout copies of the big tensors (weights.py)
            for lin in b.linears():
                lin.release_reference_layout()
        # packed RoPE tables (reference pack_rotemb layout) per token count, real sin / cos of random angles
        self.rot = {}
        for M in (IMG_TOKENS, TXT_TOKENS, IMG_TOKENS + TXT_TOKENS):
            Mp = (M + 255) // 256 * 256
            ang = torch.rand(Mp, 64, generator=g, device=device) * 6.2831853
            self.rot[M] = pack_rotemb(torch.sin(ang), torch.cos(ang))
        self.h_img = torch.randn(IMG_TOKENS, DIM, generator=g, device=device).to(dtype)
        self.h_txt = torch.randn(TXT_TOKENS, DIM, generator=g, device=device).to(dtype)
        self.result = torch.empty(IMG_TOKENS + TXT_TOKENS, DIM, dtype=dtype, device=device)
        self.launches = 0

    def set_inputs(self, img, txt):
        self.h_img.copy_(img, non_blocking=True)
        self.h_txt.copy_(txt, non_blocking=True)

    def _stream_block(self, b: Block, h):
        """LayerNorm -> QKV(+RMSNorm+RoPE epilogue) -> [attention not run] -> out ; LayerNorm -> fc1 -> GELU -> fc2 ; add"""
        glue, M = self.glue, b.M
        n1 = glue.layernorm(h, None, None, 1e-6)
        qkv = b.qkv.forward_qkv(n1, b.norm_q, b.norm_k, self.rot[M])
        qkv_gemm_launches = self.lib.nb200_last_launch_count()   # 1 (fused RoPE epilogue) or 2 (plain GEMM + in-place RMSNorm/RoPE kernel)
        attn = qkv.view(-1)[: M * DIM].view(M, DIM)            # stand-in for the attention output: freshly written, L2-hot
        o = b.out.forward(attn.view(1, M, DIM)).view(M, DIM)
        n2 = n1 if b.tag.startswith("single") else glue.layernorm(o, None, None, 1e-6)
        fuse = self.fused._fuse_fc1(b.fc1, M)
        f = b.fc1.forward_mlp(n2, b.fc2, fuse=fuse)
        self.launches += 1 + (1 + qkv_gemm_launches) + 2 + (0 if n2 is n1 else 1) + 4 + 1   # (fused MLP: quantize, fc1 + its partial-sum reduction, fc2; split: quantize, fc1, quantize, fc2)
        return glue.add(o, f)

    overlap_streams = True   # joint blocks: the 256-token text stream's kernels go to a second CUDA stream (they fill SMs the image stream's
                             # kernels leave idle: quantizer grids of 128-136 CTAs, GEMM tails); without attention the two streams are independent

    def step(self):
        torch = self.torch
        h_img, h_txt = self.h_img, self.h_txt
        i = 0
        if self.overlap_streams:
            cur = torch.cuda.current_stream()
            if getattr(self, "_side", None) is None:
                self._side = torch.cuda.Stream()
            side = self._side
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                for b in range(N_JOINT):
                    h_txt = self._stream_block(self.blocks[2 * b + 1], h_txt)
            for b in range(N_JOINT):
                h_img = self._stream_block(self.blocks[2 * b], h_img)
            cur.wait_stream(side)
            h_txt.record_stream(cur)
            i = 2 * N_JOINT
        else:
            for _ in range(N_JOINT):
                h_img = self._stream_block(self.blocks[i], h_img)
                h_txt = self._stream_block(self.blocks[i + 1], h_txt)
                i += 2
        h = torch.cat([h_img, h_txt], dim=0)      # one copy per step (the model concatenates the streams here too)
        for _ in range(N_SINGLE):
            h = self._stream_block(self.blocks[i], h)
            i += 1
        self.result.copy_(h)
        return self.result


class FullRunner(StackRunner):
    """One denoising step of the WHOLE transformer (secondary figure "full_step"): what StackRunner runs plus everything SURVEY section 8(f)
    added this round -- AdaLN modulation through the AWQ W4A16 GEMV (row N2: silu(temb) -> GEMV -> split -> LayerNorm * (1 + scale) + shift),
    the QKV projection's PackQKV hand-off and attention_fp16 (row N1) over the joint [text; image] sequence, gates and residuals as the
    reference's blocks apply them (src/FluxModel.cpp:JointTransformerBlock / FluxSingleTransformerBlock)."""

    def __init__(self, torch, precision, dtype, device):
        super().__init__(torch, precision, dtype, device)
        from nunchaku_b200.ops.attention import attention_fp16
        from nunchaku_b200.ops.gemv import AWQW4A16Linear

        self.attention = attention_fp16
        g = torch.Generator(device=device).manual_seed(4321)
        T = IMG_TOKENS + TXT_TOKENS
        self.Tpad = (T + 255) // 256 * 256
        self.q = torch.zeros(1, HEADS, self.Tpad, 128, dtype=torch.float16, device=device)
        self.k = torch.full_like(self.q, float("nan"))       # pad keys are the mask (NaN), written once
        self.v = torch.zeros_like(self.q)
        self.attn_out = torch.empty(1, self.Tpad, DIM, dtype=dtype, device=device)
        self.temb = torch.randn(1, DIM, generator=g, device=device).to(dtype)

        def awq(n_out):
            m = AWQW4A16Linear(DIM, n_out, bias=True, torch_dtype=dtype, device=device)
            with torch.no_grad():
                m.qweight.copy_(torch.randint(-2 ** 31, 2 ** 31 - 1, m.qweight.shape, generator=g, device=device, dtype=torch.int64).to(torch.int32))
                m.wscales.copy_((0.01 + 0.01 * torch.rand(m.wscales.shape, generator=g, device=device)).to(dtype))
                m.wzeros.copy_((-0.08 * torch.rand(m.wzeros.shape, generator=g, device=device)).to(dtype))
                m.bias.copy_((0.1 * torch.randn(n_out, generator=g, device=device)).to(dtype))
            return m

        # one modulation linear per stream-block: 6 * dim for the joint blocks' two streams, 3 * dim for the single blocks
        self.mod = [awq((3 if b.tag.startswith("single") else 6) * DIM) for b in self.blocks]

    def _modulate(self, i, h):
        """AdaLayerNormZero(/Single): chunks of the modulation vector, LayerNorm(h) * (1 + scale_msa) + shift_msa"""
        glue = self.glue
        single = self.blocks[i].tag.startswith("single")
        emb = self.mod[i](self.temb, fuse_silu=True)                 # silu -> W4A16 GEMV -> + bias, one launch
        ch = glue.split_mod(emb.view(1, -1), 3 if single else 6)     # shift_msa, scale_msa, gate_msa[, shift_mlp, scale_mlp, gate_mlp]
        return glue.layernorm_mod(h, ch[1], ch[0], 1e-6), ch         # LayerNorm * (1 + scale) + shift, one pass

    def _qkv_attn(self, blocks_rows):
        """blocks_rows: [(block, normed input, first row in the joint sequence)] -> attention output rows [T, dim]"""
        for b, n, row0 in blocks_rows:
            views = tuple(t[:, :, row0:] for t in (self.q, self.k, self.v))
            b.qkv.forward_qkv(n, b.norm_q, b.norm_k, self.rot[b.M], out_qkv=views, attn_tokens=b.M)
        self.attention(self.q, self.k, self.v, self.attn_out, 128 ** -0.5)
        return self.attn_out[0]

    def step(self):
        torch, glue = self.torch, self.glue
        h_img, h_txt = self.h_img, self.h_txt
        i = 0
        for _ in range(N_JOINT):
            bi, bt = self.blocks[i], self.blocks[i + 1]
            n_img, c_img = self._modulate(i, h_img)
            n_txt, c_txt = self._modulate(i + 1, h_txt)
            attn = self._qkv_attn([(bt, n_txt, 0), (bi, n_img, TXT_TOKENS)])       # text tokens first, as the reference concatenates them
            outs = []
            for b, h, ch, rows in ((bi, h_img, c_img, slice(TXT_TOKENS, TXT_TOKENS + IMG_TOKENS)), (bt, h_txt, c_txt, slice(0, TXT_TOKENS))):
                M = b.M
                o = b.out.forward(attn[rows].reshape(1, M, DIM)).view(M, DIM)
                glue.mul_add_batch(o.view(1, -1, DIM), ch[2], True, 0.0, h.view(1, -1, DIM), True)        # h + gate_msa * attn_out
                n2 = glue.layernorm_mod(o, ch[4], ch[3], 1e-6)
                f = b.fc1.forward_mlp(n2, b.fc2, fuse=self.fused._fuse_fc1(b.fc1, M))
                glue.mul_add_batch(f.view(1, -1, DIM), ch[5], True, 0.0, o.view(1, -1, DIM), True)        # + gate_mlp * ff
                outs.append(f)
            h_img, h_txt = outs
            i += 2
        h = torch.cat([h_txt, h_img], dim=0)
        for _ in range(N_SINGLE):
            b = self.blocks[i]
            M = b.M
            n, ch = self._modulate(i, h)
            attn = self._qkv_attn([(b, n, 0)])
            o = b.out.forward(attn[:M].reshape(1, M, DIM)).view(M, DIM)
            f = b.fc1.forward_mlp(n, b.fc2, fuse=self.fused._fuse_fc1(b.fc1, M))
            s = glue.add(o, f)
            glue.mul_add_batch(s.view(1, -1, DIM), ch[2], True, 0.0, h.view(1, -1, DIM), True)             # h + gate * (attn_out + ff)
            h = s
            i += 1
        self.result.copy_(h)
        return self.result


class GemmRecorder:
    """Records every fused-GEMM call of one eager step (arguments kept alive) so that the GEMMs alone can be replayed from
    a CUDA graph: the roofline of the dominant kernel is measured under the same replay conditions as the step."""

    def __init__(self):
        self.calls = []

    def __enter__(self):
        import nunchaku_b200.models.linear as L

        self.L, self.orig = L, L.gemm_b200

        def rec(*a, **k):
            self.calls.append((a, k))
            return self.orig(*a, **k)

        L.gemm_b200 = rec
        return self

    def __exit__(self, *exc):
        self.L.gemm_b200 = self.orig

    def flops(self):
        total = 0
        for a, k in self.calls:
            w = a[3]
            rows = a[0].shape[0]
            out = k.get("out")
            M = out.shape[0] if out is not None else rows
            total += 2 * M * w.K * w.N + 2 * M * w.rank * w.N
            if k.get("next_w") is not None:
                total += 2 * M * k["next_w"].rank * w.N
        return total

    def replay(self):
        for a, k in self.calls:
            self.orig(*a, **k)


def capture(torch, fn):
    """the package's own capture helper (nunchaku_b200/graph.py, SURVEY row N3)"""
    from nunchaku_b200.graph import GraphedStep

    step = GraphedStep(fn, (), warmup=1)
    step.replay()
    torch.cuda.synchronize()
    return step


def time_replays(torch, graph, n, barrier):
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        graph.replay()
    e1.record()
    barrier()
    return e0.elapsed_time(e1)


# --------------------------------------------------------------------------------------------
# comparison legs on the same GPU
# --------------------------------------------------------------------------------------------
def cublas_bf16_leg(torch, device, steps):
    """The 16-bit ceiling (BASELINE.md section 2): the same 304 GEMM shapes as plain bf16 cuBLAS matmuls on de-quantised weights
    (random bf16 of the same shapes; no low-rank branch, no epilogue), CUDA-graph replay."""
    shapes = {}
    for _, M, K, N in layer_list():
        shapes[(M, K, N)] = shapes.get((M, K, N), 0) + 1
    g = torch.Generator(device=device).manual_seed(7)
    ops = []
    for (M, K, N), cnt in shapes.items():
        x = torch.randn(M, K, generator=g, device=device).to(torch.bfloat16)
        ws = [torch.randn(N, K, generator=g, device=device).to(torch.bfloat16) for _ in range(min(cnt, 8))]   # > L2 in total
        y = torch.empty(M, N, dtype=torch.bfloat16, device=device)
        ops.append((x, ws, y, cnt))

    def run():
        for x, ws, y, cnt in ops:
            for i in range(cnt):
                torch.matmul(x, ws[i % len(ws)].t(), out=y)

    graph = capture(torch, run)
    ms = time_replays(torch, graph, steps, torch.cuda.synchronize) / steps
    f_main, _ = step_flops()
    return {"ms_per_step": ms, "tflops": f_main / (ms * 1e-3) / 1e12, "what": "304 torch.matmul (cuBLAS) bf16 GEMMs of the same shapes, graph replay"}


def reference_gpu_leg(torch, device):
    """The REFERENCE's own INT4 kernels (oracle/_ref/libnunchaku_ref.so = its unmodified sources built for sm_100a,
    oracle/ref_build/build_ref.sh) timed on this GPU per distinct layer shape (quantize + GEMM through its C++ class
    GEMM_W4A4, and the fused fc1->fc2 MLP), CUDA events, summed with the step's multiplicities.  NVFP4 cannot run: the
    reference's NVFP4 kernels need sm_120a (SURVEY F3)."""
    try:
        from oracle import refgpu as R   # test / comparison infrastructure: never on the product path
    except Exception as e:
        return {"unavailable": f"oracle.refgpu import failed: {e!r}"}
    if not R.available("ref"):
        return {"unavailable": "oracle/_ref/libnunchaku_ref.so not built (oracle/ref_build/build_ref.sh needs /root/reference)"}
    dtype = torch.bfloat16
    g = torch.Generator(device=device).manual_seed(3)

    def ref_lin(K, N):
        m = R.RefLinear(K, N, bias=True, fp4=False, dtype=dtype)
        m.load(qweight=torch.randint(-128, 128, (N, K // 2), generator=g, device=device, dtype=torch.int8),
               wscales=((0.75 + 0.5 * torch.rand(K // 64, N, generator=g, device=device)) / (4.6 * K ** 0.5)).to(dtype),
               bias=(0.1 * torch.randn(N, generator=g, device=device)).to(dtype),
               smooth=(0.75 + 0.5 * torch.rand(K, generator=g, device=device)).to(dtype),
               lora_down=(torch.randn(K, RANK, generator=g, device=device) / K ** 0.5).to(dtype),
               lora_up=(0.1 * torch.randn(N, RANK, generator=g, device=device) / RANK ** 0.5).to(dtype))
        return m

    def t_ms(fn, iters=3):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    per = {}
    total = 0.0
    counts = {}
    for _, M in block_list():
        counts[M] = counts.get(M, 0) + 1
    qkv, out, fc1, fc2 = ref_lin(DIM, 3 * DIM), ref_lin(DIM, DIM), ref_lin(DIM, MLP), ref_lin(MLP, DIM)
    for M, cnt in counts.items():
        x = torch.randn(M, DIM, generator=g, device=device).to(dtype)
        nq = torch.ones(128, dtype=dtype, device=device)
        rot = torch.zeros(1, (M + 255) // 256 * 256, 128, dtype=torch.float32, device=device)
        t = {"qkv_rope": t_ms(lambda: qkv.forward_qkv(x, nq, nq, rot)), "out": t_ms(lambda: out.forward(x)),
             "mlp_fused": t_ms(lambda: fc1.forward_mlp(fc2, x))}
        per[str(M)] = {k: round(v, 3) for k, v in t.items()}
        total += cnt * sum(t.values())
    f_main, f_lr = step_flops()
    return {"ms_per_step": total, "value": (1.0 / STEPS_PER_IMAGE) / (total * 1e-3), "unit": "images/s", "precision": "int4",
            "tflops": (f_main + f_lr) / (total * 1e-3) / 1e12, "per_shape_ms": per,
            "what": "reference kernels (unmodified sources, sm_100a build) through its C++ GEMM_W4A4 class: quantize + GEMM per layer, fused fc1->fc2; "
                    "CUDA events per distinct shape x multiplicity in the step; LayerNorm / add glue not included"}


class CpuSample:
    """Bounded CPU sample of the workload: one 3072x3072 r=32 SVDQuant linear on M=256 rows (the text-stream shape, BASELINE
    config 1) through the oracle's reference-emulating path -- the plain-C restatement oracle/svdq_ref.c (pinned bit-exact
    against the reference's GPU kernels via tests/test_ref_gpu_golden.py) on the host threads this process may use."""

    def __init__(self, torch, precision: str):
        from oracle import svdq as O

        self.O = O
        fp4 = precision == "nvfp4"
        self.layer = O.make_synthetic_layer(DIM, DIM, RANK, fp4=fp4, hT=torch.bfloat16, seed=0)
        self.x = O.make_activations(TXT_TOKENS, DIM, torch.bfloat16, seed=1, smooth=self.layer.smooth)
        self.flops = 2 * TXT_TOKENS * DIM * DIM + 2 * TXT_TOKENS * RANK * (DIM + DIM)
        self.cores = host_threads()
        try:
            from oracle import csvdq

            csvdq.build()
            self.fn = lambda: csvdq.linear_forward(self.layer, self.x)
            self.impl = "plain-C oracle (oracle/svdq_ref.c, OpenMP)"
            # "all the host threads it can use" = the team size that is actually fastest on this box: every hyper-thread of a 2-socket host is
            # not (3072 weight rows over 128 threads: 24 rows each, memory-bound decode on two NUMA nodes).  One warm + one timed rep per size.
            tried = {}
            n = self.cores
            while n >= 1:
                csvdq.set_threads(n)
                self.fn()
                t0 = time.perf_counter()
                self.fn()
                tried[n] = time.perf_counter() - t0
                if n <= 8:
                    break
                n //= 2
            self.cores = min(tried, key=tried.get)
            self.tried = tried
            csvdq.set_threads(self.cores)
        except Exception as e:  # no gcc on the box: the torch restatement
            torch.set_num_threads(min(self.cores, 32))
            self.cores = torch.get_num_threads()
            self.fn = lambda: O.svdq_linear_forward(self.layer, self.x, mode="ref")
            self.impl = f"Python oracle (C oracle unavailable: {type(e).__name__})"
        self.fn()  # warm (page in, OpenMP team start)

    def run(self, budget_s: float):
        t0 = time.perf_counter()
        reps = 0
        while reps == 0 or time.perf_counter() - t0 < budget_s:
            self.fn()
            reps += 1
        return (time.perf_counter() - t0) / reps, reps

    def describe(self, precision: str, dt: float, reps: int) -> str:
        tried = getattr(self, "tried", None)
        how = ("fastest team size of " + ", ".join(f"{n}: {t * 1e3:.0f} ms" for n, t in tried.items())) if tried else "sched_getaffinity / cgroup quota"
        return (f"1 SVDQuant linear 3072x3072 r32 M=256 ({precision}), reference-emulating arithmetic, {self.impl}, {self.cores} threads "
                f"({how}): {reps} reps x {dt * 1e3:.1f} ms")


def run_reference_arm(args):
    import torch

    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    f_main, f_lr = step_flops()
    flops_per_image = (f_main + f_lr) * STEPS_PER_IMAGE
    cs = CpuSample(torch, args.precision)
    times, reps_total = [], 0
    for i in range(args.warmup + args.steps):   # a "step" of this arm is a bounded ~4 s sample of the CPU path
        dt_i, reps = cs.run(4.0)
        if i >= args.warmup:
            times.append(dt_i)
            reps_total += reps
    dt = sum(times) / len(times)
    value = (cs.flops / dt) / flops_per_image
    sample = cs.describe(args.precision, dt, reps_total)
    _emit({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int4" if args.precision == "int4" else "nvfp4", "data": "synthetic", "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": cs.cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the reference has no CPU implementation of this path (SURVEY F6); this is the CPU oracle (port, pinned to the reference's GPU kernels) "
                "on the host threads; value extrapolates the sample's FLOP rate to one image's hot-path FLOPs",
    })
    return 0


def workload_config(args):
    return {"workload": "FLUX.1-schnell 1024x1024 4-step bs=1: per step 304 SVDQuant linears (19 joint x (img 4096 + txt 256 tokens) + 38 single x 4352 "
                        "tokens; dim 3072, mlp 12288, rank 32, 24 heads) chained through LayerNorm / RMSNorm+RoPE epilogue / GELU-quantise / add; attention not run",
            "precision": args.precision, "parallelism": f"replica x{args.gpus}",
            "l2": "inputs larger than L2 (4.3 GB of 4-bit weights streamed per step)",
            "streams": "one" if getattr(args, "no_overlap", False) else "joint blocks: text-stream kernels on a second CUDA stream (both captured in the one graph)"}


_REAL_STDOUT = None


def _quiet_stdout() -> None:
    """stdout must carry exactly ONE JSON line, but native libraries write there too (NCCL banner): point fd 1 at stderr for
    the run and keep the real stdout for the final line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def _emit(line: dict) -> None:
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


def dump_outputs(path: str, arrays: dict) -> None:
    """--dump-outputs: every array as DIR/<name>.npy, float32"""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.float().cpu().numpy())


def load_peaks():
    """roofline denominators: tensor-pipe peaks measured on a B200 by tools/ubench/mma_peak.cu (committed: profiles/r02_mma_peaks.json)
    and the driver's MEASURED_PEAKS.json (HBM, cuBLAS bf16)."""
    peaks = {}
    for name in ("MEASURED_PEAKS.json", os.path.join("profiles", "r02_mma_peaks.json")):
        try:
            peaks.update(json.load(open(os.path.join(ROOT, name))))
        except Exception:
            pass
    return peaks


def main() -> int:
    _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    # NVFP4 is what the reference itself selects on Blackwell (nunchaku/utils.py:190-231 -> "fp4" for sm_12x; its INT4 mma.sync.s4 is
    # emulated on sm_100, SURVEY F4) and the only 4-bit format tcgen05 runs natively; INT4 is measured in the same run ("secondary").
    ap.add_argument("--precision", default=os.environ.get("NB200_BENCH_PRECISION", "nvfp4"), choices=["int4", "nvfp4"])
    ap.add_argument("--no-secondary", action="store_true", help="skip the other precision's device-resident measurement")
    ap.add_argument("--no-legs", action="store_true", help="skip the cuBLAS-bf16 and reference-GPU comparison legs")
    ap.add_argument("--no-overlap", action="store_true", help="joint blocks: run the text stream's kernels on the main CUDA stream instead of a second one")
    ap.add_argument("--no-full", action="store_true", help="skip the whole-transformer-step figure (attention + AdaLN modulation on top of the linear stack)")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of a captured CUDA graph")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's hidden states to DIR/hidden_states.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    from nunchaku_b200 import replica

    rank, world, local = replica.world()
    assert torch.cuda.is_available(), "bench.py needs a GPU (use --impl reference for the CPU arm)"
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    replica.init("nccl", device)
    from nunchaku_b200._C import check, lib

    check(lib.nb200_check_device(), "check_device")
    dtype = torch.bfloat16
    StackRunner.overlap_streams = not args.no_overlap
    runner = StackRunner(torch, args.precision, dtype, device)

    def barrier():
        torch.cuda.synchronize()
        replica.barrier()
        torch.cuda.synchronize()

    # ---- warm-up ----------------------------------------------------------------------------------
    for _ in range(args.warmup):
        runner.launches = 0
        runner.step()
    launches_per_step = runner.launches   # our kernels only (quantize, GEMM, LayerNorm, add); memsets / the one cat+copy per step are not counted
    torch.cuda.synchronize()

    # ---- device-resident throughput: captured CUDA graph of one step ---------------------------------
    graph = None
    if not args.no_graph:
        try:
            graph = capture(torch, runner.step)
        except Exception as e:  # pragma: no cover
            print(f"[bench] CUDA graph capture failed ({e}); timing eager launches", file=sys.stderr)
            graph = None

    class Eager:
        def replay(self):
            runner.step()

    stepper = graph if graph is not None else Eager()
    with ClockSampler(local) as clocks:
        ms = time_replays(torch, stepper, args.steps, barrier)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"hidden_states": runner.result})
    ms_per_step = replica.max_over_ranks(ms, device) / args.steps
    images_per_s = world * (1.0 / STEPS_PER_IMAGE) / (ms_per_step * 1e-3)
    f_main, f_lr = step_flops()
    clk = clocks.summary()

    # ---- e2e through the public API with HOST buffers ---------------------------------------------------
    img_h = torch.randn(IMG_TOKENS, DIM).to(dtype).pin_memory()
    txt_h = torch.randn(TXT_TOKENS, DIM).to(dtype).pin_memory()
    out_h = torch.empty(IMG_TOKENS + TXT_TOKENS, DIM, dtype=dtype).pin_memory()
    h2d = img_h.numel() * 2 + txt_h.numel() * 2
    d2h = out_h.numel() * 2
    # Every step copies its inputs host -> device and its result device -> host on a second stream through double-buffered
    # staging tensors, so step i+1's upload and step i's download overlap the kernels (what a serving loop does).
    copy_s = torch.cuda.Stream()
    st_img = [torch.empty(IMG_TOKENS, DIM, dtype=dtype, device=device) for _ in range(2)]
    st_txt = [torch.empty(TXT_TOKENS, DIM, dtype=dtype, device=device) for _ in range(2)]
    st_out = [torch.empty(IMG_TOKENS + TXT_TOKENS, DIM, dtype=dtype, device=device) for _ in range(2)]
    up_done, up_free = [torch.cuda.Event() for _ in range(2)], [torch.cuda.Event() for _ in range(2)]
    dn_ready, dn_done = [torch.cuda.Event() for _ in range(2)], [torch.cuda.Event() for _ in range(2)]

    def upload(b):
        with torch.cuda.stream(copy_s):
            copy_s.wait_event(up_free[b])
            st_img[b].copy_(img_h, non_blocking=True)
            st_txt[b].copy_(txt_h, non_blocking=True)
            up_done[b].record(copy_s)

    def e2e_loop(n):
        cur = torch.cuda.current_stream()
        for b in range(2):
            up_free[b].record(cur)
            dn_done[b].record(cur)
        upload(0)
        for i in range(n):
            b = i & 1
            cur.wait_event(up_done[b])
            runner.set_inputs(st_img[b], st_txt[b])      # device -> device, microseconds
            up_free[b].record(cur)
            if i + 1 < n:
                upload(b ^ 1)
            stepper.replay()
            cur.wait_event(dn_done[b])                    # st_out[b] was downloaded two steps ago
            st_out[b].copy_(runner.result, non_blocking=True)
            dn_ready[b].record(cur)
            with torch.cuda.stream(copy_s):
                copy_s.wait_event(dn_ready[b])
                out_h.copy_(st_out[b], non_blocking=True)
                dn_done[b].record(copy_s)
        torch.cuda.synchronize()

    e2e_loop(2)
    barrier()
    t0 = time.perf_counter()
    e2e_loop(args.steps)
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_images = world * (1.0 / STEPS_PER_IMAGE) / (replica.max_over_ranks(e2e_s, device) / args.steps)

    # ---- roofline of the dominant kernel (fused GEMM): the step's 304 GEMM launches alone, graph replay, CUDA events ------------
    with GemmRecorder() as rec:
        runner.step()
    torch.cuda.synchronize()
    g_graph = capture(torch, rec.replay)
    g_ms = time_replays(torch, g_graph, args.steps, torch.cuda.synchronize) / args.steps
    g_fl = rec.flops()
    n_gemm = len(rec.calls)
    peaks = load_peaks()
    fp4 = args.precision == "nvfp4"
    key = "nvf4_cg2" if fp4 else "bf16_cg1"
    if key in peaks:
        # burst figure when the run's median clock sat near the maximum, sustained (power-limited clocks) otherwise
        near_max = clk["sm_mhz"] is not None and clk["sm_max_mhz"] and clk["sm_mhz"] >= 0.9 * clk["sm_max_mhz"]
        which = "tflops_burst" if near_max else "tflops_sustained"
        peak = float(peaks[key][which])
        peak_basis = f"{key}.{which} measured by tools/ubench/mma_peak.cu on a B200 (profiles/r02_mma_peaks.json); run median SM clock {clk['sm_mhz']} MHz"
    else:
        peak = float(peaks.get("bf16_tflops", 1746.5)) * (4.0 if fp4 else 1.0)
        peak_basis = "fallback: MEASURED_PEAKS.json bf16_tflops" + (" x4" if fp4 else "")
    achieved = g_fl / (g_ms * 1e-3) / 1e12
    # dram bytes of ONE launch on the primary shape (M=4096, K=N=3072, r=32) from the committed `ncu --set full` captures (profiles/)
    traffic = {"int4": 12.5e6, "nvfp4": 13.2e6}[args.precision]
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_basis": "dram bytes per launch, primary shape 4096x3072x3072, ncu --set full (profiles/r02e_gemm_nvfp4_ncu.txt, profiles/r01x_gemm_int4_ncu.txt; algorithmic: 37.6 MB incl. the 25 MB output that stays in L2)",
                "kernel": "gemm_nvfp4_cluster_kernel" if fp4 else "gemm_w4a4_kernel", "launches": n_gemm, "avg_launch_us": g_ms * 1e3 / n_gemm,
                "timing": "the step's 304 fused-GEMM operator calls alone (the 57 large-M QKV calls include their in-place RMSNorm+RoPE kernel), CUDA-graph replay, CUDA events on the launch stream", "peak_basis": peak_basis,
                "gemm_share_of_step": g_ms / ms_per_step}
    del g_graph, rec

    # ---- comparison legs on the same GPU (rank 0, N=1) --------------------------------------------------------
    legs = {}
    if not args.no_legs and world == 1:
        try:
            legs["cublas_bf16"] = cublas_bf16_leg(torch, device, args.steps)
        except Exception as e:  # pragma: no cover
            legs["cublas_bf16"] = {"unavailable": repr(e)}
        try:
            legs["reference_gpu"] = reference_gpu_leg(torch, device)
        except Exception as e:
            legs["reference_gpu"] = {"unavailable": repr(e)}

    # ---- the other 4-bit format, device-resident graph replay only ---------------------------------------------
    secondary = None
    timing_mode = "cuda graph replay" if graph is not None else "eager launches"
    if not args.no_secondary:
        other = "int4" if fp4 else "nvfp4"
        del graph, stepper
        runner2 = StackRunner(torch, other, dtype, device)
        for _ in range(args.warmup):
            runner2.step()
        torch.cuda.synchronize()
        g2 = capture(torch, runner2.step)
        ms2 = replica.max_over_ranks(time_replays(torch, g2, args.steps, barrier), device) / args.steps
        secondary = {"precision": other, "ms_per_step": ms2, "value": world * (1.0 / STEPS_PER_IMAGE) / (ms2 * 1e-3), "unit": "images/s",
                     "tflops": world * (f_main + f_lr) / (ms2 * 1e-3) / 1e12, "timing": "cuda graph replay"}
        ref = legs.get("reference_gpu", {})
        if other == "int4" and "ms_per_step" in ref:
            secondary["speedup_vs_reference_gpu_kernels"] = ref["ms_per_step"] / ms2

    # ---- the whole transformer step: + AdaLN modulation (AWQ GEMV), PackQKV, attention_fp16, gates (SURVEY section 8f rows N1 / N2) -----------
    full_step = None
    if not args.no_full:
        try:
            runner3 = FullRunner(torch, args.precision, dtype, device)
            for _ in range(args.warmup):
                runner3.step()
            torch.cuda.synchronize()
            g3 = capture(torch, runner3.step)
            ms3 = replica.max_over_ranks(time_replays(torch, g3, args.steps, barrier), device) / args.steps
            attn_flops = 4.0 * HEADS * (IMG_TOKENS + TXT_TOKENS) ** 2 * 128 * (N_JOINT + N_SINGLE)
            full_step = {"ms_per_step": ms3, "value": world * (1.0 / STEPS_PER_IMAGE) / (ms3 * 1e-3), "unit": "images/s", "precision": args.precision,
                         "tflops": world * (f_main + f_lr + attn_flops) / (ms3 * 1e-3) / 1e12, "timing": "cuda graph replay",
                         "what": "the step above plus what the linear stack leaves out: AdaLN modulation through the AWQ W4A16 GEMV (57 + 19 launches, 1.6 GB of 4-bit "
                                 "weights), PackQKV hand-off, attention_fp16 on tcgen05 over the 4352-token joint sequence (57 launches, 13.3 TFLOP), gates and residuals; "
                                 "text encoders / VAE / scheduler are outside the transformer and not run"}
            del g3, runner3
        except Exception as e:  # the headline numbers above must still be reported
            print(f"[bench] full-step leg failed: {e!r}", file=sys.stderr)
            full_step = {"unavailable": repr(e)}

    if rank == 0:
        cpu = None
        if not args.skip_cpu and world == 1:   # the CPU baseline is an N=1 figure (rank 0's host cores)
            try:
                cs = CpuSample(torch, args.precision)
                dt, reps = cs.run(10.0)
                cpu_v = (cs.flops / dt) / ((f_main + f_lr) * STEPS_PER_IMAGE)
                cpu = {"value": cpu_v, "unit": "images/s", "cores": cs.cores, "kind": "port", "sample": cs.describe(args.precision, dt, reps)}
            except Exception as e:  # the GPU numbers above must still be reported
                print(f"[bench] CPU baseline leg failed: {e!r}", file=sys.stderr)
                cpu = {"value": None, "unit": "images/s", "cores": host_threads(), "kind": "port", "sample": f"failed: {e!r}"}
        _emit({
            "metric": METRIC, "value": images_per_s, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int4" if args.precision == "int4" else "nvfp4", "data": "synthetic", "config": workload_config(args),
            "tflops": world * (f_main + f_lr) / (ms_per_step * 1e-3) / 1e12, "timing": timing_mode, "clocks": clk,
            "e2e": {"value": e2e_images, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "path": ("CUDA graph of the per-layer module calls" if timing_mode.startswith("cuda graph") else "module calls launched from Python per layer")
                            + " (SVDQW4A4Linear.forward / forward_qkv / forward_mlp, glue.layernorm / add); pinned host in/out every step, copies on a second stream"},
            "gpu_launches": args.steps * launches_per_step, "roofline": roofline, "cpu_baseline": cpu, "secondary": secondary, "full_step": full_step, **legs,
        })
    replica.shutdown()
    return 0


if __name__ == "__main__":
    sys.exit(main())
