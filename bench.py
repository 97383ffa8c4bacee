#!/usr/bin/env python
"""bench.py — decode tok/s of the quantized-MoE hot path at DeepSeek-V3 shapes.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload): DeepSeek-V3 671B Q4_K_M single-stream decode, the MoE-block hot path of every
token: 58 MoE layers x [router (fp32 GEMV + grouped top-8) -> 8 routed experts (gate/up Q4_K, down Q6_K,
H=7168, I=2048, 256 experts resident per layer) -> 1 shared expert].  671B does not fit one B200, so a step
walks 58 layers over `--resident-layers` distinct full-size weight sets (each 7.4 GB >> L2, revisit distance
>= 2 sets >> L2: every byte comes from HBM); attention / dense layers / lm_head are NOT in the step and the
metric says so.  Weights are synthetic well-formed GGUF blocks, activations random (data: synthetic).

One step = one token per GPU through the 58 layers.  N > 1: experts are sharded E/N per GPU
(expert-parallel); per layer the N tokens are all-gathered, each GPU runs the (token, expert) pairs it owns
and a reduce-scatter returns every token's combined output — value = N tokens / step time (weak scaling).

Printed JSON line: see the task contract; `roofline` is for the dominant kernel (gate/up GEMV) from a live
CUDA-event pass, `cpu_baseline` / `--impl reference` time the reference's own CPU implementation
(oracle/_ref, the unmodified llamafile MoE) on this box's host cores.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

E, K, H, I, N_MOE_LAYERS = 256, 8, 7168, 2048, 58
N_GROUP, TOPK_GROUP, ROUTED_SCALE = 8, 4, 2.5
Q4_K, Q6_K, BF16, F32 = 12, 14, 30, 0
BYTES_GATE_UP_PER_EXPERT = 2 * I * H * 144 // 256           # 16,515,072
BYTES_DOWN_PER_EXPERT = H * I * 210 // 256                  # 12,042,240
BYTES_PER_EXPERT = BYTES_GATE_UP_PER_EXPERT + BYTES_DOWN_PER_EXPERT   # 28,557,312 (SURVEY §8d)
PREFILL_TOKENS = 1024   # the reference's group_max_len (experts.py:209): one chunk of MOE::forward_many


def committed_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed ncu summary
    (profiles/traffic.json, written by profiles/summarize.py from an `ncu --set full` capture); None when absent."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        return d.get(kernel, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def rows(self) -> int:
        try:
            return sum(1 for l in open(self.f.name) if l.strip())
        except Exception:
            return 0

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm = [float(r[1]) for r in rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        if sm:
            out["sm_mhz"] = statistics.median(sm)
            out["sm_max_mhz"] = float(rows[0][2])
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for i, n in enumerate(names):
                if any(len(r) >= 9 and r[5 + i].strip().lower() == "active" for r in rows):
                    out["reasons"].append(n)
            out["samples"] = len(sm)
        return out


# ----------------------------------------------------------------------------------------------- reference arm
def host_threads() -> int:
    """logical CPUs this process may use: affinity mask capped by the cgroup CPU quota."""
    try:
        n = max(1, len(os.sched_getaffinity(0)))
    except Exception:
        n = max(1, os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


class RefCpuMoe:
    """The reference's own CPU MoE (oracle/_ref: unmodified moe.cpp + llamafile + ggml) on synthetic weights of
    the real per-expert shapes.  `n_experts` experts are resident in host RAM (bounded sample of the 256)."""

    def __init__(self, n_experts=32, threads=None, tokens=1):
        import numpy as np
        import torch

        from ktransformers_b200.util.synth import synth_blocks
        from oracle.bindings import Oracle, Ref
        self.np = np
        self.kind = "reference" if Ref.available() else "port"
        self.threads = threads or host_threads()
        self.n = n_experts
        self.gate = synth_blocks(Q4_K, n_experts * I * H, "cpu", 101).numpy()
        self.up = synth_blocks(Q4_K, n_experts * I * H, "cpu", 102).numpy()
        self.down = synth_blocks(Q6_K, n_experts * H * I, "cpu", 103).numpy()
        if self.kind == "reference":
            self.ref = Ref.get(self.threads)
            self.threads = self.ref.threads
            self.isa = self.ref.isa()
            self.h = self.ref.moe_create(n_experts, K, H, I, self.gate, self.up, self.down, Q4_K, Q4_K, Q6_K, BF16)
        else:
            self.port = Oracle()
            self.isa = "plain C (oracle/ktoracle.c, OpenMP)"
        rng = np.random.default_rng(0)
        self.tokens = tokens          # tokens per layer-forward (the --gpus N arm decodes N tokens per step)
        self.x = (rng.standard_normal((tokens, H)) / 100).astype(np.float32)
        from oracle.bindings import f32_to_bf16_bits
        self.xb = f32_to_bf16_bits(self.x)
        self.ids = [np.stack([rng.permutation(n_experts)[:K] for _ in range(tokens)]).astype(np.uint64) for _ in range(N_MOE_LAYERS)]
        self.w = rng.random((tokens, K)).astype(np.float32)
        self.out = np.zeros((tokens, H), np.uint16)
        self.tuned = None
        if self.kind == "reference" and threads is None:
            self.tune_threads()

    def tune_threads(self):
        """The reference sizes CPUInfer to the physical core count (bench_moe.py:30-32); its work-stealing pool spins,
        so oversubscribing SMT siblings or a cgroup quota is catastrophic.  Give it its best shot: try a ladder of
        thread counts and keep the fastest."""
        cap = host_threads()
        ladder = sorted({n for n in (4, 8, 16, 24, 32, 48, 64, 96, 128, cap // 2, cap) if 1 <= n <= cap})
        best = None
        self.tuned = {}
        for n in ladder:
            self.threads = self.ref.init(n)
            for l in range(2):
                self.layer(l)
            t0 = time.perf_counter()
            for l in range(5):
                self.layer(l)
            dt = (time.perf_counter() - t0) / 5
            self.tuned[n] = round(dt * 1e3, 3)
            if best is None or dt < best[1]:
                best = (n, dt)
            if dt > 4 * best[1]:
                break
        self.threads = self.ref.init(best[0])

    def layer(self, l):
        if self.kind == "reference":
            self.ref.moe_forward_handle(self.h, H, BF16, self.ids[l % N_MOE_LAYERS], self.w, self.xb, self.out)
        else:
            self.port.moe_forward(self.n, H, I, self.gate, self.up, self.down, Q4_K, Q4_K, Q6_K, BF16,
                                  self.ids[l % N_MOE_LAYERS].astype(self.np.int64), self.w, self.xb)

    def token(self):
        for l in range(N_MOE_LAYERS):
            self.layer(l)

    def describe(self, layers_timed):
        tuned = f" (thread ladder ms/layer: {self.tuned})" if self.tuned else ""
        return (f"{self.kind} CPU MoE ({self.isa}), {self.threads} host threads{tuned}: routed experts only (the reference keeps "
                f"router/shared experts on the GPU), {layers_timed} layer-forwards of {self.tokens} token(s) x 8-of-{self.n} resident experts "
                f"at real shapes; tok/s = tokens/(58 x mean layer time)")


def amx_baseline(seconds=6.0):
    """The reference's AMX INT4 MoE (kt_kernel_ext.moe.AMXInt4_MOE, the "CPU-AMX" path of north_star) through the shimmed
    build oracle/_ref/libktamx.so — only on hosts with AMX; otherwise says why not.  Build-host numbers: profiles/."""
    try:
        import numpy as np

        from oracle.bindings import AmxRef, f32_to_bf16_bits
        if not AmxRef.available():
            return {"unavailable": AmxRef.why_unavailable(), "build_host_measurement": "profiles/r02_amx_baseline_buildhost.json"}
        En = 16
        rng = np.random.default_rng(0)
        mk = lambda shape: f32_to_bf16_bits(rng.standard_normal(shape, dtype=np.float32))  # noqa: E731
        g, u, d = mk((En, I, H)), mk((En, I, H)), mk((En, H, I))
        x = f32_to_bf16_bits((rng.standard_normal((1, H)) / 100).astype(np.float32))
        w = rng.random((1, K)).astype(np.float32)
        out = np.zeros((1, H), np.uint16)
        best = None
        cap = host_threads()
        for th in sorted({n for n in (4, 8, 16, 32, 64, cap) if n <= cap}):
            amx = AmxRef.get(th)
            h = amx.moe_create(En, K, H, I, g, u, d)
            ids = [np.stack([rng.permutation(En)[:K]]).astype(np.int64) for _ in range(16)]
            for i in range(3):
                amx.moe_forward(h, ids[i], w, x, out)
            t0 = time.perf_counter(); n = 0
            while time.perf_counter() - t0 < seconds / 4:
                amx.moe_forward(h, ids[n % 16], w, x, out); n += 1
            dt = (time.perf_counter() - t0) / n
            amx.moe_destroy(h)
            if best is None or dt < best[1]:
                best = (th, dt)
        return {"value": 1.0 / (N_MOE_LAYERS * best[1]), "unit": "tok/s", "cores": best[0], "kind": "reference (shimmed numa/hwloc build)",
                "ms_per_layer": best[1] * 1e3, "sample": f"AMXInt4_MOE, 1 token x 8-of-{En} experts at real shapes"}
    except Exception as e:  # pragma: no cover
        return {"unavailable": f"{type(e).__name__}: {e}"}


def run_reference_arm(args, rank):
    if rank != 0:
        return
    world = max(1, args.gpus)
    cpu = RefCpuMoe(tokens=world)            # same config as the B200 arm: `world` tokens per step
    for _ in range(args.warmup):
        cpu.token()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu.token()
    dt = (time.perf_counter() - t0) / args.steps
    v = world / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "tok/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int8xint4->int32, fp32 scales (llamafile Q8_K x Q4_K/Q6_K)", "data": "synthetic", "config": workload_config(args, world),
            "cpu_baseline": {"value": v, "unit": "tok/s", "cores": cpu.threads, "kind": cpu.kind, "sample": cpu.describe(args.steps * N_MOE_LAYERS)},
            "e2e": {"value": v, "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


METRIC = "decode tok/s DeepSeek-V3 671B INT4 (Q4_K_M) MoE-block hot path; HBM GB/s vs roofline"


def workload_config(args, world):
    return {"workload": ("DeepSeek-V3 671B Q4_K_M decode bs=1 per GPU, MoE-block hot path: 58 layers x [router fp32 256x7168 + 8 routed "
                         "experts (gate/up Q4_K, down Q6_K, H=7168 I=2048, E=256 resident/layer) + 1 shared expert]; attention, dense "
                         "layers and lm_head NOT included"),
            "resident_layer_sets": args.resident_layers, "layers_per_step": N_MOE_LAYERS, "tokens_per_step": world,
            "parallelism": f"ep{world}" if world > 1 else "single",
            "block_launch": ("plain grid + programmatic dependent launch" if os.environ.get("KTB200_BLK_COOP", "1") == "0"
                             else "cooperative + programmatic dependent launch"),
            "l2": "inputs larger than L2: each layer set is 7.4 GB and is revisited after >= 2 other sets",
            "next_layer_prefetch": os.environ.get("KTB200_BENCH_PREFETCH", "0") != "0" and world == 1,
            "note": "layer inputs are not chained (random-init weights overflow bf16 within a few layers); every layer routes and computes on the step's hidden state with its own router/expert weights"}



# ----------------------------------------------------------------------------------------------- whole decode step
def full_decode_leg(args, lib, native, dev, local_rank, layers, L, moe_layer_call, world):
    """The WHOLE DeepSeek-V3 decode step (BASELINE config 2: "... decode bs=1 ... MLA path"), one CUDA graph:
    61 x [input RMSNorm -> q_a / kv_a (Q4_K, ktb200_linear) -> q_a norm -> q_b -> kv norm + RoPE + paged cache write
    (ktb200_mla_prep) -> W_UK absorb (bmm) -> MLA paged decode over `ctx` cached tokens (ktb200_mla_decode, tcgen05) -> W_UV
    (bmm) -> o_proj -> residual + post RMSNorm -> dense MLP (3 layers) | MoE block (58 layers)] -> final norm -> lm_head.
    Weights synthetic at the real shapes and all resident and distinct except the MoE sets (the resident `layers`)."""
    import ctypes as C

    import torch

    from ktransformers_b200.util.synth import synth_blocks
    ctx = args.ctx
    NL, NH, QL, KVL, ROPE, NOPE, VD, DI, VOCAB = 61, 128, 1536, 512, 64, 128, 128, 18432, 129280
    PAGE = 64
    S = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731
    g = torch.Generator(device=dev); g.manual_seed(4242)
    bf = torch.bfloat16

    def linear(inf, outf, t, seed):
        w = synth_blocks(t, outf * inf, dev, seed)
        h = C.c_void_p()
        native.check(lib.ktb200_linear_create(inf, outf, w.data_ptr(), t, BF16, 8, local_rank, C.byref(h)))
        native.check(lib.ktb200_linear_load_weights(h, S()))
        return h, w

    def normw(n):
        return (1.0 + 0.1 * torch.randn(n, device=dev, generator=g)).to(bf)

    pages = (ctx + PAGE) // PAGE + 1
    att = []
    for l in range(NL):
        d = dict(qkv_a=linear(H, QL + KVL + ROPE, Q4_K, 9000 + 10 * l), q_b=linear(QL, NH * (NOPE + ROPE), Q4_K, 9002 + 10 * l),
                 o=linear(NH * VD, H, Q4_K, 9003 + 10 * l),
                 w_uk=(torch.randn(NH, NOPE, KVL, device=dev, generator=g) * 0.05).to(bf), w_uv=(torch.randn(NH, VD, KVL, device=dev, generator=g) * 0.05).to(bf),
                 ln_in=normw(H), ln_qa=normw(QL), ln_kv=normw(KVL), ln_post=normw(H),
                 cache=(torch.randn(pages, PAGE, KVL + ROPE, device=dev, generator=g) * 0.5).to(bf))
        att.append(d)
    dense = []
    for l in range(3):
        gw, uw, dw = synth_blocks(Q4_K, DI * H, dev, 7000 + l), synth_blocks(Q4_K, DI * H, dev, 7100 + l), synth_blocks(Q6_K, H * DI, dev, 7200 + l)
        mh = C.c_void_p()
        native.check(lib.ktb200_mlp_create(H, DI, gw.data_ptr(), uw.data_ptr(), dw.data_ptr(), Q4_K, Q4_K, Q6_K, BF16, 8, local_rank, C.byref(mh)))
        native.check(lib.ktb200_mlp_load_weights(mh, S()))
        dense.append((mh, gw, uw, dw))
    lm_head = linear(H, VOCAB, Q6_K, 6000)
    ln_final = normw(H)
    # static buffers
    x = torch.zeros(1, H, dtype=bf, device=dev); hbuf = torch.zeros(1, H, dtype=bf, device=dev); y = torch.zeros(1, H, dtype=bf, device=dev)
    qkva = torch.zeros(1, QL + KVL + ROPE, dtype=bf, device=dev)          # q_a and kv_a share their input: one projection, rows stacked
    qa, kva = qkva[:, :QL], qkva[:, QL:]
    qan = torch.zeros(1, QL, dtype=bf, device=dev)
    q = torch.zeros(1, NH * (NOPE + ROPE), dtype=bf, device=dev); q_pe = torch.zeros(NH, ROPE, dtype=bf, device=dev)
    q_abs = torch.zeros(NH, 1, KVL, dtype=bf, device=dev); lat = torch.zeros(1, NH, KVL, dtype=bf, device=dev)
    o_in = torch.zeros(NH, 1, VD, dtype=bf, device=dev); attn_out = torch.zeros(1, H, dtype=bf, device=dev)
    logits = torch.zeros(1, VOCAB, dtype=bf, device=dev)
    ids = torch.zeros(1, K, dtype=torch.int64, device=dev); wts = torch.zeros(1, K, dtype=torch.float32, device=dev)
    inv = 1.0 / (10000.0 ** (torch.arange(0, ROPE, 2, device=dev).float() / ROPE))
    ang = torch.cat([inv * ctx, inv * ctx])[None]
    cos, sin = ang.cos().contiguous(), ang.sin().contiguous()
    pidx = torch.tensor([ctx // PAGE], dtype=torch.int32, device=dev); poff = torch.tensor([ctx % PAGE], dtype=torch.int32, device=dev)
    ptab = torch.arange(pages, dtype=torch.int32, device=dev)[None].contiguous()
    klen = torch.tensor([ctx + 1], dtype=torch.int32, device=dev)
    wsb = lib.ktb200_mla_workspace_bytes(1, NH, 0)
    ws = torch.zeros(wsb, dtype=torch.uint8, device=dev)
    mla = [native.MlaParams(1, NH, PAGE, pages, 0, float((NOPE + ROPE) ** -0.5), q_abs.data_ptr(), q_pe.data_ptr(), a["cache"].data_ptr(), ptab.data_ptr(),
                            klen.data_ptr(), lat.data_ptr(), None, ws.data_ptr(), wsb, pages * PAGE) for a in att]
    eps = 1e-6

    def lin(hd, src, dst):
        native.check(lib.ktb200_linear_forward(hd[0], 1, src.data_ptr(), dst.data_ptr(), None, None, S()))

    def step(with_moe=True, with_attn=True):
        delta = None
        for l in range(NL):
            a = att[l]
            native.check(lib.ktb200_add_rmsnorm(x.data_ptr(), delta.data_ptr() if delta is not None else None, a["ln_in"].data_ptr(), eps, hbuf.data_ptr(), 1, H, S()))
            if with_attn:
                lin(a["qkv_a"], hbuf, qkva)
                native.check(lib.ktb200_add_rmsnorm(qa.data_ptr(), None, a["ln_qa"].data_ptr(), eps, qan.data_ptr(), 1, QL, S()))
                lin(a["q_b"], qan, q)
                native.check(lib.ktb200_mla_prep(q.data_ptr(), NH, NOPE, kva.data_ptr(), a["ln_kv"].data_ptr(), eps, cos.data_ptr(), sin.data_ptr(),
                                                 a["cache"].data_ptr(), PAGE, pidx.data_ptr(), poff.data_ptr(), q_pe.data_ptr(), 1, S()))
                native.check(lib.ktb200_mla_absorb_q(q.data_ptr(), NOPE + ROPE, NH * (NOPE + ROPE), a["w_uk"].data_ptr(), NH, NOPE, KVL, q_abs.data_ptr(), 1, S()))
                native.check(lib.ktb200_mla_decode(C.byref(mla[l]), S()))
                native.check(lib.ktb200_mla_absorb_o(lat.data_ptr(), a["w_uv"].data_ptr(), NH, VD, KVL, o_in.data_ptr(), 1, S()))
                lin(a["o"], o_in.view(1, NH * VD), attn_out)
                native.check(lib.ktb200_add_rmsnorm(x.data_ptr(), attn_out.data_ptr(), a["ln_post"].data_ptr(), eps, hbuf.data_ptr(), 1, H, S()))
            if l < 3:
                native.check(lib.ktb200_mlp_forward(dense[l][0], 1, hbuf.data_ptr(), y.data_ptr(), 0, None, S()))
            elif with_moe:
                moe_layer_call(l - 3, hbuf, y, ids, wts)
            delta = y
        native.check(lib.ktb200_add_rmsnorm(x.data_ptr(), y.data_ptr(), ln_final.data_ptr(), eps, hbuf.data_ptr(), 1, H, S()))
        lin(lm_head, hbuf, logits)

    def timed(fn, steps):
        n0 = native.launch_count()
        fn(); torch.cuda.synchronize()
        launches = native.launch_count() - n0
        side = torch.cuda.Stream(); side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            fn()
        torch.cuda.current_stream().wait_stream(side); torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            fn()
        for _ in range(3):
            x.normal_(0, 0.02); gr.replay()
        torch.cuda.synchronize()
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            gr.replay()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps, launches

    ms_full, launches = timed(lambda: step(True, True), args.steps)
    ms_noattn, _ = timed(lambda: step(True, False), args.steps)
    attn_bytes = NL * ((H * QL + H * (KVL + ROPE) + QL * NH * (NOPE + ROPE) + NH * VD * H) * 144 // 256 + 2 * NH * NOPE * KVL * 2 + (ctx + 1) * (KVL + ROPE) * 2)
    moe_bytes = N_MOE_LAYERS * ((K + 1) * BYTES_PER_EXPERT + E * H * 4) // (1 if world == 1 else 1)
    other_bytes = 3 * (2 * DI * H * 144 // 256 + H * DI * 210 // 256) + VOCAB * H * 210 // 256
    total = attn_bytes + moe_bytes + other_bytes
    peak = measured_peak_gbs()[0]
    x_host = torch.zeros(1, H, dtype=bf).pin_memory(); lg_host = torch.zeros(1, VOCAB, dtype=bf).pin_memory()
    return {"what": "whole DeepSeek-V3 decode step per GPU (61 attention + 3 dense + 58 MoE layers + lm_head), one CUDA graph", "ctx": ctx,
            "tok_s": world * 1000.0 / ms_full, "ms_per_token": ms_full, "ms_without_attention": ms_noattn, "ms_attention_61_layers": ms_full - ms_noattn,
            "our_launches_per_token": launches, "algorithmic_bytes_per_token": {"attention": attn_bytes, "moe": moe_bytes, "dense_mlp_lm_head": other_bytes, "total": total},
            "achieved_GBps": total / (ms_full * 1e-3) / 1e9, "frac_of_peak": total / (ms_full * 1e-3) / 1e9 / peak,
            "attention_GBps": attn_bytes / ((ms_full - ms_noattn) * 1e-3) / 1e9,
            "note": "every kernel in the step is this repo's (no library GEMM); q_a and kv_a are one stacked projection"}

# ----------------------------------------------------------------------------------------------- B200 arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--resident-layers", type=int, default=8)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ctx", type=int, default=4096, help="cached tokens per sequence in the whole-step leg")
    ap.add_argument("--no-full-step", action="store_true")
    ap.add_argument("--no-prefill", action="store_true", help="skip the 1024-token grouped-GEMM leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy: the MoE block output, routed ids "
                         "and weights of its last layer (every layer of a step writes the same buffers)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the b200 arm")
    # This process owns the GPU and decodes on ONE stream: the persistent MoE-block kernel is launched as a plain grid
    # with programmatic dependent launch (its 148 CTAs become co-resident as the previous layer's CTAs exit) instead of
    # cooperatively — the cooperative attribute (library default: safe when several streams share the GPU) makes every
    # launch wait for the previous grid to drain and costs ~4 % here.  Recorded in config["block_launch"].
    os.environ.setdefault("KTB200_BLK_COOP", "0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    from ktransformers_b200 import native
    from ktransformers_b200.util.synth import synth_blocks

    assert torch.cuda.is_available(), "the B200 path has no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = native.lib()
    stream = torch.cuda.current_stream()
    S = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731

    E_local = E // world
    L = args.resident_layers

    # ---- expert-parallel exchange buffers (world > 1): one symmetric allocation per rank holds the message buffer
    # ({x, ids, weights} rows), the fp32 partial buffer and the flag block of ktb200_moe_ep_block_forward; torch's symmetric
    # memory maps the peers' copies.  KTB200_EP_P2P=0 (or a failing rendezvous) keeps NCCL collectives + separate kernels.
    T = world                                                  # tokens in flight per layer (one per GPU)
    ep = None
    ep_mode = "nccl all_gather + reduce_scatter, separate kernels"
    if world > 1 and os.environ.get("KTB200_EP_P2P", "1") != "0":
        try:
            import torch.distributed._symmetric_memory as symm_mem
            msg_b, part_b, flag_b = T * lib.ktb200_ep_msg_bytes(H, BF16), T * H * 4, 4 * (2 * T + 2)
            o_part = (msg_b + 255) // 256 * 256
            o_flag = o_part + (part_b + 255) // 256 * 256
            total_b = o_flag + (flag_b + 255) // 256 * 256
            sym = symm_mem.empty(total_b, dtype=torch.uint8, device=dev)
            sym.zero_()
            hdl = symm_mem.rendezvous(sym, dist.group.WORLD)
            base = [int(p_) for p_ in hdl.buffer_ptrs]
            ep = native.EpComm.make(rank, world, H, BF16, base, [b + o_part for b in base], [b + o_flag for b in base])
            ep_flags = sym[o_flag:o_flag + flag_b].view(torch.int32)
            torch.cuda.synchronize(); dist.barrier()
            ep_mode = "ONE launch per layer (ktb200_moe_ep_block_forward): router of the own token, NVLink peer-memory push of {x, ids, w}, owned (token, expert) pairs, push of partial sums, combine"
        except Exception as e:  # pragma: no cover
            if rank == 0:
                print(f"# symmetric memory unavailable ({type(e).__name__}: {e}); using NCCL", file=sys.stderr)
            ep = None
        ok = torch.tensor([1 if ep is not None else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)               # all ranks or none
        if int(ok.item()) == 0:
            ep, ep_mode = None, "nccl all_gather + reduce_scatter, separate kernels"
    hid = BF16 if (world == 1 or ep is not None) else F32      # NCCL route: fp32 partial sums are reduce-scattered, then rounded once
    hid_torch = torch.bfloat16 if hid == BF16 else torch.float32

    # ---- resident weight sets ---------------------------------------------------------------------------------
    layers = []
    raw0 = None                                                 # layer 0's down tensor before the in-place Q6_K re-tiling (parity check)
    for l in range(L):
        seed = 1000 * l + 17 * rank
        gate = synth_blocks(Q4_K, E_local * I * H, dev, seed + 1)
        up = synth_blocks(Q4_K, E_local * I * H, dev, seed + 2)
        down = synth_blocks(Q6_K, E_local * H * I, dev, seed + 3)
        sg, su, sd = (synth_blocks(Q4_K, I * H, dev, 1000 * l + 5), synth_blocks(Q4_K, I * H, dev, 1000 * l + 6),
                      synth_blocks(Q6_K, H * I, dev, 1000 * l + 7))
        if l == 0:
            raw0 = dict(down=down.clone(), sg=sg.cpu().numpy(), su=su.cpu().numpy(), sd=sd.cpu().numpy())
        cfg = native.MoeConfig(E_local, K, H, I, 64, 10, PREFILL_TOKENS if world == 1 else max(8, world), 1, gate.data_ptr(), up.data_ptr(), down.data_ptr(),
                               Q4_K, Q4_K, Q6_K, hid, rank * E_local)
        h = C.c_void_p()
        native.check(lib.ktb200_moe_create(C.byref(cfg), local_rank, C.byref(h)))
        native.check(lib.ktb200_moe_load_weights(h, S()))
        mh = C.c_void_p()
        native.check(lib.ktb200_mlp_create(H, I, sg.data_ptr(), su.data_ptr(), sd.data_ptr(), Q4_K, Q4_K, Q6_K, BF16, 8, local_rank, C.byref(mh)))
        native.check(lib.ktb200_mlp_load_weights(mh, S()))
        g = torch.Generator(device=dev); g.manual_seed(1000 * l + 9)
        Wr = torch.randn((E, H), device=dev, generator=g, dtype=torch.float32)
        # e_score_correction_bias: a trained model's bias keeps the experts balanced; a randn bias (std 1 against sigmoid
        # scores in 0.3..0.7) would send EVERY token to the same few experts — harmless at N = 1, a pathological 2x load
        # imbalance for expert-parallel shards (measured: profiles/ep_trace_n8_r02.txt).  The reference's own MoE bench routes
        # uniformly at random (kt-kernel/bench/bench_moe.py:235-239); a small bias keeps the routing token-dependent.
        br = 0.01 * torch.randn((E,), device=dev, generator=g, dtype=torch.float32)
        gcfg = native.GateConfig(E, H, K, N_GROUP, TOPK_GROUP, 0, 0, 1, ROUTED_SCALE, Wr.data_ptr(), br.data_ptr(), BF16)
        layers.append(dict(moe=h, mlp=mh, gcfg=gcfg, keep=(gate, up, down, sg, su, sd, Wr, br)))
    if world == 1 and os.environ.get("KTB200_BENCH_PREFETCH", "0") != "0":
        # chain the layers: while layer i streams its down projection it pulls layer i+1's router rows and shared-expert
        # gate/up rows into L2 (ktb200_moe_block_prefetch_hint) — the same bytes, requested earlier
        for i, Lr in enumerate(layers):
            nxt = layers[(i + 1) % L]["keep"]
            ptrs = (C.c_void_p * 3)(nxt[6].data_ptr(), nxt[3].data_ptr(), nxt[4].data_ptr())
            sizes = (C.c_size_t * 3)(nxt[6].numel() * 4, nxt[3].numel(), nxt[4].numel())
            native.check(lib.ktb200_moe_block_prefetch_hint(Lr["moe"], ptrs, sizes, 3))
    torch.cuda.synchronize()

    # ---- static buffers ---------------------------------------------------------------------------------------
    x_own = torch.zeros((1, H), dtype=torch.bfloat16, device=dev)          # this GPU's token
    x_all = torch.zeros((T, H), dtype=torch.bfloat16, device=dev)
    x_all_f32 = torch.zeros((T, H), dtype=torch.float32, device=dev)
    ids = torch.zeros((T, K), dtype=torch.int64, device=dev)
    wts = torch.zeros((T, K), dtype=torch.float32, device=dev)
    part = torch.zeros((T, H), dtype=hid_torch, device=dev)                # NCCL route: fp32 partial sums
    own_f32 = torch.zeros((1, H), dtype=torch.float32, device=dev)
    y = torch.zeros((1, H), dtype=torch.bfloat16, device=dev)              # layer output for this GPU's token
    x_host = torch.zeros((1, H), dtype=torch.bfloat16).pin_memory()
    y_host = torch.zeros((1, H), dtype=torch.bfloat16).pin_memory()
    out_host = torch.zeros((1, H), dtype=torch.bfloat16).pin_memory()
    side_stream = torch.cuda.Stream() if world > 1 else None
    y_sh = torch.zeros((1, H), dtype=torch.bfloat16, device=dev)

    def layer_device(l):
        Lr = layers[l % L]
        if world == 1:
            # KDeepseekV3MoE.forward in one call: router + routed experts + shared expert (one persistent launch)
            native.check(lib.ktb200_moe_block_forward(C.byref(Lr["gcfg"]), Lr["moe"], Lr["mlp"], 1, x_own.data_ptr(), y.data_ptr(),
                                                      ids.data_ptr(), wts.data_ptr(), None, S()))
            return
        if ep is not None:
            native.check(lib.ktb200_moe_ep_block_forward(C.byref(Lr["gcfg"]), Lr["moe"], Lr["mlp"], C.byref(ep), x_own.data_ptr(), y.data_ptr(),
                                                         ids.data_ptr(), wts.data_ptr(), 7, S()))
            return
        main = torch.cuda.current_stream()
        # NCCL route: the shared expert of this GPU's own token needs no communication: it runs on a side stream under the
        # all-gather, and joins as the second rounded term
        side_stream.wait_stream(main)
        with torch.cuda.stream(side_stream):
            native.check(lib.ktb200_mlp_forward(Lr["mlp"], 1, x_own.data_ptr(), y_sh.data_ptr(), 0, None, S()))
        dist.all_gather_into_tensor(x_all, x_own)
        native.check(lib.ktb200_moe_gate_forward(C.byref(Lr["gcfg"]), T, x_all.data_ptr(), ids.data_ptr(), wts.data_ptr(), None, None, S()))
        x_all_f32.copy_(x_all)
        native.check(lib.ktb200_moe_forward(Lr["moe"], T, K, ids.data_ptr(), wts.data_ptr(), x_all_f32.data_ptr(), part.data_ptr(), None, S()))
        dist.reduce_scatter_tensor(own_f32, part)
        y.copy_(own_f32)
        main.wait_stream(side_stream)
        y.add_(y_sh)

    def step_device():
        for l in range(N_MOE_LAYERS):
            layer_device(l)

    rng = np.random.default_rng(1234 + rank)

    def fresh_input(gen=rng):
        x_host.copy_(torch.from_numpy((gen.standard_normal((1, H)) / 100).astype(np.float32)).to(torch.bfloat16))

    # ---- parity check (outside every timed region): layer 0's output for this step's token against the CPU oracle ------
    parity = None
    try:
        from oracle.bindings import Oracle, bf16_to_f32
        from oracle import gate_oracle
        orc = Oracle()
        fresh_input(); x_own.copy_(x_host); torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        layer_device(0)
        torch.cuda.synchronize()
        Lr = layers[0]
        gate_t, up_t = Lr["keep"][0], Lr["keep"][1]
        gbytes, dbytes = gate_t.numel() // E_local, raw0["down"].numel() // E_local
        bits = lambda t: t.detach().cpu().contiguous().view(torch.int16).numpy().view(np.uint16)
        if world > 1:
            xs_all = torch.zeros((T, H), dtype=torch.bfloat16, device=dev); dist.all_gather_into_tensor(xs_all, x_own)
            ids_all = torch.zeros((T, K), dtype=torch.int64, device=dev); dist.all_gather_into_tensor(ids_all, ids[:1].contiguous())
            w_all = torch.zeros((T, K), dtype=torch.float32, device=dev); dist.all_gather_into_tensor(w_all, wts[:1].contiguous())
        else:
            xs_all, ids_all, w_all = x_own, ids[:1], wts[:1]
        ids_np, w_np, xs_bits = ids_all.cpu().numpy(), w_all.cpu().numpy(), bits(xs_all)
        # routing of the own token vs the float64 router restatement
        Wr, br = Lr["keep"][6].cpu().numpy(), Lr["keep"][7].cpu().numpy()
        oidx, _, margin, _ = gate_oracle.route(bf16_to_f32(xs_bits[rank:rank + 1]), Wr, br, top_k=K, n_group=N_GROUP, topk_group=TOPK_GROUP,
                                               routed_scaling_factor=ROUTED_SCALE, dtype=np.float64)
        ids_equal = bool(np.array_equal(np.sort(ids_np[rank]), np.sort(oidx[0])))
        # routed experts: the oracle over the experts THIS rank owns, for all `world` tokens, in fp32; ranks are summed
        own = (ids_np >= rank * E_local) & (ids_np < (rank + 1) * E_local)
        sel = sorted(set(ids_np[own].tolist()))
        remap = {e: i for i, e in enumerate(sel)}
        loc = np.vectorize(lambda e: remap.get(int(e), -1))(ids_np).astype(np.int64)
        if sel:
            g_np = torch.cat([gate_t[(e - rank * E_local) * gbytes:(e - rank * E_local + 1) * gbytes] for e in sel]).cpu().numpy()
            u_np = torch.cat([up_t[(e - rank * E_local) * gbytes:(e - rank * E_local + 1) * gbytes] for e in sel]).cpu().numpy()
            d_np = torch.cat([raw0["down"][(e - rank * E_local) * dbytes:(e - rank * E_local + 1) * dbytes] for e in sel]).cpu().numpy()
            routed = orc.moe_forward(len(sel), H, I, g_np, u_np, d_np, Q4_K, Q4_K, Q6_K, F32, loc, w_np, bf16_to_f32(xs_bits))
        else:
            routed = np.zeros((T, H), np.float32)
        routed_t = torch.from_numpy(routed).to(dev)
        if world > 1:
            dist.all_reduce(routed_t)
        shared = orc.mlp_forward(H, I, raw0["sg"], raw0["su"], raw0["sd"], Q4_K, Q4_K, Q6_K, BF16, xs_bits[rank:rank + 1])
        want = (routed_t[rank:rank + 1].to(torch.bfloat16).cpu() + torch.from_numpy(shared.view(np.int16)).view(torch.bfloat16)).float().numpy()
        got = y.float().cpu().numpy()
        max_rel = float(np.abs(got - want).max() / max(np.abs(want).max(), 1e-30))
        stat = torch.tensor([max_rel, 0.0 if ids_equal else 1.0, float(margin[0] < 1e-5)], device=dev)
        if world > 1:
            dist.all_reduce(stat, op=dist.ReduceOp.MAX)
        parity = {"layer": 0, "checked_against": "oracle/ktoracle.c (routed experts, fp32 partial sums summed over ranks) + gate_oracle (float64 router)",
                  "max_rel": float(stat[0]), "ids_equal": bool(stat[1] == 0.0), "knife_edge_token": bool(stat[2] > 0), "tolerance": "2^-7 (1 bf16 ulp of the two rounded terms) + 1e-3"}
        if ep is not None:
            parity["ep_wait_timeouts"] = int(ep_flags[2 * T + 1].item())
    except Exception as e:  # pragma: no cover  (the checker must never take the bench down)
        parity = {"error": f"{type(e).__name__}: {e}"}
    raw0 = None
    torch.cuda.empty_cache()

    # warm (allocations inside the library happen here, before capture)
    n0 = native.launch_count()
    step_device()
    torch.cuda.synchronize()
    launches_per_step = native.launch_count() - n0
    graph = None
    if not args.no_graph:
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                step_device()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                step_device()
            torch.cuda.synchronize()
        except Exception as e:  # pragma: no cover
            if rank == 0:
                print(f"# CUDA graph capture failed ({e}); running eagerly", file=sys.stderr)
            graph = None
            torch.cuda.synchronize()

    def run_step():
        if graph is not None:
            graph.replay()
        else:
            step_device()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: inputs resident in HBM ------------------------------------------------------------------------
    sampler = ClockSampler(local_rank) if rank == 0 else None     # sampling spans the warm-up steps too: the same work, enough samples
    for _ in range(max(3, args.warmup)):
        fresh_input(); x_own.copy_(x_host, non_blocking=True); run_step()
    barrier()
    # nvidia-smi needs up to a few seconds before its first row on a fresh box and the timed region lasts ~0.1 s: keep the GPU(s)
    # under the same load (more untimed steps) until rank 0's sampler is live, so that the timed region is actually sampled.
    # Every rank must run the same steps (the expert-parallel layer is a collective): rank 0 decides, everyone follows.
    t_wait = time.perf_counter()
    while True:
        more = 1 if (sampler is not None and sampler.p is not None and sampler.rows() == 0 and time.perf_counter() - t_wait < 8.0) else 0
        if world > 1:
            flag = torch.tensor([more], device=dev, dtype=torch.int32)
            dist.broadcast(flag, 0)
            more = int(flag.item())
        if not more:
            break
        run_step(); torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    # the timed token has a generator of its own: it does not depend on how many draws the parity check and warm-up took
    fresh_input(np.random.default_rng(4321 + rank)); x_own.copy_(x_host); barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        run_step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    t_ms = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(t_ms.item()) / args.steps
    value = world * 1000.0 / ms_per_step

    # ---- the last timed step's outputs, for comparing two builds on the same seeded inputs --------------------------------
    # Every layer of a step reads the same token and writes these buffers, so they hold what the step's last layer returned.
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in (("moe_out", y.float().cpu().numpy()), ("topk_ids", ids.cpu().numpy().astype(np.float64)),
                          ("topk_weights", wts.cpu().numpy())):
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)

    # ---- e2e: host buffers, copies inside the timed region ----------------------------------------------------
    if world == 1:
        # the reference-facing call: per layer ids/weights come off the GPU router into pinned memory, then
        # MOE.forward(qlen,k,ids,w,input,output) with HOST pointers == ktb200_moe_forward_host
        def e2e_step():
            for l in range(N_MOE_LAYERS):
                Lr = layers[l % L]
                native.check(lib.ktb200_moe_block_forward_host(C.byref(Lr["gcfg"]), Lr["moe"], Lr["mlp"], 1, x_host.data_ptr(), out_host.data_ptr(),
                                                               None, None, S()))
            return out_host
        h2d = N_MOE_LAYERS * H * 2
        d2h = N_MOE_LAYERS * H * 2
        e2e_api = "per layer: ktb200_moe_block_forward_host(pinned host token -> pinned host output): H2D copy, one launch whose stores land in the pinned output (the D2H transfer), sync"
    else:
        # same shape as N=1: every layer is one plugin call with HOST buffers (token up, layer, output back, synchronise)
        def e2e_step():
            for l in range(N_MOE_LAYERS):
                x_own.copy_(x_host, non_blocking=True)
                layer_device(l)
                y_host.copy_(y, non_blocking=True)
                torch.cuda.current_stream().synchronize()
        h2d, d2h = N_MOE_LAYERS * H * 2, N_MOE_LAYERS * H * 2
        e2e_api = "per layer and rank: pinned host token -> H2D -> expert-parallel layer (one launch, NVLink exchange inside) -> D2H -> sync"
    for _ in range(3):
        fresh_input(); e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fresh_input(); e2e_step()
    barrier()
    e2e_s = (time.perf_counter() - t0) / args.steps
    t_e = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e_value = world / float(t_e.item())

    # ---- roofline: live CUDA-event pass over the two MoE kernels, cold weights every layer --------------------
    roof = roof_down = roof_block = None
    if rank == 0 and world == 1:
        # the persistent MoE-block kernel, one launch per layer, CUDA events on the launching stream
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(N_MOE_LAYERS)]
        tb = []
        for rep in range(3):
            n0 = native.launch_count()
            for l in range(N_MOE_LAYERS):
                Lr = layers[l % L]
                evs[l][0].record()
                native.check(lib.ktb200_moe_block_forward(C.byref(Lr["gcfg"]), Lr["moe"], Lr["mlp"], 1, x_own.data_ptr(), y.data_ptr(),
                                                          ids.data_ptr(), wts.data_ptr(), None, S()))
                evs[l][1].record()
            torch.cuda.synchronize()
            fused_launches = native.launch_count() - n0 == N_MOE_LAYERS
            if rep:
                tb += [a_.elapsed_time(b_) for a_, b_ in evs]
        if fused_launches:
            peak, how = measured_peak_gbs()
            ms_b = statistics.mean(tb)
            bytes_b = (K + 1) * BYTES_PER_EXPERT + E * H * 4
            roof_block = {"kernel": "moe_block_kernel<BulkQ6K4T> (router GEMV + top-k + gate/up + SiLU*mul + down + combine, 1 launch/layer)",
                          "bound": "hbm", "achieved": bytes_b / (ms_b * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                          "frac": bytes_b / (ms_b * 1e-3) / 1e9 / peak, "peak_source": how,
                          "traffic": committed_traffic("moe_block_kernel"),
                          "bytes_per_launch": bytes_b, "ms_per_launch": ms_b}
    if rank == 0 and hid == BF16:
        gu, dn = [], []
        a, b = C.c_float(), C.c_float()
        xin = x_own
        for rep in range(2):
            for l in range(N_MOE_LAYERS):
                Lr = layers[l % L]
                native.check(lib.ktb200_moe_gate_forward(C.byref(Lr["gcfg"]), 1, x_own.data_ptr(), ids.data_ptr(), wts.data_ptr(), None, None, S()))
                if world > 1:
                    ids.remainder_(E_local).add_(rank * E_local)     # all 8 local: measures the kernel, not the sharding
                native.check(lib.ktb200_moe_forward_timed(Lr["moe"], 1, K, ids.data_ptr(), wts.data_ptr(), xin.data_ptr(), part.data_ptr(), S(), C.byref(a), C.byref(b)))
                if rep:
                    gu.append(a.value); dn.append(b.value)
        peak, how = measured_peak_gbs()
        ms_gu, ms_dn = statistics.mean(gu), statistics.mean(dn)
        ach = K * BYTES_GATE_UP_PER_EXPERT / (ms_gu * 1e-3) / 1e9   # routed launch only (ktb200_moe_forward_timed has no shared slot)
        roof = {"kernel": "rows_bulk_q4k_kernel<PAIR> (gate/up GEMV + SiLU*mul; separate-launch path)", "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                "frac": ach / peak, "peak_source": how, "traffic": None, "bytes_per_launch": K * BYTES_GATE_UP_PER_EXPERT, "ms_per_launch": ms_gu}
        achd = K * BYTES_DOWN_PER_EXPERT / (ms_dn * 1e-3) / 1e9
        roof_down = {"kernel": "reduce_bulk_kernel<BulkQ6K4T> (down GEMV + weighted sum; separate-launch path)", "bound": "hbm", "achieved": achd, "peak": peak, "unit": "GB/s",
                     "frac": achd / peak, "bytes_per_launch": K * BYTES_DOWN_PER_EXPERT, "ms_per_launch": ms_dn}

    # ---- prefill-sized batch through the same handles: router + grouped tensor-core expert GEMMs (MOE::forward_many) ---------
    prefill = None
    if rank == 0 and world == 1 and not args.no_prefill:
        try:
            Tp = PREFILL_TOKENS
            gp_ = torch.Generator(device=dev); gp_.manual_seed(4242)
            xp = (torch.randn((Tp, H), device=dev, generator=gp_) / 10).to(torch.bfloat16)
            idp = torch.zeros((Tp, K), dtype=torch.int64, device=dev)
            wtp = torch.zeros((Tp, K), dtype=torch.float32, device=dev)
            yp = torch.zeros((Tp, H), dtype=torch.bfloat16, device=dev)

            # routing of the reference's own MoE bench (kt-kernel/bench/bench_moe.py:235-239): uniformly random experts, rand weights
            idp.copy_(torch.rand((Tp, E), device=dev, generator=gp_).argsort(dim=1)[:, :K])
            wtp.copy_(torch.rand((Tp, K), device=dev, generator=gp_))

            def prefill_layer(l):
                Lr = layers[l % L]
                native.check(lib.ktb200_moe_forward(Lr["moe"], Tp, K, idp.data_ptr(), wtp.data_ptr(), xp.data_ptr(), yp.data_ptr(), None, S()))
            for l in range(L):
                prefill_layer(l)
            torch.cuda.synchronize()
            n0 = native.launch_count()
            reps = 2 * L
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for l in range(reps):
                prefill_layer(l)        # L resident layer sets of 7.3 GB each: far larger than L2, every pass is cold
            e1.record(); torch.cuda.synchronize()
            ms_l = e0.elapsed_time(e1) / reps
            experts_hit = int(torch.unique(idp).numel())
            peak, how = measured_peak_gbs()
            bytes_l = experts_hit * BYTES_PER_EXPERT
            prefill = {"tokens": Tp, "ms_per_layer": ms_l, "launches_per_layer": (native.launch_count() - n0) // reps,
                       "tok_s_moe_58_layers": Tp / (N_MOE_LAYERS * ms_l * 1e-3), "experts_hit": experts_hit,
                       "tflops_equiv": 2.0 * Tp * K * 3 * H * I / (ms_l * 1e-3) / 1e12,
                       "hbm": {"algorithmic_bytes": bytes_l, "achieved_GBps": bytes_l / (ms_l * 1e-3) / 1e9, "frac": bytes_l / (ms_l * 1e-3) / 1e9 / peak, "peak_source": how},
                       "path": "MOE.forward on 1024 tokens, routing like kt-kernel/bench/bench_moe.py (uniform random): count/scan/scatter + Q8_K quantise + 3 grouped tcgen05 kind::i8 GEMMs + combine (csrc/grouped.cu); parity: tests/test_gpu_parity.py -k grouped"}
        except Exception as e:  # pragma: no cover
            prefill = {"error": f"{type(e).__name__}: {e}"}

    # ---- FP8 128 x 128 linear (KLinearFP8, BASELINE configs 3 / 5) at two DeepSeek-V3 projection shapes, bs 1 -------------------
    fp8 = None
    if rank == 0 and world == 1 and not args.no_prefill:
        try:
            fp8 = {"kernel": "fp8_linear_kernel (TMA -> tcgen05.mma.kind::f8f6f4 -> TMEM, csrc/fp8_linear.cu)", "bound": "hbm", "shapes": {}}
            peak, how = measured_peak_gbs()
            for name, Kf, Nf, copies in (("lm_head 7168->129280", 7168, 129280, 2), ("o_proj 16384->7168", 16384, 7168, 4)):
                hs, keep = [], []
                for c in range(copies):     # cycled weight copies: no call finds its weights in L2
                    wq = torch.randint(0, 120, (Nf, Kf), dtype=torch.uint8, device=dev)
                    wsc = torch.rand(((Nf + 127) // 128, Kf // 128), device=dev) * 0.01 + 0.001
                    hh_ = C.c_void_p()
                    native.check(lib.ktb200_fp8_linear_create(Kf, Nf, wq.data_ptr(), wsc.data_ptr(), BF16, local_rank, C.byref(hh_)))
                    hs.append(hh_); keep.append((wq, wsc))
                xf = (torch.randn(1, Kf, device=dev) / 10).to(torch.bfloat16); yf = torch.zeros(1, Nf, dtype=torch.bfloat16, device=dev)
                for i in range(copies):
                    native.check(lib.ktb200_fp8_linear_forward(hs[i], 1, xf.data_ptr(), yf.data_ptr(), None, S()))
                torch.cuda.synchronize()
                n_it = 5 * copies
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(n_it):
                    native.check(lib.ktb200_fp8_linear_forward(hs[i % copies], 1, xf.data_ptr(), yf.data_ptr(), None, S()))
                e1.record(); torch.cuda.synchronize()
                us = e0.elapsed_time(e1) / n_it * 1e3
                fp8["shapes"][name] = {"us": us, "achieved_GBps": Kf * Nf / us / 1e3, "frac": Kf * Nf / us / 1e3 / peak, "bytes": Kf * Nf}
                for hh_ in hs:
                    lib.ktb200_fp8_linear_destroy(hh_)
                del keep
            fp8["peak"], fp8["peak_source"] = peak, how
        except Exception as e:  # pragma: no cover
            fp8 = {"error": f"{type(e).__name__}: {e}"}

    # ---- the whole decode step (attention + dense + MoE + lm_head), every rank its own token ------------------------
    full = None
    if not args.no_full_step:
        try:
            def moe_call(i, xin, yout, ids_, wts_):
                Lr = layers[i % L]
                if world == 1:
                    native.check(lib.ktb200_moe_block_forward(C.byref(Lr["gcfg"]), Lr["moe"], Lr["mlp"], 1, xin.data_ptr(), yout.data_ptr(),
                                                              ids_.data_ptr(), wts_.data_ptr(), None, S()))
                elif ep is not None:
                    native.check(lib.ktb200_moe_ep_block_forward(C.byref(Lr["gcfg"]), Lr["moe"], Lr["mlp"], C.byref(ep), xin.data_ptr(), yout.data_ptr(),
                                                                 ids_.data_ptr(), wts_.data_ptr(), 7, S()))
                else:
                    raise RuntimeError("whole-step leg needs the peer-memory EP path")
            full = full_decode_leg(args, lib, native, dev, local_rank, layers, L, moe_call, world)
        except Exception as e:  # pragma: no cover
            full = {"error": f"{type(e).__name__}: {e}"}
        if world > 1:
            dist.barrier()

    # ---- CPU baseline (rank 0, N=1 only): the reference's CPU MoE on this box's host cores ---------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = RefCpuMoe()
        for l in range(20):
            cpu.layer(l)
        t0 = time.perf_counter(); n = 0
        while time.perf_counter() - t0 < 12.0 and n < 4000:
            cpu.layer(n); n += 1
        t_layer = (time.perf_counter() - t0) / n
        cpu_baseline = {"value": 1.0 / (N_MOE_LAYERS * t_layer), "unit": "tok/s", "cores": cpu.threads, "kind": cpu.kind,
                        "sample": cpu.describe(n), "ms_per_layer": t_layer * 1e3,
                        "gbs": K * BYTES_PER_EXPERT / t_layer / 1e9, "amx": amx_baseline()}

    if rank == 0:
        step_bytes = N_MOE_LAYERS * ((K + 1) * BYTES_PER_EXPERT + E * H * 4)
        line = {"metric": METRIC, "value": value, "unit": "tok/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "int8xint4/int6->int32 dp4a, fp32 scales+accumulate, bf16 in/out", "data": "synthetic",
                "config": {**workload_config(args, world), **({"ep_exchange": ep_mode} if world > 1 else {})}, "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "tok/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "api": e2e_api},
                "gpu_launches": launches_per_step * args.steps, "cuda_graph": graph is not None,
                "roofline": roof_block if roof_block else roof, "roofline_gate_up": roof, "roofline_down": roof_down, "cpu_baseline": cpu_baseline,
                "parity_check": parity, "full_decode": full, "prefill_grouped": prefill, "fp8_linear": fp8,
                "step_hbm": {"algorithmic_bytes_per_token_per_gpu": step_bytes, "achieved_GBps": step_bytes / (ms_per_step * 1e-3) / 1e9,
                             "frac_of_peak": step_bytes / (ms_per_step * 1e-3) / 1e9 / measured_peak_gbs()[0]}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        # tearing NCCL down with captured graphs alive can hang in destroy_process_group: leave by the fast door
        os._exit(0)


if __name__ == "__main__":
    main()
