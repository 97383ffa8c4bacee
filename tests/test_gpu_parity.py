"""GPU parity tests proper: the CUDA path, called through the C-ABI (include/ktb200.h), against
  (1) the committed golden vectors minted from the unmodified reference,
  (2) the CPU oracle (oracle/ktoracle.c) on the same seeded inputs at sizes it finishes in seconds,
  (3) size-independent properties at BASELINE's full DeepSeek-V3 shapes.
Tolerances: activation quantisation and routed ids are exact; fp32 outputs within 1e-3 of the reference
(north_star) — typically 1e-6, the bound leaves room for the one-LSB int8 knife-edge flips that even two
builds of the reference exhibit between each other; bf16 outputs additionally within 1 bf16 ulp."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from ktransformers_b200 import native
from ktransformers_b200.util.synth import synth_blocks
from oracle import gate_oracle
from oracle.bindings import (BF16, F16, F32, IQ4_XS, Q2_K, Q3_K, Q4_K, Q5_K, Q6_K, Q8_0, Q8_K, TYPE_NAMES, bf16_to_f32,
                             f32_to_bf16_bits)
import gpu_util as G

pytestmark = pytest.mark.gpu
TYPES = {n: t for t, n in TYPE_NAMES.items()}
FP_TOL = 1e-3


def relmax(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def assert_bf16_close(got_bits, want_bits, min_exact=0.97, ulps=1):
    a, b = bf16_to_f32(got_bits), bf16_to_f32(want_bits)
    assert (np.abs(a - b) <= ulps * 2.0 ** -7 * np.maximum(np.abs(a), np.abs(b)) + FP_TOL * np.abs(b).max()).all()
    assert (got_bits == want_bits).mean() > min_exact, (got_bits == want_bits).mean()


def test_library_is_the_cuda_path():
    assert os.path.exists(native.LIB_PATH)
    assert b"sm_100a" in native.lib().ktb200_version()
    assert torch.cuda.get_device_capability()[0] == 10


# ------------------------------------------------------------------------------------------ activation quantisation
def test_q8k_q8_0_quantisation_byte_exact_vs_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "act_quant.npz"))
    x = g["x"]
    got = G.quantize(x, F32, Q8_K)
    want = g["q8k"].copy()
    for i in range(x.shape[0]):
        for b in range(x.shape[1] // 256):
            if not x[i, b * 256:(b + 1) * 256].any():
                want[i, b * 292 + 260:(b + 1) * 292] = 0      # stale bsums of an all-zero block in the reference
    assert np.array_equal(got, want)
    assert np.array_equal(G.quantize(x, F32, Q8_0), g["q8_0"])


@pytest.mark.parametrize("hid", [F32, BF16, F16])
def test_q8k_quantisation_byte_exact_vs_oracle(oracle, hid):
    rng = np.random.default_rng(7)
    x = (rng.standard_normal((33, 2048)) * np.exp(rng.uniform(-6, 3, (33, 1)))).astype(np.float32)
    x[3, 256:512] = 0
    x[5, :] = -x[5, :].__abs__()           # all-negative row: sign of `max`
    if hid == BF16:
        xin = f32_to_bf16_bits(x); xf = bf16_to_f32(xin)
    elif hid == F16:
        xin = x.astype(np.float16); xf = xin.astype(np.float32)
    else:
        xin = x; xf = x
    got = G.quantize(xin, hid, Q8_K)
    want = np.stack([oracle.from_float(r, Q8_K) for r in xf])
    assert np.array_equal(got, want)
    assert np.array_equal(G.quantize(xin, hid, Q8_0), np.stack([oracle.from_float(r, Q8_0) for r in xf]))


# ------------------------------------------------------------------------------------------ dequantisation
@pytest.mark.parametrize("name", ["Q2_K", "Q3_K", "Q4_K", "Q5_K", "Q6_K", "IQ4_XS", "Q8_0"])
def test_dequantise_vs_golden(golden_dir, name):
    g = np.load(os.path.join(golden_dir, "dequant.npz"))
    want = g[f"val_{name}"]
    got = G.dequantize(g[f"raw_{name}"], TYPES[name], want.size, F32).numpy()
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-6)     # archive/ktransformers/tests/dequant_gpu.py:39
    got16 = G.dequantize(g[f"raw_{name}"], TYPES[name], want.size, BF16).float().numpy()
    assert np.abs(got16 - want).max() <= 2.0 ** -8 * np.abs(want).max() + 1e-6


# ------------------------------------------------------------------------------------------ MoE vs golden
@pytest.mark.parametrize("case", ["a", "b"])
def test_moe_forward_vs_golden(moe_small, case):
    g = moe_small
    E, k, H, I = (int(g[f"{case}_{n}"]) for n in ("E", "k", "H", "I"))
    gt, ut, dt = (int(g[f"{case}_{n}"]) for n in ("gate_type", "up_type", "down_type"))
    for hid in (F32, BF16):
        m = G.Moe(E, k, H, I, g[f"{case}_gate"], g[f"{case}_up"], g[f"{case}_down"], gt, ut, dt, hid)
        for qlen in (1, 3, 12):
            if f"{case}_x_{qlen}" not in g:
                continue
            x, ids, w = g[f"{case}_x_{qlen}"], g[f"{case}_ids_{qlen}"], g[f"{case}_w_{qlen}"]
            if hid == F32:
                out = m.forward(ids, w, x)
                assert relmax(out, g[f"{case}_out_f32_{qlen}"]) < FP_TOL
                assert np.array_equal(m.forward_host(ids, w, x), out)      # host-buffer entry point == device entry point
            else:
                assert_bf16_close(m.forward(ids, w, f32_to_bf16_bits(x)), g[f"{case}_out_bf16_{qlen}"])
        m.close()


# ------------------------------------------------------------------------------------------ MoE vs oracle
def _synth(t, n, seed):
    return synth_blocks(t, n, device="cuda", seed=seed)


COMBOS = [
    (Q4_K, Q4_K, Q6_K, 8, 4, 1024, 512), (Q4_K, Q4_K, Q4_K, 8, 4, 1024, 512), (Q6_K, Q6_K, Q6_K, 4, 2, 512, 256),
    (Q5_K, Q5_K, Q5_K, 4, 2, 512, 512), (Q2_K, Q2_K, Q3_K, 4, 2, 512, 256), (IQ4_XS, IQ4_XS, IQ4_XS, 4, 2, 256, 256),
    (Q4_K, Q5_K, Q6_K, 4, 3, 768, 256), (Q3_K, Q3_K, Q2_K, 4, 2, 256, 512), (Q4_K, Q4_K, Q6_K, 6, 6, 2048, 1536),
    # shapes that take the bulk-copy kernels (gemv_bulk.cuh): >= 16 blocks per gate/up row (16 / 40 / 32 lanes-worth),
    # down items of 8, 32 and 64 (row, block) pairs, Q4_K down
    (Q4_K, Q4_K, Q6_K, 4, 3, 4096, 512), (Q4_K, Q4_K, Q4_K, 3, 2, 10240, 256), (Q4_K, Q4_K, Q6_K, 3, 2, 512, 4096),
    (Q4_K, Q4_K, Q6_K, 4, 2, 4096, 2048), (Q4_K, Q4_K, Q4_K, 2, 2, 8192, 256),
]


@pytest.mark.parametrize("gt,ut,dt,E,k,H,I", COMBOS)
@pytest.mark.parametrize("hid", [F32, BF16])
def test_moe_forward_vs_oracle(oracle, gt, ut, dt, E, k, H, I, hid):
    gate, up, down = _synth(gt, E * I * H, 1), _synth(ut, E * I * H, 2), _synth(dt, E * H * I, 3)
    g_np, u_np, d_np = gate.cpu().numpy(), up.cpu().numpy(), down.cpu().numpy()   # copies BEFORE the in-place repack
    m = G.Moe(E, k, H, I, gate, up, down, gt, ut, dt, hid)
    rng = np.random.default_rng(E * 1000 + H)
    for qlen in (1, 2, 9, 33):
        x = (rng.standard_normal((qlen, H)) / 100).astype(np.float32)
        ids = np.stack([rng.permutation(E)[:k] for _ in range(qlen)]).astype(np.int64)
        w = rng.random((qlen, k)).astype(np.float32)
        xin = x if hid == F32 else f32_to_bf16_bits(x)
        got = m.forward(ids, w, xin)
        want = oracle.moe_forward(E, H, I, g_np, u_np, d_np, gt, ut, dt, hid, ids, w, xin)
        if hid == F32:
            assert relmax(got, want) < FP_TOL, f"{TYPE_NAMES[gt]}/{TYPE_NAMES[ut]}/{TYPE_NAMES[dt]} qlen={qlen}"
        else:
            assert_bf16_close(got, want)
    m.close()


@pytest.mark.parametrize("H,I", [(512, 256), (4096, 512)])   # register-staged kernels / bulk-copy kernels
def test_moe_edge_cases(oracle, H, I):
    E, k = 8, 4
    gate, up, down = _synth(Q4_K, E * I * H, 11), _synth(Q4_K, E * I * H, 12), _synth(Q6_K, E * H * I, 13)
    g_np, u_np, d_np = gate.cpu().numpy(), up.cpu().numpy(), down.cpu().numpy()
    m = G.Moe(E, k, H, I, gate, up, down, Q4_K, Q4_K, Q6_K, F32, max_tokens=16)
    rng = np.random.default_rng(5)
    x = (rng.standard_normal((6, H)) / 50).astype(np.float32)
    w = rng.random((6, k)).astype(np.float32)
    # ids < 0 or >= E are skipped (kt-kernel/operators/common.hpp:255-258); duplicates are legal
    ids = np.array([[0, 1, 2, 3], [-1, 7, 7, 2], [8, 100, 3, 3], [-5, -1, 9, 1 << 40], [5, 4, 3, 2], [1, 1, 1, 1]], np.int64)
    got = m.forward(ids, w, x)
    want = oracle.moe_forward(E, H, I, g_np, u_np, d_np, Q4_K, Q4_K, Q6_K, F32, ids, w, x)
    assert relmax(got, want) < FP_TOL
    assert not got[3].any()                                   # every expert of token 3 is invalid -> zeros
    # k smaller than routed_expert_num
    got2 = m.forward(ids[:, :2], w[:, :2], x)
    assert relmax(got2, oracle.moe_forward(E, H, I, g_np, u_np, d_np, Q4_K, Q4_K, Q6_K, F32, ids[:, :2], w[:, :2], x)) < FP_TOL
    # device-side batch size: rows >= bsz untouched
    sentinel = torch.full((6, H), 7.0, device="cuda")
    got3 = m.forward(ids, w, x, bsz=2, out=sentinel)
    assert np.array_equal(got3[:2], got[:2]) and (got3[2:] == 7.0).all()
    # error behaviour mirrors the reference's exceptions
    with pytest.raises(ValueError):
        m.forward(np.zeros((17, k), np.int64), np.zeros((17, k), np.float32), np.zeros((17, H), np.float32))   # qlen > group_max_len
    with pytest.raises(ValueError):
        m.forward(np.zeros((1, k + 1), np.int64), np.zeros((1, k + 1), np.float32), x[:1])                     # k > routed_expert_num
    with pytest.raises(ValueError):
        G.Moe(E, k, H, I, gate, up, down, 2, Q4_K, Q6_K, F32)                                               # Q4_0: unsupported ggml type
    with pytest.raises(ValueError):
        G.Moe(E, k, 500, I, gate, up, down, Q4_K, Q4_K, Q6_K, F32)                                          # H not a multiple of 256
    m.close()


@pytest.mark.parametrize("H", [512, 4096])
def test_moe_expert_parallel_shards_sum_to_full(H):
    E, k, I = 8, 4, 512
    gate, up, down = _synth(Q4_K, E * I * H, 21), _synth(Q4_K, E * I * H, 22), _synth(Q6_K, E * H * I, 23)
    gbytes, dbytes = gate.numel() // E, down.numel() // E
    rng = np.random.default_rng(9)
    x = (rng.standard_normal((5, H)) / 50).astype(np.float32)
    ids = np.stack([rng.permutation(E)[:k] for _ in range(5)]).astype(np.int64)
    w = rng.random((5, k)).astype(np.float32)
    full = G.Moe(E, k, H, I, gate.clone(), up.clone(), down.clone(), Q4_K, Q4_K, Q6_K, F32).forward(ids, w, x)
    acc = np.zeros_like(full)
    for r in range(2):
        sl = slice(r * (E // 2), (r + 1) * (E // 2))
        sh = G.Moe(E // 2, k, H, I, gate[sl.start * gbytes: sl.stop * gbytes].clone(), up[sl.start * gbytes: sl.stop * gbytes].clone(),
                   down[sl.start * dbytes: sl.stop * dbytes].clone(), Q4_K, Q4_K, Q6_K, F32, offset=sl.start)
        acc += sh.forward(ids, w, x)
    assert relmax(acc, full) < 1e-5


@pytest.mark.parametrize("H", [1024, 4096])
@pytest.mark.parametrize("sgt,sdt,fused", [(Q4_K, Q6_K, True), (Q5_K, Q4_K, False)])
def test_moe_with_shared_expert_matches_two_rounded_terms(oracle, sgt, sdt, fused, H):
    """KDeepseekV3MoE: y = experts(x); y += shared_experts(x) on bf16 tensors — each term rounded, then the sum.
    Same quant types as the routed experts -> the shared expert is an extra slot inside the two routed launches;
    different types -> it runs as a separate MLP.  Both must give the reference's two-rounding result."""
    E, k, I = 8, 4, 512
    gate, up, down = _synth(Q4_K, E * I * H, 71), _synth(Q4_K, E * I * H, 72), _synth(Q6_K, E * H * I, 73)
    sg, su, sd = _synth(sgt, I * H, 74), _synth(sgt, I * H, 75), _synth(sdt, H * I, 76)
    g_np, u_np, d_np, sg_np, su_np, sd_np = (t.cpu().numpy() for t in (gate, up, down, sg, su, sd))
    m = G.Moe(E, k, H, I, gate, up, down, Q4_K, Q4_K, Q6_K, BF16)
    mlp = G.Mlp(H, I, sg, su, sd, sgt, sgt, sdt, BF16)
    rng = np.random.default_rng(17)
    for qlen in (1, 5):
        x = f32_to_bf16_bits((rng.standard_normal((qlen, H)) / 100).astype(np.float32))
        ids = np.stack([rng.permutation(E)[:k] for _ in range(qlen)]).astype(np.int64)
        w = rng.random((qlen, k)).astype(np.float32)
        n0 = native.launch_count()
        got = G.moe_forward_shared(m, mlp, ids, w, x)
        assert native.launch_count() - n0 == (2 if fused else 4)
        routed = oracle.moe_forward(E, H, I, g_np, u_np, d_np, Q4_K, Q4_K, Q6_K, BF16, ids, w, x)
        shared = oracle.mlp_forward(H, I, sg_np, su_np, sd_np, sgt, sgt, sdt, BF16, x)
        want = (torch.from_numpy(routed.view(np.int16)).view(torch.bfloat16) + torch.from_numpy(shared.view(np.int16)).view(torch.bfloat16))
        assert_bf16_close(got, want.view(torch.int16).numpy().view(np.uint16))
        assert np.array_equal(G.moe_forward_shared(m, None, ids, w, x), m.forward(ids, w, x))
    m.close(); mlp.close()


def test_moe_with_shared_expert_prefill_sized_batch(oracle):
    """ktb200_moe_forward_shared at 60 tokens: the routed experts take the grouped tensor-core path, the shared expert follows as a
    separate MLP that accumulates in bf16 — the same two rounded terms."""
    E, k, H, I, qlen = 8, 4, 1024, 512, 60
    gate, up, down = _synth(Q4_K, E * I * H, 81), _synth(Q4_K, E * I * H, 82), _synth(Q6_K, E * H * I, 83)
    sg, su, sd = _synth(Q4_K, I * H, 84), _synth(Q4_K, I * H, 85), _synth(Q6_K, H * I, 86)
    g_np, u_np, d_np, sg_np, su_np, sd_np = (t.cpu().numpy() for t in (gate, up, down, sg, su, sd))
    m = G.Moe(E, k, H, I, gate, up, down, Q4_K, Q4_K, Q6_K, BF16)
    mlp = G.Mlp(H, I, sg, su, sd, Q4_K, Q4_K, Q6_K, BF16)
    rng = np.random.default_rng(23)
    x = f32_to_bf16_bits((rng.standard_normal((qlen, H)) / 100).astype(np.float32))
    ids = np.stack([rng.permutation(E)[:k] for _ in range(qlen)]).astype(np.int64)
    w = rng.random((qlen, k)).astype(np.float32)
    n0 = native.launch_count()
    got = G.moe_forward_shared(m, mlp, ids, w, x)
    assert native.launch_count() - n0 >= 12          # 10 grouped launches + the shared MLP's
    routed = oracle.moe_forward(E, H, I, g_np, u_np, d_np, Q4_K, Q4_K, Q6_K, BF16, ids, w, x)
    shared = oracle.mlp_forward(H, I, sg_np, su_np, sd_np, Q4_K, Q4_K, Q6_K, BF16, x)
    want = (torch.from_numpy(routed.view(np.int16)).view(torch.bfloat16) + torch.from_numpy(shared.view(np.int16)).view(torch.bfloat16))
    assert_bf16_close(got, want.view(torch.int16).numpy().view(np.uint16))
    m.close(); mlp.close()


# ------------------------------------------------------------------------------------------ linear / mlp
def test_linear_and_mlp_vs_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "linear_mlp.npz"))
    H, I, O = int(g["H"]), int(g["I"]), int(g["O"])
    assert relmax(G.linear_forward(H, O, g["wl"], Q4_K, F32, g["x"]), g["lin_f32"]) < FP_TOL
    assert relmax(G.linear_forward(H, O, g["wl6"], Q6_K, F32, g["x"]), g["lin6_f32"]) < FP_TOL
    assert relmax(G.mlp_forward(H, I, g["g"], g["u"], g["d"], Q4_K, Q4_K, Q6_K, F32, g["x"]), g["mlp_f32"]) < FP_TOL
    assert_bf16_close(G.linear_forward(H, O, g["wl"], Q4_K, BF16, f32_to_bf16_bits(g["x"])), g["lin_bf16"])
    assert_bf16_close(G.mlp_forward(H, I, g["g"], g["u"], g["d"], Q4_K, Q4_K, Q6_K, BF16, f32_to_bf16_bits(g["x"])), g["mlp_bf16"])


@pytest.mark.parametrize("t,in_f,out_f", [(Q4_K, 7168, 1536), (Q6_K, 2048, 7168), (Q5_K, 1536, 512), (Q6_K, 512, 100), (Q3_K, 256, 64),
                                           # the dense segment-ring kernel (dense_bulk.cuh): 5 rows per segment with a ragged tail,
                                           # two and three segments per row, one block per row
                                           (Q4_K, 1536, 2048 + 3), (Q4_K, 16384, 512), (Q4_K, 18432, 256), (Q4_K, 256, 777), (Q4_K, 7168, 2112)])
def test_linear_vs_oracle(oracle, t, in_f, out_f):
    w = _synth(t, out_f * in_f, 31)
    w_np = w.cpu().numpy()
    rng = np.random.default_rng(in_f)
    x = (rng.standard_normal((3, in_f)) / 10).astype(np.float32)
    bias = rng.standard_normal(out_f).astype(np.float32)
    want = oracle.linear_forward(in_f, out_f, w_np, t, F32, x)
    assert relmax(G.linear_forward(in_f, out_f, w.clone(), t, F32, x), want) < FP_TOL
    assert relmax(G.linear_forward(in_f, out_f, w.clone(), t, F32, x, bias=bias), want + bias) < FP_TOL


def test_mlp_accumulate_matches_torch_bf16_add(oracle):
    H, I = 512, 256
    g, u, d = _synth(Q4_K, I * H, 41), _synth(Q4_K, I * H, 42), _synth(Q6_K, H * I, 43)
    g_np, u_np, d_np = g.cpu().numpy(), u.cpu().numpy(), d.cpu().numpy()
    rng = np.random.default_rng(3)
    x = f32_to_bf16_bits((rng.standard_normal((4, H)) / 10).astype(np.float32))
    y = f32_to_bf16_bits(rng.standard_normal((4, H)).astype(np.float32))
    shared = oracle.mlp_forward(H, I, g_np, u_np, d_np, Q4_K, Q4_K, Q6_K, BF16, x)
    want = (torch.from_numpy(y.view(np.int16)).view(torch.bfloat16) + torch.from_numpy(shared.view(np.int16)).view(torch.bfloat16))
    got = G.mlp_forward(H, I, g, u, d, Q4_K, Q4_K, Q6_K, BF16, x, accumulate_into=y)
    assert_bf16_close(got, want.view(torch.int16).numpy().view(np.uint16))


# ------------------------------------------------------------------------------------------ router
def test_gate_vs_golden_reference_torch(golden_dir):
    g = np.load(os.path.join(golden_dir, "gate_v3_small.npz"))
    idx, w, logits = G.gate_forward(g["x"], g["W"], g["bias"], 6, 8, 4, want_logits=True)
    _, _, margin, _ = gate_oracle.route(g["x"], g["W"], g["bias"], top_k=6, n_group=8, topk_group=4, routed_scaling_factor=2.5, dtype=np.float64)
    ok = margin > 1e-5
    print(f"knife-edge tokens excluded (relative margin < 1e-5 in float64): {int((~ok).sum())} of {ok.size}")
    assert (~ok).sum() <= 1
    assert np.array_equal(np.sort(idx[ok], axis=1), np.sort(g["idx"][ok], axis=1))        # bit-exact routed ids
    np.testing.assert_allclose(logits, g["logits64"], rtol=0, atol=1e-4)
    for t in np.nonzero(ok)[0]:
        ref_w = dict(zip(g["idx"][t].tolist(), g["w"][t].tolist()))
        for e, wv in zip(idx[t].tolist(), w[t].tolist()):
            assert abs(ref_w[e] - wv) < 1e-5 * max(1.0, abs(wv))


@pytest.mark.parametrize("E,H,k,ng,tg,scoring,method,norm,scale", [
    (256, 7168, 8, 8, 4, 0, 0, 1, 2.5),     # DeepSeek-V3 (kt-kernel/examples/test_gate.py shapes)
    (384, 7168, 8, 1, 1, 0, 0, 1, 2.827),   # Kimi-K2
    (64, 2048, 6, 1, 1, 1, 1, 0, 1.0),      # V2-Lite: softmax greedy
    (160, 5120, 6, 8, 3, 1, 2, 0, 16.0),    # V2: softmax group_limited_greedy
])
def test_gate_vs_oracle_full_shapes(E, H, k, ng, tg, scoring, method, norm, scale):
    rng = np.random.default_rng(42)
    T = 64
    W = rng.standard_normal((E, H)).astype(np.float32)
    bias = rng.standard_normal(E).astype(np.float32) if method == 0 else None
    x = (rng.standard_normal((T, H)) / 10).astype(np.float32)
    kw = dict(top_k=k, n_group=ng, topk_group=tg, scoring=["sigmoid", "softmax"][scoring],
              topk_method=["noaux_tc", "greedy", "group_limited_greedy"][method], norm_topk_prob=bool(norm), routed_scaling_factor=scale)
    idx, w, _ = G.gate_forward(x, W, bias, k, ng, tg, scoring, method, norm, scale)
    oidx, ow, margin, _ = gate_oracle.route(x, W, bias, dtype=np.float64, **kw)
    ok = margin > 1e-5
    print(f"knife-edge tokens excluded (relative margin < 1e-5 in float64): {int((~ok).sum())} of {ok.size}")
    assert (~ok).sum() <= 1      # a real tie needs two of ~256 fp32 scores within 1e-5: at most one of these 64 tokens
    assert np.array_equal(np.sort(idx[ok], axis=1), np.sort(oidx[ok], axis=1))
    for t in np.nonzero(ok)[0]:
        ref_w = dict(zip(oidx[t].tolist(), ow[t].tolist()))
        for e, wv in zip(idx[t].tolist(), w[t].tolist()):
            assert abs(ref_w[e] - wv) < 2e-5 * max(1.0, abs(wv))
    # bf16 activations take the same path
    idx_b, _, _ = G.gate_forward(f32_to_bf16_bits(x), W, bias, k, ng, tg, scoring, method, norm, scale, hidden_type=BF16)
    assert idx_b.shape == idx.shape and (idx_b >= 0).all() and (idx_b < E).all()


def test_gate_reference_recipe_seed42_no_exclusions(golden_dir):
    """kt-kernel/examples/test_gate.py: seed 42, W = randn(256, 7168), bias = randn(256), input = randn(64, 7168);
    expert ids must match the reference's torch MoEGate EXACTLY for every token (:214), weights < 1e-2 (:215).
    Expected values: tests/golden/gate_seed42.npz (reference source executed on CPU by make_gate_seed42.py)."""
    g = np.load(os.path.join(golden_dir, "gate_seed42.npz"))
    torch.manual_seed(42)
    W = torch.randn((256, 7168), dtype=torch.float32)
    bias = torch.randn((256,), dtype=torch.float32)
    x = torch.randn(64, 7168, dtype=torch.float32)
    probe = np.array([W[0, 0], W[255, 7167], bias[7], x[0, 0], x[63, 7167]], np.float32)
    if not np.array_equal(probe, g["probe"]):
        pytest.skip("torch CPU RNG stream differs from the one the fixture was minted with")
    idx, w, _ = G.gate_forward(x.numpy(), W.numpy(), bias.numpy(), 8, 8, 4)
    assert np.array_equal(np.sort(idx, axis=1), np.sort(g["idx"], axis=1))
    order_g, order_r = np.argsort(idx, axis=1), np.argsort(g["idx"], axis=1)
    assert np.abs(np.take_along_axis(w, order_g, 1) - np.take_along_axis(g["w"], order_r, 1)).max() < 1e-5


def test_moe_forward_ep_shard_call_matches_the_separate_calls():
    """ktb200_moe_forward_ep: routed partial sums of an expert-parallel shard (fp32) + the shared expert of ONE token in the
    same two launches == ktb200_moe_forward on the shard + ktb200_mlp_forward on that token, bit for bit."""
    import ctypes as C
    Eg, k, H, I, offset = 16, 4, 4096, 512, 8
    El = Eg - offset
    m = G.Moe(El, k, H, I, _synth(Q4_K, El * I * H, 91), _synth(Q4_K, El * I * H, 92), _synth(Q6_K, El * H * I, 93), Q4_K, Q4_K, Q6_K, F32, offset=offset)
    sg, su, sd = _synth(Q4_K, I * H, 94), _synth(Q4_K, I * H, 95), _synth(Q6_K, H * I, 96)
    mlp = G.Mlp(H, I, sg, su, sd, Q4_K, Q4_K, Q6_K, BF16)
    rng = np.random.default_rng(3)
    lib = native.lib()
    for qlen, own in ((1, 0), (3, 1), (8, 7)):
        xb = f32_to_bf16_bits((rng.standard_normal((qlen, H)) / 10).astype(np.float32))
        x = bf16_to_f32(xb)                                              # the shard's kernels take the gathered rows as fp32
        ids = np.stack([rng.permutation(Eg)[:k] for _ in range(qlen)]).astype(np.int64)
        w = rng.random((qlen, k)).astype(np.float32)
        want = m.forward(ids, w, x)
        x_d, ids_d, w_d = G.dev(x), G.dev(ids), G.dev(w)
        part = torch.zeros((qlen, H), dtype=torch.float32, device="cuda")
        sh_out = torch.zeros((H,), dtype=torch.bfloat16, device="cuda")
        n0 = native.launch_count()
        native.check(lib.ktb200_moe_forward_ep(m.h, mlp.h, qlen, k, ids_d.data_ptr(), w_d.data_ptr(), x_d.data_ptr(), part.data_ptr(), own,
                                               sh_out.data_ptr(), None, G.stream()))
        torch.cuda.synchronize()
        assert native.launch_count() - n0 == 2
        assert np.array_equal(part.cpu().numpy(), want)
        sh_want = torch.zeros((1, H), dtype=torch.bfloat16, device="cuda")
        xo = G.dev(xb[own:own + 1], torch.bfloat16)
        native.check(lib.ktb200_mlp_forward(mlp.h, 1, xo.data_ptr(), sh_want.data_ptr(), 0, None, G.stream()))
        torch.cuda.synchronize()
        assert torch.equal(sh_out.view(torch.int16), sh_want[0].view(torch.int16))
    m.close(); mlp.close()


# ------------------------------------------------------------------------------------------ fused MoE block
@pytest.mark.parametrize("dt,hid,shared,offset,H,I", [
    (Q6_K, BF16, True, 0, 4096, 512),      # V3-like: Q4_K gate/up, Q6_K (tile layout) down, shared expert fused as slot k
    (Q6_K, F32, False, 0, 4096, 2048),     # no shared expert; 4 rows x 8 blocks down tiles
    (Q4_K, BF16, True, 0, 8192, 512),      # Q4_K down, 32 blocks per gate/up row
    (Q6_K, BF16, True, 8, 4096, 512),      # expert-parallel shard: owns ids 8..15 of 16, everything else is skipped
    (Q6_K, BF16, True, 0, 1024, 512),      # rows too short for the persistent kernel -> separate launches behind the same call
])
def test_moe_block_single_launch_is_bit_identical_to_separate_launches(dt, hid, shared, offset, H, I):
    """ktb200_moe_block_forward (router + experts + shared expert in ONE cooperative launch) must give exactly the bits
    of ktb200_moe_gate_forward followed by ktb200_moe_forward_shared — which are the calls checked against the oracle."""
    Eg, k, ng, tg = 16, 4, 4, 2
    El = Eg - offset if offset else Eg
    gate_w, up_w, down_w = _synth(Q4_K, El * I * H, 81), _synth(Q4_K, El * I * H, 82), _synth(dt, El * H * I, 83)
    m = G.Moe(El, k, H, I, gate_w, up_w, down_w, Q4_K, Q4_K, dt, hid, offset=offset)
    mlp = G.Mlp(H, I, _synth(Q4_K, I * H, 84), _synth(Q4_K, I * H, 85), _synth(dt, H * I, 86), Q4_K, Q4_K, dt, hid) if shared else None
    rng = np.random.default_rng(H + I)
    W = rng.standard_normal((Eg, H)).astype(np.float32)
    bias = rng.standard_normal(Eg).astype(np.float32)
    gate = G.Gate(W, bias, k, ng, tg, hidden_type=hid)
    for qlen in (1, 3, 8, 9):      # 9 > 8 tokens: the call falls back to the separate launches
        x = (rng.standard_normal((qlen, H)) / 10).astype(np.float32)
        xin = x if hid == F32 else f32_to_bf16_bits(x)
        n0 = native.launch_count()
        out, idx, w = G.moe_block_forward(gate, m, mlp, xin)
        fused = native.launch_count() - n0 == 1
        assert fused == (H >= 4096 and qlen <= 8)
        ridx, rw, _ = G.gate_forward(xin, W, bias, k, ng, tg, hidden_type=hid)
        assert np.array_equal(idx, ridx) and np.array_equal(w, rw)
        want = G.moe_forward_shared(m, mlp, ridx, rw, xin)
        assert np.array_equal(out, want), f"qlen={qlen}"
        if offset:
            assert ((ridx < offset).any(axis=1)).any()          # some slots really are skipped in this case
    # the barrier words reset themselves: repeated launches and CUDA-graph replays give the same bits
    x = f32_to_bf16_bits((rng.standard_normal((2, H)) / 10).astype(np.float32)) if hid == BF16 else (rng.standard_normal((2, H)) / 10).astype(np.float32)
    once = G.moe_block_forward(gate, m, mlp, x)
    again = G.moe_block_forward(gate, m, mlp, x, repeats=5)
    replay = G.moe_block_forward(gate, m, mlp, x, repeats=4, graph=True)
    for a, b, c in zip(once, again, replay):
        assert np.array_equal(a, b) and np.array_equal(a, c)
    m.close()
    if mlp is not None:
        mlp.close()


@pytest.mark.parametrize("name,E,H,I,k,ng,tg,scale", [
    ("DeepSeek-V3", 256, 7168, 2048, 8, 8, 4, 2.5),       # the configuration bench.py times: 28 blocks/row, 6 router splits
    ("Kimi-K2", 384, 7168, 2048, 8, 1, 1, 2.827),
    ("H5120", 64, 5120, 1536, 6, 8, 3, 1.0),              # 20 blocks/row, I not a multiple of the CTA count
])
def test_moe_block_full_shape_vs_oracle(oracle, name, E, H, I, k, ng, tg, scale):
    """The ONE-launch MoE block (ktb200_moe_block_forward: router + top-k + routed experts + shared expert) at the full
    shapes bench.py times, against the CPU oracle: ids vs the numpy router restatement (float64 margins), output vs
    oracle.moe_forward + oracle.mlp_forward as two separately rounded bf16 terms (experts.py:984-1011)."""
    gate_w, up_w, down_w = _synth(Q4_K, E * I * H, 301), _synth(Q4_K, E * I * H, 302), _synth(Q6_K, E * H * I, 303)
    sg, su, sd = _synth(Q4_K, I * H, 304), _synth(Q4_K, I * H, 305), _synth(Q6_K, H * I, 306)
    down_raw = down_w.clone()                                  # load_weights re-tiles Q6_K in place
    sg_np, su_np, sd_np = sg.cpu().numpy(), su.cpu().numpy(), sd.cpu().numpy()
    gb, db = gate_w.numel() // E, down_w.numel() // E
    m = G.Moe(E, k, H, I, gate_w, up_w, down_w, Q4_K, Q4_K, Q6_K, BF16, max_tokens=8)
    mlp = G.Mlp(H, I, sg, su, sd, Q4_K, Q4_K, Q6_K, BF16)
    rng = np.random.default_rng(E + H)
    W = rng.standard_normal((E, H)).astype(np.float32)
    bias = rng.standard_normal(E).astype(np.float32)
    gate = G.Gate(W, bias, k, ng, tg, scale=scale, hidden_type=BF16)
    for qlen in (1, 8):
        xb = f32_to_bf16_bits((rng.standard_normal((qlen, H)) / 100).astype(np.float32))
        n0 = native.launch_count()
        out, idx, w = G.moe_block_forward(gate, m, mlp, xb)
        assert native.launch_count() - n0 == 1, "the persistent single-launch kernel must take this configuration"
        # routing: exact ids wherever the decision is not a float64 knife edge
        oidx, ow, margin, _ = gate_oracle.route(bf16_to_f32(xb), W, bias, top_k=k, n_group=ng, topk_group=tg, routed_scaling_factor=scale, dtype=np.float64)
        ok = margin > 1e-5
        print(f"{name} qlen={qlen}: knife-edge tokens excluded {int((~ok).sum())} of {qlen}")
        assert (~ok).sum() <= 1 and ok.any()
        assert np.array_equal(np.sort(idx[ok], axis=1), np.sort(oidx[ok], axis=1))
        for t in np.nonzero(ok)[0]:
            ref_w = dict(zip(oidx[t].tolist(), ow[t].tolist()))
            for e, wv in zip(idx[t].tolist(), w[t].tolist()):
                assert abs(ref_w[e] - wv) < 2e-5 * max(1.0, abs(wv))
        # experts: the oracle on the selected experts only (remapped to 0..n-1), with the routing the kernel produced
        sel = sorted(set(idx.reshape(-1).tolist()))
        remap = {e: i for i, e in enumerate(sel)}
        g_np = torch.cat([gate_w[e * gb:(e + 1) * gb] for e in sel]).cpu().numpy()
        u_np = torch.cat([up_w[e * gb:(e + 1) * gb] for e in sel]).cpu().numpy()
        d_np = torch.cat([down_raw[e * db:(e + 1) * db] for e in sel]).cpu().numpy()
        ids_l = np.vectorize(remap.get)(idx).astype(np.int64)
        routed = oracle.moe_forward(len(sel), H, I, g_np, u_np, d_np, Q4_K, Q4_K, Q6_K, BF16, ids_l, w, xb)
        shared = oracle.mlp_forward(H, I, sg_np, su_np, sd_np, Q4_K, Q4_K, Q6_K, BF16, xb)
        want = (torch.from_numpy(routed.view(np.int16)).view(torch.bfloat16) + torch.from_numpy(shared.view(np.int16)).view(torch.bfloat16))
        # y = round(routed) + round(shared), rounded again: the error budget is one bf16 ulp of EACH term (the terms may cancel)
        a, b = bf16_to_f32(out), bf16_to_f32(want.view(torch.int16).numpy().view(np.uint16))
        tol = 2.0 ** -7 * (np.abs(bf16_to_f32(routed)) + np.abs(bf16_to_f32(shared)) + np.abs(b)) + FP_TOL * np.abs(b).max()
        assert (np.abs(a - b) <= tol).all(), float((np.abs(a - b) / tol).max())
        assert (a == b).mean() > 0.9
    m.close(); mlp.close()


# ------------------------------------------------------------------------------------------ expert-parallel block
@pytest.mark.parametrize("world,shared", [(1, True), (2, True), (4, True), (8, False)])
def test_moe_ep_block_loopback_matches_single_gpu(world, shared):
    """ktb200_moe_ep_block_forward — the one-launch expert-parallel layer — emulated on ONE GPU: `world` shard handles
    (experts E/world each) with their own message / partial / flag buffers in the same device memory; the three phases
    (route+send, experts+deliver, combine) run as separate launches rank by rank, which is a legal schedule of the
    real concurrent execution.  Every rank's token must come out as the single-GPU block (ktb200_moe_block_forward
    over all E experts) computes it: same routing bits, output within fp32 re-association of the partial sums."""
    import ctypes as C
    E, k, H, I, ng, tg = 32, 4, 4096, 512, 4, 2
    El = E // world
    lib = native.lib()
    gate_w, up_w, down_w = _synth(Q4_K, E * I * H, 401), _synth(Q4_K, E * I * H, 402), _synth(Q6_K, E * H * I, 403)
    sgs = (_synth(Q4_K, I * H, 404), _synth(Q4_K, I * H, 405), _synth(Q6_K, H * I, 406))
    gb, db = gate_w.numel() // E, down_w.numel() // E
    rng = np.random.default_rng(world)
    Wr = rng.standard_normal((E, H)).astype(np.float32)
    bias = rng.standard_normal(E).astype(np.float32)
    gate = G.Gate(Wr, bias, k, ng, tg, hidden_type=BF16)
    full = G.Moe(E, k, H, I, gate_w.clone(), up_w.clone(), down_w.clone(), Q4_K, Q4_K, Q6_K, BF16, max_tokens=8)
    full_mlp = G.Mlp(H, I, *(t.clone() for t in sgs), Q4_K, Q4_K, Q6_K, BF16) if shared else None
    shards, mlps = [], []
    for r in range(world):
        sl = slice(r * El, (r + 1) * El)
        shards.append(G.Moe(El, k, H, I, gate_w[sl.start * gb: sl.stop * gb].clone(), up_w[sl.start * gb: sl.stop * gb].clone(),
                            down_w[sl.start * db: sl.stop * db].clone(), Q4_K, Q4_K, Q6_K, BF16, max_tokens=8, offset=sl.start))
        mlps.append(G.Mlp(H, I, *(t.clone() for t in sgs), Q4_K, Q4_K, Q6_K, BF16) if shared else None)
    msgb = lib.ktb200_ep_msg_bytes(H, BF16)
    msg = [torch.zeros(world * msgb, dtype=torch.uint8, device="cuda") for _ in range(world)]
    part = [torch.zeros((world, H), dtype=torch.float32, device="cuda") for _ in range(world)]
    flags = [torch.zeros(2 * world + 2, dtype=torch.int32, device="cuda") for _ in range(world)]
    comms = [native.EpComm.make(r, world, H, BF16, [t.data_ptr() for t in msg], [t.data_ptr() for t in part], [t.data_ptr() for t in flags])
             for r in range(world)]
    for layer in range(3):                                   # epochs advance; buffers are reused
        xs = [f32_to_bf16_bits((rng.standard_normal((1, H)) / 10).astype(np.float32)) for _ in range(world)]
        x_d = [G.dev(x, torch.bfloat16) for x in xs]
        y = [torch.zeros((1, H), dtype=torch.bfloat16, device="cuda") for _ in range(world)]
        idx = [torch.zeros((1, k), dtype=torch.int64, device="cuda") for _ in range(world)]
        w = [torch.zeros((1, k), dtype=torch.float32, device="cuda") for _ in range(world)]
        n0 = native.launch_count()
        masks = (7,) if world == 1 else (1, 2, 4)
        for mask in masks:
            for r in range(world):
                native.check(lib.ktb200_moe_ep_block_forward(C.byref(gate.cfg), shards[r].h, mlps[r].h if shared else None, C.byref(comms[r]),
                                                             x_d[r].data_ptr(), y[r].data_ptr(), idx[r].data_ptr(), w[r].data_ptr(), mask, G.stream()))
        torch.cuda.synchronize()
        assert native.launch_count() - n0 == len(masks) * world
        for r in range(world):
            assert int(flags[r][2 * world + 1]) == 0, "a peer wait timed out"
            want, widx, ww = G.moe_block_forward(gate, full, full_mlp, xs[r])
            assert np.array_equal(idx[r].cpu().numpy(), widx) and np.array_equal(w[r].cpu().numpy(), ww)
            got = y[r].cpu().view(torch.int16).numpy().view(np.uint16)
            if world == 1:
                assert np.array_equal(got, want)                # one rank: the same FMA chain, bit for bit
            else:
                assert_bf16_close(got, want, min_exact=0.9, ulps=2)
    for h in shards + [full] + [m_ for m_ in mlps + [full_mlp] if m_ is not None]:
        h.close()


# ------------------------------------------------------------------------------------------ MLA decode
def _mla_case(rng, B, Hq, page_size, lens, shuffle_pages=True):
    from oracle.mla_oracle import bf16_round
    max_pages = max((l + page_size - 1) // page_size for l in lens)
    n_pages = B * max_pages + 3
    kv = bf16_round(rng.standard_normal((n_pages, page_size, 576)).astype(np.float32))
    perm = rng.permutation(n_pages) if shuffle_pages else np.arange(n_pages)
    page_table = perm[: B * max_pages].reshape(B, max_pages).astype(np.int32)
    q_nope = bf16_round((rng.standard_normal((B, Hq, 512)) * 0.5).astype(np.float32))
    q_pe = bf16_round((rng.standard_normal((B, Hq, 64)) * 0.5).astype(np.float32))
    return q_nope, q_pe, kv, page_table, np.array(lens, np.int32)


@pytest.mark.parametrize("B,Hq,page_size,lens,splits", [
    (1, 128, 64, [1], 0), (1, 128, 64, [33], 0), (1, 128, 64, [1000], 0), (1, 128, 64, [4096], 0),
    (3, 128, 64, [17, 640, 2049], 0), (2, 16, 32, [95, 128], 0), (1, 128, 256, [777], 3), (2, 40, 64, [64, 65], 1),
])
def test_mla_decode_vs_oracle(B, Hq, page_size, lens, splits):
    from oracle import mla_oracle
    rng = np.random.default_rng(sum(lens) + Hq)
    q_nope, q_pe, kv, pt, kl = _mla_case(rng, B, Hq, page_size, lens)
    scale = (128 + 64) ** -0.5
    out, lse = G.mla_decode(q_nope, q_pe, kv, pt, kl, scale, num_kv_splits=splits)
    want, want_lse = mla_oracle.mla_decode(q_nope, q_pe, kv, pt, kl, scale, p_bf16=True)
    exact, _ = mla_oracle.mla_decode(q_nope, q_pe, kv, pt, kl, scale, p_bf16=False)
    ref_mag = np.abs(exact).max()
    # vs the bf16-P restatement: bf16 output rounding + fp32 accumulation order only
    assert np.abs(out - want).max() <= 2.0 ** -7 * ref_mag + 1e-3 * ref_mag
    # vs exact softmax attention: bf16 P noise (reference's own bound is 1e-1 max / 2e-1 rel-mean, test_mla_qlen.py:345)
    assert np.abs(out - exact).max() <= 2e-2 * ref_mag
    assert np.abs(out - exact).mean() <= 5e-3 * np.abs(exact).mean() + 1e-6
    np.testing.assert_allclose(lse, want_lse, rtol=0, atol=2e-3)


@pytest.mark.parametrize("name", ["a", "b", "c"])
def test_mla_decode_vs_reference_golden(golden_dir, name):
    """ktb200_mla_decode against outputs of the reference's attention_ref_torch (tests/golden/mla_ref.npz)."""
    g = np.load(os.path.join(golden_dir, "mla_ref.npz"))
    f = lambda k: bf16_to_f32(g[f"{name}_{k}"])
    q_nope, q_pe, kv, scale, want, lse2 = f("q_nope"), f("q_pe"), f("kv"), float(g[f"{name}_scale"]), f("out"), g[f"{name}_lse2"]
    B, L = kv.shape[0], kv.shape[1]
    for page in (32, 64):
        npg = (L + page - 1) // page
        rng = np.random.default_rng(page)
        cache = np.full((B * npg + 2, page, 576), np.nan, np.float32)      # unwritten cache rows are NaN: they must not leak
        table = rng.permutation(B * npg + 2)[: B * npg].reshape(B, npg).astype(np.int32)
        for b in range(B):
            for i in range(npg):
                rows = kv[b, i * page:(i + 1) * page]
                cache[table[b, i], : rows.shape[0]] = rows
        for splits in (0, 1, 2):
            out, lse = G.mla_decode(q_nope, q_pe, cache, table, np.full(B, L, np.int32), scale, num_kv_splits=splits)
            mag = np.abs(want).max()
            assert np.isfinite(out).all()
            assert np.abs(out - want).max() <= 2e-2 * mag                  # bf16 P (reference: fp32 P), bf16 output
            assert np.abs(out - want).mean() <= 4e-3 * np.abs(want).mean() + 1e-6
            np.testing.assert_allclose(lse / np.log(2.0), lse2, rtol=0, atol=2e-3)


def test_mla_decode_lazy_rescale_and_padding_slots():
    """(1) keys whose scores grow by >> 2^8 along the sequence force the lazily raised reference maximum (the O^T
    rescale in tensor memory) several times; (2) kv_len == 0 (padded CUDA-graph batch slot) gives zeros, not NaN."""
    from oracle import mla_oracle
    rng = np.random.default_rng(11)
    B, Hq, page = 2, 128, 64
    L = 700
    q_nope, q_pe, kv, pt, kl = _mla_case(rng, B, Hq, page, [L, L])
    ramp = np.linspace(0.02, 3.0, page * pt.shape[1], dtype=np.float32)
    for b in range(B):
        for i, pg in enumerate(pt[b]):
            kv[pg] = mla_oracle.bf16_round(kv[pg] * ramp[i * page:(i + 1) * page, None])
    kl[1] = 0
    out, lse = G.mla_decode(q_nope, q_pe, kv, pt, kl, 0.3)
    want, want_lse = mla_oracle.mla_decode(q_nope[:1], q_pe[:1], kv, pt[:1], kl[:1], 0.3, p_bf16=True)
    mag = np.abs(want).max()
    assert np.abs(out[0] - want[0]).max() <= (2.0 ** -7 + 2e-3) * mag
    np.testing.assert_allclose(lse[0], want_lse[0], rtol=0, atol=2e-3)
    assert not out[1].any() and np.isneginf(lse[1]).all()


def test_mla_kv_write_then_decode_roundtrip():
    """StaticCache.update semantics: writing tokens through the paged write kernel and attending over them equals
    attending over a cache built on the host."""
    rng = np.random.default_rng(5)
    B, Hq, page_size, L = 1, 128, 64, 200
    q_nope, q_pe, kv, pt, kl = _mla_case(rng, B, Hq, page_size, [L])
    kv_t = torch.zeros(kv.shape, dtype=torch.bfloat16, device="cuda")
    toks = np.arange(L)
    from oracle.mla_oracle import gather_kv
    rows = gather_kv(kv, pt[0], L, page_size)
    ckv = torch.from_numpy(rows[:, :512].copy()).to(torch.bfloat16).cuda()
    kpe = torch.from_numpy(rows[:, 512:].copy()).to(torch.bfloat16).cuda()
    pidx = torch.from_numpy(pt[0][toks // page_size].astype(np.int32)).cuda()
    poff = torch.from_numpy((toks % page_size).astype(np.int32)).cuda()
    G.mla_kv_write(kv_t, page_size, ckv, kpe, pidx, poff)
    written = kv_t.float().cpu().numpy()
    assert np.array_equal(gather_kv(written, pt[0], L, page_size), rows)
    a, _ = G.mla_decode(q_nope, q_pe, written, pt, kl, 0.07)
    b, _ = G.mla_decode(q_nope, q_pe, kv, pt, kl, 0.07)
    assert np.array_equal(a, b)


# ------------------------------------------------------------------------------------------ full BASELINE shapes
def test_v3_full_shape_decode_vs_oracle_and_properties(oracle):
    """DeepSeek-V3 routed experts at real size (E=256 resident, k=8, H=7168, I=2048, Q4_K/Q4_K/Q6_K), bs=1."""
    E, k, H, I = 256, 8, 7168, 2048
    gate, up, down = _synth(Q4_K, E * I * H, 51), _synth(Q4_K, E * I * H, 52), _synth(Q6_K, E * H * I, 53)
    rng = np.random.default_rng(0)
    ids = rng.permutation(E)[:k].astype(np.int64)[None, :]
    w = rng.random((1, k)).astype(np.float32)
    x = f32_to_bf16_bits((rng.standard_normal((1, H)) / 100).astype(np.float32))
    gb, db = gate.numel() // E, down.numel() // E
    # oracle on the k selected experts only (copied out before the in-place Q6_K re-layout)
    sel = ids[0].tolist()
    g_np = torch.cat([gate[e * gb:(e + 1) * gb] for e in sel]).cpu().numpy()
    u_np = torch.cat([up[e * gb:(e + 1) * gb] for e in sel]).cpu().numpy()
    d_np = torch.cat([down[e * db:(e + 1) * db] for e in sel]).cpu().numpy()
    want = oracle.moe_forward(k, H, I, g_np, u_np, d_np, Q4_K, Q4_K, Q6_K, BF16, np.arange(k, dtype=np.int64)[None, :], w, x)
    m = G.Moe(E, k, H, I, gate, up, down, Q4_K, Q4_K, Q6_K, BF16, max_tokens=8)
    got = m.forward(ids, w, x)
    assert_bf16_close(got, want)
    # determinism: same launch twice -> identical bits
    assert np.array_equal(got, m.forward(ids, w, x))
    # batch of 8 distinct tokens == the 8 single-token calls (no cross-token interaction)
    xs = f32_to_bf16_bits((rng.standard_normal((8, H)) / 100).astype(np.float32))
    idss = np.stack([rng.permutation(E)[:k] for _ in range(8)]).astype(np.int64)
    ws = rng.random((8, k)).astype(np.float32)
    batched = m.forward(idss, ws, xs)
    for t in range(8):
        assert np.array_equal(batched[t], m.forward(idss[t:t + 1], ws[t:t + 1], xs[t:t + 1])[0])
    m.close()


def test_v3_full_shape_relu_scaling_is_bit_exact():
    """With relu (use_silu=0) the path is positively homogeneous of degree 2 in x, and a power-of-two scale
    leaves every int8 activation unchanged: out(2x) == 4*out(x) bit-for-bit in fp32."""
    E, k, H, I = 16, 8, 7168, 2048
    gate, up, down = _synth(Q4_K, E * I * H, 61), _synth(Q4_K, E * I * H, 62), _synth(Q6_K, E * H * I, 63)
    m = G.Moe(E, k, H, I, gate, up, down, Q4_K, Q4_K, Q6_K, F32, use_silu=0)
    rng = np.random.default_rng(1)
    x = (rng.standard_normal((2, H)) / 100).astype(np.float32)
    ids = np.stack([rng.permutation(E)[:k] for _ in range(2)]).astype(np.int64)
    w = rng.random((2, k)).astype(np.float32)
    a, b = m.forward(ids, w, x), m.forward(ids, w, 2 * x)
    assert np.array_equal(b, 4 * a)
    # and linear in the routing weights
    c = m.forward(ids, 2 * w, x)
    assert np.array_equal(c, 2 * a)
    m.close()


# ------------------------------------------------------------------------------------------ grouped (prefill) path
@pytest.mark.parametrize("dt,E,k,H,I", [(Q6_K, 8, 4, 1024, 512), (Q4_K, 8, 4, 1024, 512), (Q6_K, 6, 6, 2048, 1536), (Q6_K, 16, 8, 7168, 2048)])
@pytest.mark.parametrize("hid", [F32, BF16])
def test_moe_grouped_tensor_core_path_vs_oracle(oracle, dt, E, k, H, I, hid):
    """qlen >= KTB200_GROUPED_MIN takes MOE::forward_many's shape (moe.cpp:248-365): per-expert GEMMs on tcgen05 with operands
    that hold the reference's integers exactly.  Same oracle, same tolerances as the per-pair kernels, and the launch count proves
    the grouped kernels ran (10 per chunk)."""
    gate, up, down = _synth(Q4_K, E * I * H, 21), _synth(Q4_K, E * I * H, 22), _synth(dt, E * H * I, 23)
    g_np, u_np, d_np = gate.cpu().numpy(), up.cpu().numpy(), down.cpu().numpy()
    m = G.Moe(E, k, H, I, gate, up, down, Q4_K, Q4_K, dt, hid, max_tokens=512)
    rng = np.random.default_rng(E * 1000 + H + dt)
    for qlen in ((101,) if H >= 7168 else (48, 131, 300)):
        x = (rng.standard_normal((qlen, H)) / 100).astype(np.float32)
        ids = np.stack([rng.permutation(E)[:k] for _ in range(qlen)]).astype(np.int64)
        if qlen > 100:
            ids[5:90, 0] = 1          # a crowded expert: several 32-token tiles, duplicates inside a token
            ids[7, :] = [-1, E, 1 << 40, -7][:k] + [0] * max(0, k - 4)   # invalid ids are skipped
            ids[ids == 2] = 3         # an expert nobody picks
        w = rng.random((qlen, k)).astype(np.float32)
        xin = x if hid == F32 else f32_to_bf16_bits(x)
        n0 = native.launch_count()
        got = m.forward(ids, w, xin)
        assert native.launch_count() - n0 == 10, "the grouped path did not run"
        want = oracle.moe_forward(E, H, I, g_np, u_np, d_np, Q4_K, Q4_K, dt, hid, ids, w, xin)
        if hid == F32:
            assert relmax(got, want) < FP_TOL, f"qlen={qlen}"
        else:
            assert_bf16_close(got, want)
    # device-side batch size: rows >= bsz untouched, rows < bsz identical
    sentinel = torch.full((qlen, H), 7.0, device="cuda", dtype=torch.float32 if hid == F32 else torch.bfloat16)
    got3 = m.forward(ids, w, xin, bsz=50, out=sentinel)
    assert np.array_equal(got3[:50], got[:50]) and (sentinel[50:] == 7.0).all()
    m.close()


def test_moe_grouped_matches_per_pair_kernels():
    """The integer dot of a super-block is the same number whichever kernel computes it (Q4_K everywhere: no fp16 rounding can
    occur below 2048); what differs is the fp32 order in which the per-block terms are added (lanes vs sequential)."""
    E, k, H, I = 8, 4, 2048, 768
    gate, up, down = _synth(Q4_K, E * I * H, 31), _synth(Q4_K, E * I * H, 32), _synth(Q4_K, E * H * I, 33)
    m = G.Moe(E, k, H, I, gate, up, down, Q4_K, Q4_K, Q4_K, F32, max_tokens=256)
    rng = np.random.default_rng(9)
    qlen = 200
    x = (rng.standard_normal((qlen, H)) / 100).astype(np.float32)
    ids = np.stack([rng.permutation(E)[:k] for _ in range(qlen)]).astype(np.int64)
    w = rng.random((qlen, k)).astype(np.float32)
    big = m.forward(ids, w, x)
    small = np.concatenate([m.forward(ids[i:i + 25], w[i:i + 25], x[i:i + 25]) for i in range(0, qlen, 25)])
    assert relmax(big, small) < 1e-5
    m.close()


@pytest.mark.parametrize("qlen", [16, 64, 4096])
def test_moe_grouped_vs_compiled_reference_forward_many(ref, qlen):
    """VERDICT r1 item 6: against the UNMODIFIED reference's MOE::forward_many (oracle/_ref, moe.cpp:248-365; it takes over from
    forward_one at group_min_len = 10) at qlen 16 (per-pair kernels here), 64 and 4096 (grouped path; four 1024-token chunks here,
    group_max_len 4096 there).  fp32 hidden: same tolerance as the decode path."""
    E, k, H, I = 8, 4, 1024, 512
    gate, up, down = _synth(Q4_K, E * I * H, 41), _synth(Q4_K, E * I * H, 42), _synth(Q6_K, E * H * I, 43)
    g_np, u_np, d_np = gate.cpu().numpy(), up.cpu().numpy(), down.cpu().numpy()
    m = G.Moe(E, k, H, I, gate, up, down, Q4_K, Q4_K, Q6_K, F32, max_tokens=4096)
    rng = np.random.default_rng(qlen)
    x = (rng.standard_normal((qlen, H)) / 100).astype(np.float32)
    ids = np.stack([rng.permutation(E)[:k] for _ in range(qlen)]).astype(np.int64)
    w = rng.random((qlen, k)).astype(np.float32)
    n0 = native.launch_count()
    got = m.forward(ids, w, x)
    assert native.launch_count() - n0 == (10 * ((qlen + 1023) // 1024) if qlen >= 48 else 2)
    want = ref.moe_forward(E, H, I, g_np, u_np, d_np, Q4_K, Q4_K, Q6_K, F32, ids, w, x, group_max_len=4096)
    assert relmax(got, want) < FP_TOL
    m.close()


# ------------------------------------------------------------------------------------------ FP8 128 x 128 linear
def _fp8_case(rng, T, K, N):
    from oracle import fp8_oracle as F
    x = f32_to_bf16_bits((rng.standard_normal((T, K)) / 10).astype(np.float32))
    w = F.to_e4m3_bytes((rng.standard_normal((N, K)) * 0.7).astype(np.float32))
    ws = (rng.random(((N + 127) // 128, K // 128)) * 0.02 + 0.001).astype(np.float32)
    return x, w, ws


def _fp8_run(x_bits, w, ws, bsz=None, out=None):
    lib = native.lib()
    T, K = x_bits.shape
    N = w.shape[0]
    w_d, ws_d = torch.from_numpy(w).cuda(), torch.from_numpy(ws).cuda()
    x_d = torch.from_numpy(x_bits.view(np.int16)).view(torch.bfloat16).cuda()
    y_d = torch.zeros((T, N), dtype=torch.bfloat16, device="cuda") if out is None else out
    h = C.c_void_p()
    native.check(lib.ktb200_fp8_linear_create(K, N, w_d.data_ptr(), ws_d.data_ptr(), BF16, 0, C.byref(h)))
    bsz_d = torch.tensor([bsz], dtype=torch.int32, device="cuda") if bsz is not None else None
    for _ in range(2):   # twice: the K-split workspace and tickets must come back zeroed
        native.check(lib.ktb200_fp8_linear_forward(h, T, x_d.data_ptr(), y_d.data_ptr(), bsz_d.data_ptr() if bsz_d is not None else None,
                                                   torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    lib.ktb200_fp8_linear_destroy(h)
    return y_d.cpu().view(torch.int16).numpy().view(np.uint16)


@pytest.mark.parametrize("T,K,N", [(1, 256, 256), (3, 1536, 24576), (8, 7168, 2112), (16, 16384, 7168), (20, 1024, 200), (1, 7168, 7168), (5, 128, 128)])
def test_fp8_linear_vs_oracle(T, K, N):
    """ktb200_fp8_linear_forward (TMA + tcgen05 kind::f8f6f4) against oracle/fp8_oracle.py (pinned to the reference's Triton
    kernels): act_quant inside the kernel, exact e4m3 products, (dot * a_s) * b_s per 128 of K in fp32; the K-split and the tensor
    core's summation order move the fp32 sum by round-off only -> bf16 outputs within 1 ulp, > 97 % identical."""
    from oracle import fp8_oracle as F
    rng = np.random.default_rng(T * 100003 + K + N)
    x, w, ws = _fp8_case(rng, T, K, N)
    got = _fp8_run(x, w, ws)
    want = f32_to_bf16_bits(F.linear_forward(bf16_to_f32(x), w, ws))
    assert_bf16_close(got, want)


@pytest.mark.parametrize("name", ["a", "b", "c"])
def test_fp8_linear_vs_reference_golden(golden_dir, name):
    """The golden vectors are the reference's own Triton kernels under the CPU interpreter, whose software casts drop a carry in
    ~2 % of the e4m3 bytes and truncate to bf16 (tests/test_oracle_pinned.py pins the oracle around both): the GPU result must
    equal the oracle and sit within those artifacts' reach of the golden output."""
    from oracle import fp8_oracle as F
    g = np.load(os.path.join(golden_dir, "fp8_ref.npz"))
    x, w, ws = g[f"{name}_x"], g[f"{name}_w"], g[f"{name}_ws"]
    got = _fp8_run(x, w, ws)
    assert_bf16_close(got, f32_to_bf16_bits(F.linear_forward(bf16_to_f32(x), w, ws)))
    a, b = bf16_to_f32(got), bf16_to_f32(g[f"{name}_c"])
    assert np.abs(a - b).max() <= 0.25 * np.abs(b).max()      # a sanity bound: the golden carries the interpreter's cast artifacts


def test_fp8_linear_bsz_rows_untouched():
    rng = np.random.default_rng(3)
    x, w, ws = _fp8_case(rng, 20, 512, 384)
    full = _fp8_run(x, w, ws)
    sentinel = torch.full((20, 384), 7.0, dtype=torch.bfloat16, device="cuda")
    part = _fp8_run(x, w, ws, bsz=18, out=sentinel)
    assert np.array_equal(part[:18], full[:18]) and (sentinel[18:] == 7.0).all()


def test_moe_block_forward_host_pinned_and_pageable_match_the_device_call():
    """ktb200_moe_block_forward_host (the reference-facing call with HOST buffers, bench.py's e2e leg): a pinned output is written
    by the kernel's own stores, pageable memory takes the staged copy — both must equal the device-pointer call bit for bit."""
    lib = native.lib()
    E, k, H, I = 8, 4, 4096, 512
    gate, up, down = _synth(Q4_K, E * I * H, 51), _synth(Q4_K, E * I * H, 52), _synth(Q6_K, E * H * I, 53)
    m = G.Moe(E, k, H, I, gate, up, down, Q4_K, Q4_K, Q6_K, BF16, max_tokens=8)
    rng = np.random.default_rng(12)
    Wg = torch.from_numpy(rng.standard_normal((E, H)).astype(np.float32)).cuda()
    bg = torch.from_numpy((0.01 * rng.standard_normal(E)).astype(np.float32)).cuda()
    gc = native.GateConfig(E, H, k, 1, 1, 0, 0, 1, 2.5, Wg.data_ptr(), bg.data_ptr(), BF16)
    s = torch.cuda.current_stream().cuda_stream
    for qlen in (1, 3):
        x = (torch.randn(qlen, H) / 10).to(torch.bfloat16)
        x_d = x.cuda()
        y_d, idx_d, w_d = torch.zeros_like(x_d), torch.zeros((qlen, k), dtype=torch.int64, device="cuda"), torch.zeros((qlen, k), device="cuda")
        native.check(lib.ktb200_moe_block_forward(C.byref(gc), m.h, None, qlen, x_d.data_ptr(), y_d.data_ptr(), idx_d.data_ptr(), w_d.data_ptr(), None, s))
        torch.cuda.synchronize()
        xp, yp = x.clone().pin_memory(), torch.zeros(qlen, H, dtype=torch.bfloat16).pin_memory()
        idp, wp = torch.zeros((qlen, k), dtype=torch.int64).pin_memory(), torch.zeros((qlen, k)).pin_memory()
        native.check(lib.ktb200_moe_block_forward_host(C.byref(gc), m.h, None, qlen, xp.data_ptr(), yp.data_ptr(), idp.data_ptr(), wp.data_ptr(), s))
        assert torch.equal(yp.view(torch.int16), y_d.cpu().view(torch.int16)) and torch.equal(idp, idx_d.cpu()) and torch.equal(wp, w_d.cpu())
        xn, yn = x.clone(), torch.zeros(qlen, H, dtype=torch.bfloat16)          # pageable
        native.check(lib.ktb200_moe_block_forward_host(C.byref(gc), m.h, None, qlen, xn.data_ptr(), yn.data_ptr(), None, None, s))
        assert torch.equal(yn.view(torch.int16), y_d.cpu().view(torch.int16))
    m.close()
