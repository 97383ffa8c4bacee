"""CPU: pins the oracle (oracle/ktoracle.c, oracle/gate_oracle.py) against the committed golden vectors that
were generated from the unmodified reference, and — where oracle/_ref is present — against the reference
itself on fresh random inputs."""
import json
import os

import numpy as np
import pytest

from oracle.bindings import (BF16, F32, IQ4_XS, Q2_K, Q3_K, Q4_K, Q5_K, Q6_K, Q8_0, Q8_K, TYPE_NAMES, bf16_to_f32,
                             f32_to_bf16_bits)
from oracle import gate_oracle

TYPES = {n: t for t, n in TYPE_NAMES.items()}


def rel(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def test_activation_quantisation_is_byte_exact(oracle, golden_dir):
    g = np.load(os.path.join(golden_dir, "act_quant.npz"))
    for i, x in enumerate(g["x"]):
        got = oracle.from_float(x, Q8_K)
        want = g["q8k"][i].copy()
        # the reference leaves bsums of an all-zero block stale; the oracle zeroes them
        for b in range(x.size // 256):
            if not x[b * 256:(b + 1) * 256].any():
                want[b * 292 + 260:(b + 1) * 292] = 0
        assert np.array_equal(got, want), f"Q8_K row {i}"
        assert np.array_equal(oracle.from_float(x, Q8_0), g["q8_0"][i]), f"Q8_0 row {i}"


def test_dequantisation_matches_reference(oracle, golden_dir):
    g = np.load(os.path.join(golden_dir, "dequant.npz"))
    for name in ("Q2_K", "Q3_K", "Q4_K", "Q5_K", "Q6_K", "IQ4_XS", "Q8_0"):
        got = oracle.to_float(g[f"raw_{name}"], TYPES[name], g[f"val_{name}"].size)
        np.testing.assert_allclose(got, g[f"val_{name}"], rtol=0, atol=1e-6, err_msg=name)


@pytest.mark.parametrize("case", ["a", "b"])
def test_moe_forward_matches_golden(oracle, moe_small, case):
    g = moe_small
    E, k, H, I = (int(g[f"{case}_{n}"]) for n in ("E", "k", "H", "I"))
    gt, ut, dt = (int(g[f"{case}_{n}"]) for n in ("gate_type", "up_type", "down_type"))
    for qlen in (1, 3, 12):
        if f"{case}_x_{qlen}" not in g:
            continue
        x, ids, w = g[f"{case}_x_{qlen}"], g[f"{case}_ids_{qlen}"], g[f"{case}_w_{qlen}"]
        out = oracle.moe_forward(E, H, I, g[f"{case}_gate"], g[f"{case}_up"], g[f"{case}_down"], gt, ut, dt, F32, ids, w, x)
        assert rel(out, g[f"{case}_out_f32_{qlen}"]) < 1e-3        # north-star tolerance; typical 3e-7
        assert rel(out, g[f"{case}_out_f32_{qlen}"]) < 2e-5, "oracle drifted from the reference beyond fp32 re-association"
        outb = oracle.moe_forward(E, H, I, g[f"{case}_gate"], g[f"{case}_up"], g[f"{case}_down"], gt, ut, dt, BF16, ids, w, f32_to_bf16_bits(x))
        want = bf16_to_f32(g[f"{case}_out_bf16_{qlen}"])
        # bf16 outputs: at most 1 bf16 ulp (2^-8 relative) on a few elements
        assert np.abs(bf16_to_f32(outb) - want).max() <= np.abs(want).max() * 2 ** -7
        assert (outb == g[f"{case}_out_bf16_{qlen}"]).mean() > 0.98


def test_linear_and_mlp_match_golden(oracle, golden_dir):
    g = np.load(os.path.join(golden_dir, "linear_mlp.npz"))
    H, I, O = int(g["H"]), int(g["I"]), int(g["O"])
    assert rel(oracle.linear_forward(H, O, g["wl"], Q4_K, F32, g["x"]), g["lin_f32"]) < 2e-5
    assert rel(oracle.linear_forward(H, O, g["wl6"], Q6_K, F32, g["x"]), g["lin6_f32"]) < 2e-5
    assert rel(oracle.mlp_forward(H, I, g["g"], g["u"], g["d"], Q4_K, Q4_K, Q6_K, F32, g["x"]), g["mlp_f32"]) < 2e-5
    got = oracle.linear_forward(H, O, g["wl"], Q4_K, BF16, f32_to_bf16_bits(g["x"]))
    assert (got == g["lin_bf16"]).mean() > 0.98


def test_gate_oracle_matches_reference_torch(golden_dir):
    g = np.load(os.path.join(golden_dir, "gate_v3_small.npz"))
    idx, w, margin, _ = gate_oracle.route(g["x"], g["W"], g["bias"], top_k=6, n_group=8, topk_group=4, scoring="sigmoid",
                                          topk_method="noaux_tc", norm_topk_prob=True, routed_scaling_factor=2.5)
    ok = margin > 1e-5
    assert ok.mean() > 0.95
    # ids: exact as sorted sets (kt-kernel/examples/test_gate.py:201-214)
    assert np.array_equal(np.sort(idx[ok], axis=1), np.sort(g["idx"][ok], axis=1))
    # weights: align by id
    for t in np.nonzero(ok)[0]:
        mine = dict(zip(idx[t].tolist(), w[t].tolist()))
        for e, wr in zip(g["idx"][t].tolist(), g["w"][t].tolist()):
            assert abs(mine[e] - wr) < 1e-5 * max(1.0, abs(wr))


def test_name_translation_matches_reference(golden_dir):
    from ktransformers_b200.util.custom_gguf import translate_name_to_gguf
    pairs = json.load(open(os.path.join(golden_dir, "name_translation.json")))
    for src, dst in pairs.items():
        assert translate_name_to_gguf(src) == dst, src


# ---- checks against the compiled reference on fresh inputs where oracle/_ref is built, else on its stored outputs ------------
def _ref_or_none():
    from oracle.bindings import Ref
    return Ref.get(min(os.cpu_count() or 1, 16)) if Ref.available() else None


def _dequant_q8(q, t):
    """float64 values of Q8_K (fp32 d, int8 qs[256], int16 bsums[16]) or Q8_0 (fp16 d, int8 qs[32]) blocks."""
    size, n, off = (292, 256, 4) if t == Q8_K else (34, 32, 2)
    b = q.reshape(-1, size)
    d = b[:, :off].copy().view(np.float32 if t == Q8_K else np.float16)[:, 0].astype(np.float64)
    return (b[:, off:off + n].view(np.int8).astype(np.float64) * d[:, None]).reshape(-1)


@pytest.mark.parametrize("wtype", [Q2_K, Q3_K, Q4_K, Q5_K, Q6_K, IQ4_XS, Q8_0])
def test_vec_dot_against_ref(oracle, golden_dir, wtype):
    """Without oracle/_ref the operands are the reference's own stored bytes (tests/golden/make_golden.py): weight blocks from its
    from_float with its to_float values (dequant.npz), activation rows with its Q8_K / Q8_0 blocks (act_quant.npz).  Its vec_dot
    result is not stored, so the oracle's is held to the exact dot product of the reference's dequantised operands instead."""
    ref = _ref_or_none()
    vdt = Q8_0 if wtype == Q8_0 else Q8_K
    if ref is not None:
        rng = np.random.default_rng(wtype)
        n = 256 * 12
        wq = ref.from_float(rng.standard_normal(n).astype(np.float32), wtype)
        x = (rng.standard_normal(n) / 7).astype(np.float32)
        xq = ref.from_float(x, vdt)
        b, wval = ref.vec_dot(wtype, n, wq, xq), ref.to_float(wq, wtype, n)
    else:
        dq, aq = np.load(os.path.join(golden_dir, "dequant.npz")), np.load(os.path.join(golden_dir, "act_quant.npz"))
        wq, wval = dq[f"raw_{TYPE_NAMES[wtype]}"], dq[f"val_{TYPE_NAMES[wtype]}"]
        n = wval.size
        rows = n // aq["x"].shape[1]                  # whole rows: blocks never straddle two of them
        x = aq["x"][:rows].reshape(-1)
        xq = np.concatenate(aq["q8_0" if vdt == Q8_0 else "q8k"][:rows])
        b = float(np.dot(wval.astype(np.float64), _dequant_q8(xq, vdt)))
    assert np.array_equal(oracle.from_float(x, vdt), xq)
    a = oracle.vec_dot(wtype, n, wq, xq)
    assert abs(a - b) <= 2e-5 * max(abs(b), 1.0)
    np.testing.assert_allclose(oracle.to_float(wq, wtype, n), wval, rtol=0, atol=1e-6)


@pytest.mark.parametrize("qlen", [1, 5, 24])
def test_moe_against_ref_fresh(oracle, moe_small, qlen):
    """Without oracle/_ref: the reference's stored MOE::forward output (moe_small case a, Q4_K/Q4_K/Q6_K, bf16) for its 12 tokens,
    cycled to qlen rows; each token's output depends on that token alone."""
    ref = _ref_or_none()
    if ref is not None:
        rng = np.random.default_rng(100 + qlen)
        E, k, H, I = 8, 4, 1024, 512
        gq = ref.from_float(rng.standard_normal((E, I, H)).astype(np.float32), Q4_K)
        uq = ref.from_float(rng.standard_normal((E, I, H)).astype(np.float32), Q4_K)
        dq = ref.from_float(rng.standard_normal((E, H, I)).astype(np.float32), Q6_K)
        x = f32_to_bf16_bits((rng.standard_normal((qlen, H)) / 100).astype(np.float32))
        ids = np.stack([rng.permutation(E)[:k] for _ in range(qlen)]).astype(np.int64)
        w = rng.random((qlen, k)).astype(np.float32)
        b = bf16_to_f32(ref.moe_forward(E, H, I, gq, uq, dq, Q4_K, Q4_K, Q6_K, BF16, ids, w, x))
    else:
        g = moe_small
        E, H, I = (int(g[f"a_{n}"]) for n in ("E", "H", "I"))
        gq, uq, dq = g["a_gate"], g["a_up"], g["a_down"]
        rows = np.arange(qlen) % 12
        x, ids, w = f32_to_bf16_bits(g["a_x_12"][rows]), g["a_ids_12"][rows], g["a_w_12"][rows]
        b = bf16_to_f32(g["a_out_bf16_12"][rows])
    a = bf16_to_f32(oracle.moe_forward(E, H, I, gq, uq, dq, Q4_K, Q4_K, Q6_K, BF16, ids, w, x))
    # a one-LSB flip of an int8 activation (knife-edge rounding under fp32 re-association) moves outputs by
    # up to ~2e-3 of the row norm; anything larger is a real divergence
    # ... on top of the 1-ulp (2^-8 relative) granularity of the bf16 output itself
    assert (np.abs(a - b) <= 2.0 ** -7 * np.maximum(np.abs(a), np.abs(b)) + 4e-3 * np.abs(b).max()).all()
    assert np.abs(a - b).mean() <= 1e-3 * np.abs(b).mean()


def _mla_fixture(golden_dir, name):
    g = np.load(os.path.join(golden_dir, "mla_ref.npz"))
    f = lambda k: bf16_to_f32(g[f"{name}_{k}"])
    return f("q_nope"), f("q_pe"), f("kv"), float(g[f"{name}_scale"]), f("out"), g[f"{name}_lse2"]


@pytest.mark.parametrize("name", ["a", "b", "c"])
def test_mla_oracle_matches_reference_attention_ref_torch(golden_dir, name):
    """oracle/mla_oracle.py against the outputs of the reference's attention_ref_torch (flashinfer_wrapper.py:30-76):
    contiguous cache rows are laid out as pages of 32 with a shuffled page table."""
    from oracle import mla_oracle
    q_nope, q_pe, kv, scale, want, lse2 = _mla_fixture(golden_dir, name)
    B, L = kv.shape[0], kv.shape[1]
    page = 32
    npg = (L + page - 1) // page
    rng = np.random.default_rng(1)
    cache = rng.standard_normal((B * npg + 2, page, 576)).astype(np.float32)
    table = rng.permutation(B * npg + 2)[: B * npg].reshape(B, npg).astype(np.int32)
    for b in range(B):
        for i in range(npg):
            rows = kv[b, i * page:(i + 1) * page]
            cache[table[b, i], : rows.shape[0]] = rows
    out, lse = mla_oracle.mla_decode(q_nope, q_pe, cache, table, np.full(B, L, np.int32), scale, p_bf16=False)
    mag = np.abs(want).max()
    assert np.abs(out - want).max() <= 2.0 ** -8 * mag * 1.01          # the reference rounds its output to bf16
    np.testing.assert_allclose(lse / np.log(2.0), lse2, rtol=0, atol=1e-4)


def test_shimmed_amx_backend_runs_the_reference_int4_moe():
    """oracle/_ref/libktamx.so: the reference's AMXInt4_MOE (kt-kernel/operators/amx) built through the numa/hwloc shim.
    Checked like the reference's own accuracy test (kt-kernel test_moe_amx_accuracy_int4: relative mean error vs the fp32
    restatement below 0.35 for INT4)."""
    from oracle.bindings import AmxRef
    if not AmxRef.available():
        pytest.skip(AmxRef.why_unavailable())
    amx = AmxRef.get(4)
    rng = np.random.default_rng(0)
    E, k, H, I = 8, 4, 1024, 512
    g, u, d = (rng.standard_normal((E, I, H)).astype(np.float32), rng.standard_normal((E, I, H)).astype(np.float32),
               rng.standard_normal((E, H, I)).astype(np.float32))
    gb, ub, db = f32_to_bf16_bits(g), f32_to_bf16_bits(u), f32_to_bf16_bits(d)
    h = amx.moe_create(E, k, H, I, gb, ub, db)
    x = f32_to_bf16_bits((rng.standard_normal((2, H)) / 100).astype(np.float32))
    ids = np.stack([rng.permutation(E)[:k] for _ in range(2)]).astype(np.int64)
    w = rng.random((2, k)).astype(np.float32)
    out = bf16_to_f32(amx.moe_forward(h, ids, w, x))
    xf, gf, uf, df = bf16_to_f32(x), bf16_to_f32(gb), bf16_to_f32(ub), bf16_to_f32(db)
    ref = np.zeros_like(xf)
    for t in range(2):
        for j in range(k):
            e = ids[t, j]
            a = gf[e] @ xf[t]
            ref[t] += ((a / (1 + np.exp(-a))) * (uf[e] @ xf[t])) @ df[e].T * w[t, j]
    assert np.abs(out - ref).mean() / np.abs(ref).mean() < 0.35
    amx.moe_destroy(h)


@pytest.mark.parametrize("name", ["a", "b", "c"])
def test_fp8_oracle_matches_the_references_triton_kernels(golden_dir, name):
    """oracle/fp8_oracle.py against tests/golden/fp8_ref.npz — outputs of the reference's own act_quant / fp8_gemm_kernel
    (fp8gemm.py) run by Triton's CPU interpreter (tests/golden/make_fp8_golden.py): scales exact, quantised bytes exact up to the
    interpreter's two cast artifacts (fp32 -> e4m3 carry, fp32 -> bf16 truncation); the fp32 GEMM accumulator is bit-identical."""
    from oracle import fp8_oracle as F
    from oracle.bindings import bf16_to_f32, f32_to_bf16_bits
    g = np.load(os.path.join(golden_dir, "fp8_ref.npz"))
    x = bf16_to_f32(g[f"{name}_x"])
    q, s = F.act_quant(x)
    assert np.array_equal(s, g[f"{name}_s"])
    # Triton's CPU interpreter casts fp32 -> e4m3 in software: it drops the carry when rounding to nearest crosses a binade
    # (124.16 -> 64 instead of 128) and rounds exact ties away from zero; the GPU's cvt.rn.satfinite and the oracle round to
    # nearest even.  Exactly those bytes differ and nothing else does:
    gq = g[f"{name}_q"]
    diff = q != gq
    assert diff.mean() < 0.03
    v = np.abs(x.reshape(x.shape[0], -1, 128) / s[..., None]).reshape(x.shape)
    lo, hi = np.abs(F.e4m3_bytes_to_f32(q)), np.abs(F.e4m3_bytes_to_f32(gq))
    step = q.astype(int) - gq.astype(int)
    carry = diff & (step == 8)             # (1) RN carried into the next binade: the interpreter kept the old exponent
    tie = diff & (step == -1)              # (2) exact ties: the interpreter rounds half away from zero, RN (GPU, oracle) to even
    assert (diff == (carry | tie)).all()
    assert ((q[carry] & 7) == 0).all() and (lo[carry] >= v[carry]).all()
    assert (v[tie] == (lo[tie] + hi[tie]) / 2).all() and ((q[tie] & 1) == 0).all()
    # the GEMM is pinned on the golden's own quantised bytes
    acc = F.fp8_gemm(g[f"{name}_q"], g[f"{name}_s"], g[f"{name}_w"], g[f"{name}_ws"])
    # ... and is bit-exact at fp32: the interpreter narrows fp32 -> bf16 by truncation (the GPU rounds to nearest even), so the
    # golden equals the upper 16 bits of this accumulator, every element
    assert np.array_equal((acc.view(np.uint32) >> 16).astype(np.uint16), g[f"{name}_c"])
    # weight_dequant (fp8gemm.py:63-73) x fp32 matmul agrees with the blockwise GEMM to fp8-activation accuracy
    dense = x @ F.weight_dequant(g[f"{name}_w"], g[f"{name}_ws"]).T
    assert np.abs(dense - acc).max() <= 0.08 * np.abs(dense).max()
