"""Generates the committed golden fixtures from the UNMODIFIED reference (oracle/_ref, built by
oracle/Makefile from /root/reference) and, for name translation / routing, by importing the
reference's Python.  Run in the build container only:

    make -C oracle ref && python tests/golden/make_golden.py

Outputs (small, committed):
    moe_small_*.npz      E=4 k=2 H=512 I=256, Q4_K/Q4_K/Q6_K + a Q5_K/Q5_K/Q4_K variant: quantised weights
                         (reference from_float), inputs, MOE::forward outputs for qlen 1,3,12 (fp32 and bf16)
    act_quant.npz        Q8_K / Q8_0 activation blocks for fp32 and bf16-valued rows (tie-heavy)
    dequant.npz          16 blocks per weight type: raw bytes + to_float values
    linear_mlp.npz       Linear / MLP forward outputs
    gate_v3.npz          MoEGate.forward (reference torch code, seed 42) ids/weights, V3 shapes scaled down + V3 full
    name_translation.json
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.bindings import (BF16, F32, IQ4_XS, Q2_K, Q3_K, Q4_K, Q5_K, Q6_K, Q8_0, Q8_K, Ref, TYPE_NAMES,  # noqa: E402
                             f32_to_bf16_bits)

OUT = os.path.dirname(os.path.abspath(__file__))
r = Ref.get(8)
print("reference build:", r.isa(), r.path)


def moe_case(rng, E, k, H, I, gt, ut, dt, qlens):
    g = rng.standard_normal((E, I, H)).astype(np.float32)
    u = rng.standard_normal((E, I, H)).astype(np.float32)
    d = rng.standard_normal((E, H, I)).astype(np.float32)
    gq, uq, dq = r.from_float(g, gt), r.from_float(u, ut), r.from_float(d, dt)
    out = {"E": E, "k": k, "H": H, "I": I, "gate_type": gt, "up_type": ut, "down_type": dt, "gate": gq, "up": uq, "down": dq}
    for qlen in qlens:
        x = (rng.standard_normal((qlen, H)) / 100).astype(np.float32)
        ids = np.stack([rng.permutation(E)[:k] for _ in range(qlen)]).astype(np.int64)
        w = rng.random((qlen, k)).astype(np.float32)
        xb = f32_to_bf16_bits(x)
        out[f"x_{qlen}"] = x
        out[f"ids_{qlen}"] = ids
        out[f"w_{qlen}"] = w
        out[f"out_f32_{qlen}"] = r.moe_forward(E, H, I, gq, uq, dq, gt, ut, dt, F32, ids, w, x)
        out[f"out_bf16_{qlen}"] = r.moe_forward(E, H, I, gq, uq, dq, gt, ut, dt, BF16, ids, w, xb)
    return out


rng = np.random.default_rng(20260922)
a = moe_case(rng, 4, 2, 512, 256, Q4_K, Q4_K, Q6_K, (1, 3, 12))
b = moe_case(rng, 4, 2, 512, 256, Q5_K, Q5_K, Q4_K, (1, 12))
moe = {**{f"a_{k}": v for k, v in a.items()}, **{f"b_{k}": v for k, v in b.items()}}
# one file per weight tensor plus one for the rest, so that no file exceeds 1 MB; tests/conftest.py joins them again
for part in ("gate", "up", "down"):
    np.savez_compressed(os.path.join(OUT, f"moe_small_{part}.npz"), **{n: v for n, v in moe.items() if n.endswith("_" + part)})
np.savez_compressed(os.path.join(OUT, "moe_small_io.npz"),
                    **{n: v for n, v in moe.items() if not n.endswith(("_gate", "_up", "_down"))})

# activation quantisation
rows = []
for i in range(8):
    x = (rng.standard_normal(1024) * (10.0 ** rng.integers(-3, 2))).astype(np.float32)
    if i % 2:
        x = (f32_to_bf16_bits(x).astype(np.uint32) << 16).view(np.float32)  # bf16-valued: many exact .5 ties
    rows.append(x)
rows[6][:256] = 0.0  # an all-zero block
X = np.stack(rows)
np.savez_compressed(os.path.join(OUT, "act_quant.npz"), x=X, q8k=np.stack([r.from_float(x, Q8_K) for x in X]),
                    q8_0=np.stack([r.from_float(x, Q8_0) for x in X]))

# dequant
dq = {}
for t in (Q2_K, Q3_K, Q4_K, Q5_K, Q6_K, IQ4_XS, Q8_0):
    n = 16 * 256
    w = rng.standard_normal(n).astype(np.float32)
    q = r.from_float(w, t)
    dq[f"raw_{TYPE_NAMES[t]}"] = q
    dq[f"val_{TYPE_NAMES[t]}"] = r.to_float(q, t, n)
np.savez_compressed(os.path.join(OUT, "dequant.npz"), **dq)

# linear / mlp
H, I, O = 512, 256, 384
wl = r.from_float(rng.standard_normal((O, H)).astype(np.float32), Q4_K)
wl6 = r.from_float(rng.standard_normal((O, H)).astype(np.float32), Q6_K)
g = r.from_float(rng.standard_normal((I, H)).astype(np.float32), Q4_K)
u = r.from_float(rng.standard_normal((I, H)).astype(np.float32), Q4_K)
d = r.from_float(rng.standard_normal((H, I)).astype(np.float32), Q6_K)
x = (rng.standard_normal((5, H)) / 10).astype(np.float32)
xb = f32_to_bf16_bits(x)
np.savez_compressed(os.path.join(OUT, "linear_mlp.npz"), H=H, I=I, O=O, wl=wl, wl6=wl6, g=g, u=u, d=d, x=x,
                    lin_f32=r.linear_forward(H, O, wl, Q4_K, F32, x), lin_bf16=r.linear_forward(H, O, wl, Q4_K, BF16, xb),
                    lin6_f32=r.linear_forward(H, O, wl6, Q6_K, F32, x),
                    mlp_f32=r.mlp_forward(H, I, g, u, d, Q4_K, Q4_K, Q6_K, F32, x),
                    mlp_bf16=r.mlp_forward(H, I, g, u, d, Q4_K, Q4_K, Q6_K, BF16, xb))

# routing: run the reference's own MoEGate.forward source (pure torch) without importing its package
import importlib.util
import types

import torch

src = open("/root/reference/archive/ktransformers/models/modeling_deepseek_v3.py").read()
start = src.index("class MoEGate(nn.Module):")
end = src.index("class DeepseekV3MoE(nn.Module):")
ns = {"torch": torch, "nn": torch.nn, "F": torch.nn.functional, "math": __import__("math")}
exec(src[start:end], ns)
RefGate = ns["MoEGate"]


def gate_case(E, H, k, n_group, topk_group, T, seed):
    torch.manual_seed(seed)
    cfg = types.SimpleNamespace(num_experts_per_tok=k, n_routed_experts=E, routed_scaling_factor=2.5, scoring_func="sigmoid",
                                topk_method="noaux_tc", n_group=n_group, topk_group=topk_group, norm_topk_prob=True, hidden_size=H)
    gate = RefGate(cfg)
    with torch.no_grad():
        gate.weight.copy_(torch.randn(E, H))                    # kt-kernel/examples/test_gate.py:33-34
        gate.e_score_correction_bias.copy_(torch.randn(E))
        x = torch.randn(1, T, H) / 10
        idx, w = gate(x)
        logits = torch.nn.functional.linear(x.view(-1, H).float(), gate.weight.float())
    return {"W": gate.weight.detach().numpy(), "bias": gate.e_score_correction_bias.detach().numpy(), "x": x[0].numpy(),
            "idx": idx.numpy(), "w": w.numpy(), "logits64": torch.nn.functional.linear(x.view(-1, H).double(), gate.weight.double()).detach().numpy()}


gs = gate_case(64, 256, 6, 8, 4, 64, 42)
np.savez_compressed(os.path.join(OUT, "gate_v3_small.npz"), **gs)

# name translation pairs from the reference's translate_name_to_gguf
src = open("/root/reference/archive/ktransformers/util/custom_gguf.py").read()
ns = {"re": __import__("re")}
exec(src[src.index("def translate_name_to_gguf_mixtral"):src.index("if __name__ == '__main__'")], ns)
names = ["model.layers.3.mlp.experts", "model.layers.3.mlp.experts.7.gate_proj.weight", "model.layers.10.mlp.gate.weight",
         "model.layers.10.mlp.gate.e_score_correction_bias", "model.layers.10.mlp.shared_experts.gate_proj.weight",
         "model.layers.10.mlp.shared_experts.up_proj.weight", "model.layers.10.mlp.shared_experts.down_proj.weight",
         "model.layers.0.mlp.down_proj.weight", "model.layers.0.mlp.gate_proj.weight", "lm_head.weight",
         "model.embed_tokens.weight", "model.norm.weight", "model.layers.5.self_attn.kv_a_proj_with_mqa.weight",
         "model.layers.5.self_attn.kv_a_layernorm.weight", "model.layers.5.self_attn.q_a_proj.weight",
         "model.layers.5.self_attn.q_a_layernorm.weight", "model.layers.5.self_attn.q_b_proj.weight",
         "model.layers.5.self_attn.o_proj.weight", "model.layers.5.input_layernorm.weight",
         "model.layers.5.post_attention_layernorm.weight", "model.layers.5.self_attn.kv_b_proj.weight",
         "blk.3.ffn_gate_exps.weight", "model.layers.2.block_sparse_moe.experts.3.w1.weight",
         "model.layers.2.block_sparse_moe.gate.weight", "model.layers.4.mlp.experts.ffn_gate_exps.weight",
         "model.layers.1.feed_forward.router.weight", "model.layers.1.mlp.shared_expert.up_proj.weight",
         "model.layers.1.mlp.shared_expert_gate.weight", "model.layers.7.mlp.experts.ffn_down_exp.weight"]
json.dump({n: ns["translate_name_to_gguf"](n) for n in names}, open(os.path.join(OUT, "name_translation.json"), "w"), indent=1)
print("golden fixtures written:", sorted(os.listdir(OUT)))
