"""Case definitions + deterministic input generation shared by ``tests/golden/make_golden.py`` (which
runs the reference on them) and the tests (which run the oracle / the CUDA kernels on them)."""
from __future__ import annotations

import types

import numpy as np
import torch

D = 128  # the kernels are specialised for head_dim 128 (all four BASELINE models)

LAYER_CASES = [
    dict(name="tuple_g2_mix", path="tuple", Hq=8, Hkv=4, gate=[1, 0, 1, 0], sink=4, recent=8, hidden=64,
         chunks=[5, 1, 1, 7, 20, 1, 1, 1, 30, 3], B=1, seed=11, theta=10000.0),
    dict(name="tuple_g4_deploy", path="tuple", Hq=8, Hkv=2, gate=[0, 1], sink=64, recent=256, hidden=64,
         chunks=[100, 300, 1, 1, 50, 1], B=1, seed=12, theta=500000.0),
    dict(name="tuple_mha_allstream", path="tuple", Hq=4, Hkv=4, gate=[0, 0, 0, 0], sink=2, recent=3, hidden=32,
         chunks=[1, 1, 1, 1, 1, 1, 1, 9, 1, 2], B=1, seed=13, theta=10000.0),
    dict(name="tuple_g4_allfull", path="tuple", Hq=8, Hkv=2, gate=[1, 1], sink=4, recent=4, hidden=32,
         chunks=[33, 1, 2, 1], B=1, seed=14, theta=10000.0),
    dict(name="tuple_b2", path="tuple", Hq=4, Hkv=2, gate=[1, 0], sink=3, recent=5, hidden=32,
         chunks=[6, 1, 4, 1, 1], B=2, seed=15, theta=10000.0),
    dict(name="static_g4_evict", path="static", Hq=8, Hkv=2, gate=[1, 0], sink=16, recent=64, hidden=64,
         chunks=[90, 40, 1, 1, 1, 17, 1], B=1, seed=21, theta=10000.0, rope_factor=None, max_size=256,
         evict_after={2: 1, 3: 1}),
    dict(name="static_g2_scaled", path="static", Hq=4, Hkv=2, gate=[0, 1], sink=8, recent=8, hidden=32,
         chunks=[10, 10, 1, 1, 30, 1], B=1, seed=22, theta=10000.0, rope_factor=8.0, max_size=64),
]

MISTRAL_CASES = ("tuple_g4_deploy", "static_g4_evict")  # also run through the reference's mistral.py twin

# INT4-KV attention (demo/int4_kv.py cache class + demo/w8a8kv4_llama.py:174-287 forward); the reference's dequantise
# wrapper assumes contiguous [:, :len] slices, i.e. batch 1 (int4_kv.py:91-112)
INT4_CASES = [
    dict(name="int4_g4_mix", Hq=8, Hkv=2, n_full=1, sink=4, recent=12, chunks=[20, 1, 1, 7, 1, 30, 1, 1], seed=41,
         max_size=96, prefill_chunk=32),
    dict(name="int4_g2_allfull", Hq=4, Hkv=2, n_full=2, sink=2, recent=3, chunks=[9, 1, 5, 1], seed=42, max_size=32,
         prefill_chunk=16),
    # (an all-streaming layer cannot run in the reference: its quantisation scratch is sized by the number of
    #  RETRIEVAL heads, int4_kv.py:231-245, so chunk * n_stream must stay <= prefill_chunk * max n_full)
    dict(name="int4_mha_1of4", Hq=4, Hkv=4, n_full=1, sink=3, recent=5, chunks=[6, 1, 1, 1, 1, 4, 1, 9, 1], seed=43,
         max_size=32, prefill_chunk=32),
]

# Training-time streaming (Lambda) masks: generate_streaming_mask + streaming_attn_sdpa (duo_attn/patch/streaming_attn.py:14-42)
TRAIN_MASK_CASES = [
    dict(name="s37_4_8", S=37, Hq=4, Hkv=2, sink=4, recent=8, seed=51),
    dict(name="s64_16_16", S=64, Hq=4, Hkv=4, sink=16, recent=16, seed=52),
    dict(name="s24_0_5", S=24, Hq=2, Hkv=1, sink=0, recent=5, seed=53),
    dict(name="s20_3_1", S=20, Hq=2, Hkv=2, sink=3, recent=1, seed=54),
    dict(name="s330_64_257", S=330, Hq=2, Hkv=1, sink=64, recent=257, seed=55),  # deploy 64/256 in the chunk-1 limit (+1)
]


def make_train_mask_inputs(case):
    g = torch.Generator().manual_seed(case["seed"])
    q = torch.randn(1, case["S"], case["Hq"], D, generator=g)
    k = torch.randn(1, case["S"], case["Hkv"], D, generator=g)
    v = torch.randn(1, case["S"], case["Hkv"], D, generator=g)
    return q, k, v


def make_int4_inputs(case):
    """Post-RoPE fp16 q/k/v per chunk (RoPE is pinned separately; the fixture isolates cache + attention)."""
    g = torch.Generator().manual_seed(case["seed"])
    out = []
    for n in case["chunks"]:
        q = (torch.randn(1, n, case["Hq"], D, generator=g) * 0.9).to(torch.float16)
        k = (torch.randn(1, n, case["Hkv"], D, generator=g) * 1.1).to(torch.float16)
        v = (torch.randn(1, n, case["Hkv"], D, generator=g)).to(torch.float16)
        out.append((q, k, v))
    return out


def int4_checksum(chunks):
    return float(sum(float(t.double().abs().sum()) for c in chunks for t in c))


def make_int4_kernel_input():
    """[2, 300, 4, 128] fp16 for the INT4 quantise / dequantise kernels: 2400 groups of 128 whose magnitudes span two
    decades."""
    rng = np.random.RandomState(2)
    return (rng.randn(2, 300, 4, D) * rng.uniform(0.05, 5, size=(2, 300, 4, 1))).astype(np.float16)


# Model-level drivers (tuple_kv_cache.py / static_kv_cache.py patched ForCausalLM forwards + enable_* functions)
MODEL_CASES = [
    dict(name="llama_tuple", kind="llama", path="tuple", gates=[[1.0, 0.0], [0.0, 1.0]], sink=4, recent=6,
         chunks=[20, 1, 1, 9, 1, 1], seed=51),
    dict(name="llama_static", kind="llama", path="static", gates=[[1.0, 0.0], [0.0, 1.0]], sink=4, recent=6,
         chunks=[20, 1, 1, 9, 1, 1], seed=51, max_size=64, evict_after={2: 1}),
    dict(name="mistral_tuple", kind="mistral", path="tuple", gates=[[0.0, 1.0], [1.0, 1.0]], sink=2, recent=5,
         chunks=[11, 1, 6, 1, 1], seed=52),
    dict(name="mistral_static", kind="mistral", path="static", gates=[[0.0, 1.0], [1.0, 1.0]], sink=2, recent=5,
         chunks=[11, 1, 6, 1, 1], seed=52, max_size=32, evict_after={3: 1}),
]
MODEL_VOCAB = 48


def make_tiny_model(case):
    """2-layer Llama/Mistral (4 q heads, 2 kv heads, head_dim 128, hidden 512 = heads * head_dim as the reference's
    cache assumes, static_kv_cache.py:33-40) with every parameter drawn from a seeded generator (independent of HF's
    initialisation order), plus the token ids of the schedule."""
    if case["kind"] == "llama":
        from transformers import LlamaConfig as Cfg, LlamaForCausalLM as M
        extra = {}
    else:
        from transformers import MistralConfig as Cfg, MistralForCausalLM as M
        extra = dict(sliding_window=None)
    cfg = Cfg(hidden_size=512, num_attention_heads=4, num_key_value_heads=2, head_dim=128, num_hidden_layers=2,
              intermediate_size=64, vocab_size=MODEL_VOCAB, max_position_embeddings=512, rope_theta=10000.0,
              attn_implementation="eager", tie_word_embeddings=False, **extra)
    model = M(cfg).eval()
    g = torch.Generator().manual_seed(case["seed"])
    tot = 0.0
    with torch.no_grad():
        for name, prm in model.named_parameters():
            if prm.dim() == 1:
                prm.copy_(1.0 + 0.1 * torch.randn(prm.shape, generator=g))
            else:
                prm.copy_(torch.randn(prm.shape, generator=g) * (1.5 / prm.shape[-1] ** 0.5))
            tot += float(prm.double().abs().sum())
    ids = [torch.randint(0, MODEL_VOCAB, (1, n), generator=g) for n in case["chunks"]]
    return model, ids, tot


REORDER_CASES = [
    dict(name="q_out_bias", seed=1, **{"in": 24, "out": 48}, bias=True, gate=[0.9, 0.1, 0.7, 0.2], repeat=12,
         channel="out"),
    dict(name="o_in", seed=2, **{"in": 48, "out": 20}, bias=False, gate=[0.0, 1.0, 0.0, 1.0], repeat=12,
         channel="in"),
    dict(name="k_out_allfull", seed=3, **{"in": 16, "out": 32}, bias=False, gate=[1.0, 1.0], repeat=16,
         channel="out"),
]


def make_layer_inputs(case):
    g = torch.Generator().manual_seed(case["seed"])
    Hq, Hkv, hid, B = case["Hq"], case["Hkv"], case["hidden"], case["B"]
    s = hid ** -0.5
    data = dict(
        B=B,
        wq=torch.randn(Hq * D, hid, generator=g) * s * 1.5,
        wk=torch.randn(Hkv * D, hid, generator=g) * s * 1.5,
        wv=torch.randn(Hkv * D, hid, generator=g) * s,
        wo=torch.randn(hid, Hq * D, generator=g) * (Hq * D) ** -0.5,
        gate=torch.tensor(case["gate"], dtype=torch.float32),
        chunks=[torch.randn(B, n, hid, generator=g) for n in case["chunks"]],
    )
    return data


def checksum(data):
    tot = 0.0
    for k in ("wq", "wk", "wv", "wo"):
        tot += float(data[k].double().sum())
    for c in data["chunks"]:
        tot += float(c.double().abs().sum())
    return tot


def hf_rotary(case, dtype=torch.float32):
    """The real transformers LlamaRotaryEmbedding for this case's theta (default rope type)."""
    from transformers import LlamaConfig
    from transformers.models.llama.modeling_llama import LlamaRotaryEmbedding

    cfg = LlamaConfig(hidden_size=case["Hq"] * D, num_attention_heads=case["Hq"],
                      num_key_value_heads=case["Hkv"], head_dim=D, num_hidden_layers=1, intermediate_size=64,
                      vocab_size=32, max_position_embeddings=4096, rope_theta=case["theta"])
    try:
        rp = dict(getattr(cfg, "rope_parameters", None) or {})
        if rp.get("rope_theta") != case["theta"]:
            rp.update(rope_theta=case["theta"], rope_type="default")
            cfg.rope_parameters = rp
    except Exception:
        pass
    return LlamaRotaryEmbedding(config=cfg)


class RefAttnModule(torch.nn.Module):
    """The attributes the reference forward reads from ``self`` (HF-4.45 LlamaAttention surface),
    with weights reordered by the REFERENCE's own reorder functions (``putils`` =
    duo_attn.patch.utils of the reference), as enable_llama_duo_attention_eval does (llama.py:523-554)."""

    def __init__(self, case, data, putils):
        super().__init__()
        Hq, Hkv, hid = case["Hq"], case["Hkv"], case["hidden"]
        self.num_heads, self.num_key_value_heads, self.head_dim = Hq, Hkv, D
        self.num_key_value_groups = Hq // Hkv
        self.hidden_size = Hq * D  # the forward only uses it for reshape(bsz, q_len, hidden_size)
        self.q_proj = torch.nn.Linear(hid, Hq * D, bias=False)
        self.k_proj = torch.nn.Linear(hid, Hkv * D, bias=False)
        self.v_proj = torch.nn.Linear(hid, Hkv * D, bias=False)
        self.o_proj = torch.nn.Linear(Hq * D, hid, bias=False)
        self.q_proj.weight.data = data["wq"].clone()
        self.k_proj.weight.data = data["wk"].clone()
        self.v_proj.weight.data = data["wv"].clone()
        self.o_proj.weight.data = data["wo"].clone()
        gate = data["gate"].clone()
        G = self.num_key_value_groups
        putils.reorder_linear_weights(self.q_proj, gate, G * D, "out")
        putils.reorder_linear_weights(self.k_proj, gate, D, "out")
        putils.reorder_linear_weights(self.v_proj, gate, D, "out")
        putils.reorder_linear_weights(self.o_proj, gate, G * D, "in")
        self.register_buffer("full_attention_heads", putils.reorder_full_attn_heads(gate))
        self.sink_size, self.recent_size = case["sink"], case["recent"]
        self.rotary_emb = hf_rotary(case)
        self.rope_theta = case["theta"]
        rs = None if case.get("rope_factor") is None else {"factor": case["rope_factor"], "type": "linear"}
        self.config = types.SimpleNamespace(rope_scaling=rs)


class FakeModel:
    """What DuoAttentionStaticKVCache.__init__ reads from ``model`` (static_kv_cache.py:33-40)."""

    def __init__(self, case, mod):
        self._mod = mod
        self.config = types.SimpleNamespace(
            num_hidden_layers=1, num_attention_heads=case["Hq"], num_key_value_heads=case["Hkv"],
            hidden_size=case["Hq"] * D)

    def parameters(self):
        return self._mod.parameters()
