"""Generate the golden fixtures in this directory by running the REFERENCE's own code.

Run in the build container (needs /root/reference; the fixtures are committed so the tests never
need it):

    python tests/golden/make_golden.py

``int4_ref_kernels.npz`` comes from the reference's compiled INT4 kernels instead, on a GPU (``make_int4_kernel_fixture``):

    python oracle/build_ref.py && python tests/golden/make_golden.py int4-kernels [OUT_DIR]

How the reference is made importable here (SURVEY.md §8c says it is not, as-is):
  * transformers 5.5 no longer re-exports ``List / Union / CrossEntropyLoss`` from modeling_llama — we add
    those three names to the real module before importing ``duo_attn.patch.llama``;
  * ``tensor_parallel``, ``accelerate``, ``matplotlib`` (absent, unused by the eval forward) are stubbed
    with empty modules;
  * the two CUDA-only third-party calls are swapped for the contract restatements in
    ``oracle/duo_oracle.py``: ``flash_attn_func`` -> ``flash_attn_contract`` and flashinfer's
    ``apply_rope_inplace`` -> ``rope_flashinfer`` (written back in place).
Everything else that runs is the reference's code, unmodified: ``llama_duo_attention_forward_one_way_
reordered`` (llama.py:146-306), ``..._static`` (:309-434), ``DuoAttentionStaticKVCache``
(static_kv_cache.py:18-315), ``reorder_linear_weights`` / ``reorder_full_attn_heads``
(patch/utils.py:6-45), ``load_attn_pattern`` / ``sparsify_attention_heads`` (duo_attn/utils.py:326-373).

Model level (``make_model_fixtures``): the reference's enable_* functions and patched ForCausalLM / Model / DecoderLayer
forwards (tuple_kv_cache.py, static_kv_cache.py) run unmodified on a tiny HF model.

INT4 (``make_int4_fixtures``): ``DuoAttentionStaticINT4KVCache`` (demo/int4_kv.py:115-492) and ``LlamaAttention.forward``
(demo/w8a8kv4_llama.py:174-287) also run unmodified, with the JIT-compiled quantisation module replaced by the NumPy
restatement of demo/quantize_int4.cu and the absent QServe packages stubbed.

Fixture inputs are regenerated from seeds by ``tests/golden_cases.py`` (shared with the tests); each
fixture stores an fp64 checksum of its inputs so RNG drift is detected rather than silently accepted.
"""
from __future__ import annotations

import json
import os
import sys
import types
import typing

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

REF = "/root/reference"


def import_reference():
    import transformers.models.llama.modeling_llama as ml
    import transformers.models.mistral.modeling_mistral as mm
    from torch.nn import CrossEntropyLoss

    for m in (ml, mm):
        for n, v in dict(List=typing.List, Union=typing.Union, CrossEntropyLoss=CrossEntropyLoss).items():
            if not hasattr(m, n):
                setattr(m, n, v)
    class _Anything(types.ModuleType):
        """Stub module: any attribute is a dummy callable (only import-time names are touched)."""

        def __getattr__(self, item):
            if item.startswith("__"):
                raise AttributeError(item)
            return lambda *a, **k: None

    for name in ("tensor_parallel", "tensor_parallel.pretrained_model", "tensor_parallel.config",
                 "tensor_parallel.communications", "tensor_parallel.aux_actions", "tensor_parallel.state_actions",
                 "tensor_parallel.autoconfig", "accelerate", "accelerate.utils", "matplotlib",
                 "matplotlib.pyplot", "matplotlib.colors", "seaborn"):
        if name not in sys.modules:
            m = _Anything(name)
            m.__path__ = []  # let `import a.b` treat it as a package
            sys.modules[name] = m
    sys.modules["tensor_parallel.pretrained_model"].TensorParallelPreTrainedModel = type("TPM", (), {})
    # put the reference FIRST so `import duo_attn` resolves to it, not to this repo's shim
    sys.path.insert(0, REF)
    for k in [k for k in sys.modules if k == "duo_attn" or k.startswith("duo_attn.")]:
        del sys.modules[k]
    import duo_attn.patch.llama as ref_llama
    import duo_attn.patch.mistral as ref_mistral
    import duo_attn.patch.utils as ref_putils

    try:
        import duo_attn.utils as ref_utils
    except Exception as e:  # pragma: no cover - only if more stubs are needed
        print("duo_attn.utils import failed:", repr(e))
        ref_utils = None
    return ref_llama, ref_mistral, ref_putils, ref_utils


def make_model_fixtures(O, GC, ref_llama, ref_mistral):
    """Run the reference's PATCHED MODELS end to end on the CPU: ``enable_{llama,mistral}_duo_attention_eval`` (tuple
    driver: tuple_kv_cache.py old_*_forward) and ``enable_*_duo_attention_static_kv_cache_eval`` (static driver:
    static_kv_cache.py:318-552 / :571-805, ``DuoAttentionStaticKVCache``, ``enable_flashinfer_rmsnorm``) on a tiny
    HF model, chunked prefill + decode [+ evict_last], last-token logits per call.

    Compatibility shims only: the HF-4.45 attention attributes the reference forwards read (num_heads,
    num_key_value_heads, hidden_size, rotary_emb, rope_theta) are added to transformers-5.5's modules, and
    ``flashinfer.norm.rmsnorm`` (CUDA-only) is served by its fp32 formula inside the reference's own
    ``flashinfer_rmsnorm_forward``."""
    import duo_attn.patch.flashinfer_utils as ref_fi
    from transformers.models.llama.modeling_llama import LlamaRotaryEmbedding
    from transformers.models.mistral.modeling_mistral import MistralRotaryEmbedding

    def rmsnorm(x, w, eps=1e-6):
        xf = x.float()
        return (xf * torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + eps) * w.float()).to(x.dtype)

    ref_fi.flashinfer = types.SimpleNamespace(norm=types.SimpleNamespace(rmsnorm=rmsnorm))
    for case in GC.MODEL_CASES:
        model, ids, wsum = GC.make_tiny_model(case)
        ref = ref_llama if case["kind"] == "llama" else ref_mistral
        Rot = LlamaRotaryEmbedding if case["kind"] == "llama" else MistralRotaryEmbedding
        for layer in model.model.layers:
            a = layer.self_attn
            a.num_heads, a.num_key_value_heads, a.hidden_size = 4, 2, 512
            a.rotary_emb = Rot(config=model.config)
            a.rope_theta = 10000.0
        if not hasattr(model.config, "rope_scaling"):
            model.config.rope_scaling = None
        gates = np.array(case["gates"])
        logits, lens = [], []
        if case["path"] == "tuple":
            getattr(ref, f"enable_{case['kind']}_duo_attention_eval")(model, gates, case["sink"], case["recent"])
            past = None
            for x in ids:
                out = model(input_ids=x, past_key_values=past, use_cache=True)
                past = out.past_key_values
                logits.append(out.logits.float())
                lens.append((past[0][0].shape[2], past[0][2].shape[2] if len(past[0]) > 2 else -1))
        else:
            getattr(ref, f"enable_{case['kind']}_duo_attention_static_kv_cache_eval")(model, gates)
            cache = ref.DuoAttentionStaticKVCache(model, gates, 1, case["max_size"], case["sink"], case["recent"])
            for i, x in enumerate(ids):
                out = model(input_ids=x, past_key_values=cache, use_cache=True)
                logits.append(out.logits.float())
                ev = case.get("evict_after", {}).get(i, 0)
                if ev:
                    cache.evict_last(ev)
                lens.append((cache.kv_seq_len, cache.streaming_kv_seq_len))
        assert all(l.shape == (1, 1, GC.MODEL_VOCAB) for l in logits), [l.shape for l in logits]
        np.savez_compressed(os.path.join(HERE, f"model_{case['name']}.npz"),
                            logits=torch.cat(logits, dim=1).numpy(), lens=np.array(lens, dtype=np.int64),
                            checksum=np.float64(wsum))
        print("wrote model", case["name"], "calls", len(ids), "lens", lens[-1])


def make_int4_fixtures(O, GC):
    """Run the reference's INT4 cache class (demo/int4_kv.py:115-492, unmodified) and its attention forward
    (demo/w8a8kv4_llama.py:174-287, unmodified, called unbound on a stand-in ``self``) on the CPU.

    Swapped, because they are CUDA-only / absent: ``torch.utils.cpp_extension.load`` returns a module whose two
    entry points are the NumPy restatement of demo/quantize_int4.cu (oracle/int4_oracle.py; pinned to the
    reference's compiled kernels on the GPU box by tests/test_gpu_kv_ops.py); ``flash_attn_func`` -> contract
    restatement; ``apply_rope_inplace`` -> identity (inputs are post-RoPE); QServe packages (qserve,
    qserve_backend) -> empty stubs, the W8A8 projections around the attention are no-ops on pre-filled buffers."""
    import torch.utils.cpp_extension as cpp

    from oracle import int4_oracle as Q

    class _K:
        @staticmethod
        def quantize_int4_with_zero_point_per_group(tensor, q_packed, scale, zero_point, group_size):
            assert group_size == 128
            p, s, z = Q.quantize_int4(tensor.detach().numpy())  # honours strides like quantize_int4.cu:163-165
            q_packed.copy_(torch.from_numpy(p))
            scale.copy_(torch.from_numpy(s))
            zero_point.copy_(torch.from_numpy(z))

        @staticmethod
        def dequantize_int4_with_zero_point_per_group(q_packed, scale, zero_point, group_size, buffer, N):
            assert q_packed.is_contiguous() and scale.is_contiguous() and zero_point.is_contiguous()  # raw data_ptr use
            out = Q.dequantize_int4(q_packed.numpy().reshape(N, 64), scale.numpy().reshape(N, 1),
                                    zero_point.numpy().reshape(N, 1))
            buffer[: N * group_size].copy_(torch.from_numpy(out).reshape(-1))

    real_load = cpp.load
    cpp.load = lambda *a, **k: _K
    class _Any(types.ModuleType):
        def __getattr__(self, item):
            if item.startswith("__"):
                raise AttributeError(item)
            return lambda *a, **k: None

    for name in ("qserve_backend", "qserve_backend.fused_attention", "qserve_backend.fused_kernels", "qserve",
                 "qserve.utils", "qserve.utils.constants", "qserve.modeling", "qserve.modeling.layers",
                 "qserve.modeling.layers.activation", "qserve.modeling.layers.layernorm",
                 "qserve.modeling.layers.quantized_linear", "qserve.modeling.layers.sampler", "qserve.sampling_params",
                 "qserve.utils.input_metadata", "qserve.utils.quant_config", "qserve.utils.weight_utils"):
        if name not in sys.modules:
            m = _Any(name)
            m.__path__ = []
            sys.modules[name] = m
            if "." in name:  # `import a.b.c` resolves a.b through attribute access on the parent module
                parent, _, leaf = name.rpartition(".")
                setattr(sys.modules[parent], leaf, m)
    try:
        import demo.int4_kv as ref_kv
        import demo.w8a8kv4_llama as ref_w8
    finally:
        cpp.load = real_load
    assert ref_kv.__file__.startswith(REF) and ref_w8.__file__.startswith(REF)
    ref_w8.flash_attn_func = O.flash_attn_contract
    ref_w8.apply_rope_inplace = lambda q, k, *a, **kw: (q, k)

    for case in GC.INT4_CASES:
        chunks = GC.make_int4_inputs(case)
        Hq, Hkv = case["Hq"], case["Hkv"]
        gate = [1.0] * case["n_full"] + [0.0] * (Hkv - case["n_full"])  # already "reordered": retrieval heads first
        holder = torch.nn.Linear(1, 1).to(torch.float16)
        model = types.SimpleNamespace(
            parameters=lambda: holder.parameters(),
            config=types.SimpleNamespace(num_hidden_layers=1, num_attention_heads=Hq, num_key_value_heads=Hkv,
                                         hidden_size=Hq * GC.D))
        cache = ref_kv.DuoAttentionStaticINT4KVCache(model, [gate], 1, case["max_size"], case["sink"], case["recent"],
                                                     case["prefill_chunk"])
        captured = {}
        me = types.SimpleNamespace(
            qkv_proj=lambda *a: None, o_proj=lambda *a: None, q_size=Hq * GC.D, kv_size=Hkv * GC.D, num_heads=Hq,
            num_kv_heads=Hkv, head_dim=GC.D, rope_theta=10000.0, layer_idx=0, hidden_size=Hq * GC.D,
            invoke_quant=lambda buf, attn: captured.__setitem__("out", attn.clone()))
        outs, lens = [], []
        for q, k, v in chunks:
            n = q.shape[1]
            buf = types.SimpleNamespace(
                quantized_hidden_states_buffer=None, quantized_scale_buffer=None, out_down_proj_act_buffer=None,
                qkv_proj_act_buffer=torch.cat([q.reshape(n, -1), k.reshape(n, -1), v.reshape(n, -1)], dim=-1),
                batched_seq_len=n)
            ref_w8.LlamaAttention.forward(me, types.SimpleNamespace(activation_buffer=buf), cache)
            outs.append(captured["out"].view(1, n, Hq, GC.D))
            lens.append((cache.kv_seq_len, cache.streaming_kv_seq_len))
        np.savez_compressed(os.path.join(HERE, f"layer_{case['name']}.npz"),
                            out=torch.cat(outs, dim=1).float().numpy(), lens=np.array(lens, dtype=np.int64),
                            checksum=np.float64(GC.int4_checksum(chunks)))
        print("wrote int4", case["name"], "tokens", sum(case["chunks"]), "final lens", lens[-1])

    # ---- the demo's enable function (demo/w8a8kv4_llama.py:659-729), unmodified, on a stand-in fused-qkv model ----
    Hq, Hkv, Dh, hid = 8, 4, 8, 24
    g = torch.Generator().manual_seed(77)
    gates = [[1.0, 0.0, 0.6, 0.2], [0.0, 0.0, 1.0, 1.0], [0.3, 0.9, 0.1, 0.7]]
    layers, before = [], []
    for _ in gates:
        qkv = types.SimpleNamespace(
            weight=types.SimpleNamespace(data=torch.randint(-128, 128, ((Hq + 2 * Hkv) * Dh, hid), generator=g,
                                                            dtype=torch.int8)),
            dequant_scale=torch.rand((Hq + 2 * Hkv) * Dh, generator=g).to(torch.float16))
        o = types.SimpleNamespace(weight=types.SimpleNamespace(data=torch.randint(-128, 128, (hid, Hq * Dh), generator=g,
                                                                                  dtype=torch.int8)))
        before.append((qkv.weight.data.clone(), qkv.dequant_scale.clone(), o.weight.data.clone()))
        attn = types.SimpleNamespace(qkv_proj=qkv, o_proj=o, q_size=Hq * Dh, kv_size=Hkv * Dh, num_heads=Hq,
                                     num_kv_heads=Hkv, head_dim=Dh)
        attn.register_buffer = lambda name, t, a=attn: setattr(a, name, t)
        layers.append(types.SimpleNamespace(self_attn=attn))
    holder = torch.nn.Linear(1, 1).to(torch.float16)
    model = types.SimpleNamespace(parameters=lambda: holder.parameters(), model=types.SimpleNamespace(layers=layers))
    ref_w8.enable_llama_duo_attention_eval(model, gates, 64, 256)
    np.savez_compressed(
        os.path.join(HERE, "w8a8kv4_enable.npz"), gates=np.array(gates),
        **{f"qkv_w_in_{i}": b[0].numpy() for i, b in enumerate(before)},
        **{f"qkv_s_in_{i}": b[1].numpy() for i, b in enumerate(before)},
        **{f"o_w_in_{i}": b[2].numpy() for i, b in enumerate(before)},
        **{f"qkv_w_{i}": l.self_attn.qkv_proj.weight.data.numpy() for i, l in enumerate(layers)},
        **{f"qkv_s_{i}": l.self_attn.qkv_proj.dequant_scale.numpy() for i, l in enumerate(layers)},
        **{f"o_w_{i}": l.self_attn.o_proj.weight.data.numpy() for i, l in enumerate(layers)},
        **{f"heads_{i}": l.self_attn.full_attention_heads.float().numpy() for i, l in enumerate(layers)})
    print("wrote w8a8kv4_enable (sink/recent attrs:", layers[0].self_attn.sink_size, layers[0].self_attn.recent_size, ")")


def make_training_mask_fixtures(GC):
    """The reference's training-time streaming mask and its SDPA streaming attention, run unmodified on the CPU
    (duo_attn/patch/streaming_attn.py:14-42; the module imports without its optional CUDA packages)."""
    sys.path.insert(0, REF)
    import importlib.util

    spec = importlib.util.spec_from_file_location("ref_streaming_attn", os.path.join(REF, "duo_attn/patch/streaming_attn.py"))
    sa = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(sa)
    out = {}
    for case in GC.TRAIN_MASK_CASES:
        q, k, v = GC.make_train_mask_inputs(case)
        mask = sa.generate_streaming_mask(case["S"], case["sink"], case["recent"], "cpu")
        o = sa.streaming_attn_sdpa(q, k, v, mask)
        out[f"mask_{case['name']}"] = mask[0, 0].numpy()
        out[f"out_{case['name']}"] = o.numpy().astype(np.float32)
        out[f"checksum_{case['name']}"] = np.float64(sum(float(t.double().abs().sum()) for t in (q, k, v)))
    np.savez_compressed(os.path.join(HERE, "training_masks.npz"), **out)
    print("wrote training masks", len(GC.TRAIN_MASK_CASES))


def make_int4_kernel_fixture(GC, out_dir):
    """The reference's INT4 quantise (K1) and dequantise (K2) kernels of demo/quantize_int4.cu, built with its own flags
    (--use_fast_math) into oracle/_ref/ by oracle/build_ref.py, on GC.make_int4_kernel_input().  Needs a GPU.  K1's
    packed codes, scales and zeros are kept for every row; K2's dequantisation of them (614 KB of fp16) is kept as the
    SHA-256 of its bytes, which the tests compare bit for bit."""
    import hashlib

    from oracle import build_ref

    ref = build_ref.load_module()
    assert ref is not None, "oracle/_ref/ not built: python oracle/build_ref.py"
    x = GC.make_int4_kernel_input()
    rows_n = x.size // 128
    dev = torch.device("cuda:0")
    xt = torch.from_numpy(x).to(dev)
    qp = torch.empty(*x.shape[:-1], 64, dtype=torch.uint8, device=dev)
    sc = torch.empty(*x.shape[:-1], 1, dtype=torch.float16, device=dev)
    zp = torch.empty(*x.shape[:-1], 1, dtype=torch.float16, device=dev)
    ref.quantize_int4_with_zero_point_per_group(xt, qp, sc, zp, 128)
    buf = torch.empty(rows_n * 128, dtype=torch.float16, device=dev)
    ref.dequantize_int4_with_zero_point_per_group(qp.view(-1, 64), sc, zp, 128, buf, rows_n)
    torch.cuda.synchronize()
    np.savez_compressed(
        os.path.join(out_dir, "int4_ref_kernels.npz"),
        packed=qp.view(-1, 64).cpu().numpy(), scale=sc.view(-1).cpu().numpy(), zero=zp.view(-1).cpu().numpy(),
        dequant_sha256=np.str_(hashlib.sha256(buf.view(-1, 128).cpu().numpy().tobytes()).hexdigest()),
        checksum=np.float64(np.abs(x.astype(np.float64)).sum()))
    print("wrote int4_ref_kernels,", rows_n, "rows")


def main():
    from oracle import duo_oracle as O
    import golden_cases as GC

    if sys.argv[1:] == ["masks"]:
        return make_training_mask_fixtures(GC)
    if sys.argv[1:2] == ["int4-kernels"]:
        return make_int4_kernel_fixture(GC, sys.argv[2] if len(sys.argv) > 2 else HERE)

    ref_llama, ref_mistral, ref_putils, ref_utils = import_reference()
    assert ref_llama.__file__.startswith(REF), ref_llama.__file__

    # swap the CUDA-only third-party calls for the contract restatements
    ref_llama.flash_attn_func = O.flash_attn_contract

    def rope_inplace(q, k, offsets, rope_scale, rope_theta, indptr=None):
        q2, k2 = O.rope_flashinfer(q, k, int(offsets.reshape(-1)[0]), rope_scale, rope_theta)
        q.copy_(q2)
        k.copy_(k2)
        return q, k

    ref_llama.apply_rope_inplace = rope_inplace
    ref_mistral.flash_attn_func = O.flash_attn_contract
    ref_mistral.apply_rope_inplace = rope_inplace

    # ---------------------------------------------------------------- attention-layer fixtures
    for case in GC.LAYER_CASES:
        name = case["name"]
        data = GC.make_layer_inputs(case)
        mod = GC.RefAttnModule(case, data, ref_putils)  # reference reorder functions run inside
        outs = []
        if case["path"] == "tuple":
            past = None
            pos = 0
            for hs in data["chunks"]:
                S = hs.shape[1]
                position_ids = torch.arange(pos, pos + S)[None]
                out, _, past = ref_llama.llama_duo_attention_forward_one_way_reordered(
                    mod, hs, position_ids=position_ids, past_key_value=past, use_cache=True)
                outs.append(out)
                pos += S
            extra = dict(final_full_len=past[0].shape[2], final_stream_len=past[1].shape[2])
        else:
            fake_model = GC.FakeModel(case, mod)
            cache = ref_llama.DuoAttentionStaticKVCache(
                fake_model, [data["gate"].numpy()], data["B"], case["max_size"], case["sink"], case["recent"])
            pos = 0
            for i, hs in enumerate(data["chunks"]):
                S = hs.shape[1]
                position_ids = torch.arange(pos, pos + S)[None]
                out, _ = ref_llama.llama_duo_attention_forward_one_way_reordered_static(
                    mod, hs, position_ids=position_ids, kv_cache=cache, layer_idx=0)
                outs.append(out)
                pos += S
                ev = case.get("evict_after", {}).get(i, 0)
                if ev:
                    cache.evict_last(ev)
                    pos -= ev
            extra = dict(final_full_len=cache.kv_seq_len, final_stream_len=cache.streaming_kv_seq_len)
        np.savez_compressed(
            os.path.join(HERE, f"layer_{name}.npz"),
            out=torch.cat(outs, dim=1).numpy().astype(np.float32),
            checksum=np.float64(GC.checksum(data)),
            **{k: np.int64(v) for k, v in extra.items()},
        )
        print("wrote layer", name, "tokens", sum(c.shape[1] for c in data["chunks"]), extra)
        # the Mistral twin (duo_attn/patch/mistral.py:146-434): same cases through the reference's mistral
        # forwards; SURVEY §2.1 found the two files identical modulo names — pinned here by running both.
        if name in GC.MISTRAL_CASES:
            mod = GC.RefAttnModule(case, data, ref_putils)
            outs_m = []
            if case["path"] == "tuple":
                past, pos = None, 0
                for hs in data["chunks"]:
                    S = hs.shape[1]
                    out, _, past = ref_mistral.mistral_duo_attention_forward_one_way_reordered(
                        mod, hs, position_ids=torch.arange(pos, pos + S)[None], past_key_value=past, use_cache=True)
                    outs_m.append(out)
                    pos += S
            else:
                cache = ref_mistral.DuoAttentionStaticKVCache(
                    GC.FakeModel(case, mod), [data["gate"].numpy()], data["B"], case["max_size"], case["sink"],
                    case["recent"])
                pos = 0
                for i, hs in enumerate(data["chunks"]):
                    S = hs.shape[1]
                    out, _ = ref_mistral.mistral_duo_attention_forward_one_way_reordered_static(
                        mod, hs, position_ids=torch.arange(pos, pos + S)[None], kv_cache=cache, layer_idx=0)
                    outs_m.append(out)
                    pos += S
                    ev = case.get("evict_after", {}).get(i, 0)
                    if ev:
                        cache.evict_last(ev)
                        pos -= ev
            same = torch.equal(torch.cat(outs_m, dim=1), torch.cat(outs, dim=1))
            np.savez_compressed(os.path.join(HERE, f"layer_mistral_{name}.npz"),
                                out=torch.cat(outs_m, dim=1).numpy().astype(np.float32),
                                identical_to_llama=np.bool_(same), checksum=np.float64(GC.checksum(data)))
            print("wrote mistral twin", name, "identical to llama:", same)

    # ---------------------------------------------------------------- model-level driver fixtures
    make_model_fixtures(O, GC, ref_llama, ref_mistral)

    # ---------------------------------------------------------------- INT4-KV fixtures
    make_int4_fixtures(O, GC)

    # ---------------------------------------------------------------- training-time streaming masks
    make_training_mask_fixtures(GC)

    # ---------------------------------------------------------------- reorder fixtures
    for case in GC.REORDER_CASES:
        torch.manual_seed(case["seed"])
        lin = torch.nn.Linear(case["in"], case["out"], bias=case["bias"])
        gate = torch.tensor(case["gate"], dtype=torch.float32)
        w0 = lin.weight.data.clone()
        b0 = None if lin.bias is None else lin.bias.data.clone()
        ref_putils.reorder_linear_weights(lin, gate, case["repeat"], case["channel"])
        g2 = ref_putils.reorder_full_attn_heads(gate.clone())
        np.savez_compressed(
            os.path.join(HERE, f"reorder_{case['name']}.npz"),
            w_in=w0.numpy(), w_out=lin.weight.data.numpy(),
            b_in=np.zeros(0) if b0 is None else b0.numpy(),
            b_out=np.zeros(0) if lin.bias is None else lin.bias.data.numpy(),
            gate_out=g2.numpy(),
        )
        print("wrote reorder", case["name"])

    # ---------------------------------------------------------------- tensor-parallel sharding rules
    if ref_utils is not None:
        # get_mistral_config (duo_attn/utils.py:132-195) builds a tensor_parallel.Config out of third-party rule objects
        # (package absent here): run it with recording stand-ins and keep the table it produces + the buffer rule
        # to_device adds (:219-221).  tests/test_tp_gloo.py holds tp.shard_model to it.
        rec = lambda kind: (lambda **kw: dict(kind=kind, **kw))
        ref_utils.Split, ref_utils.SplitInChunks = rec("Split"), rec("SplitInChunks")
        ref_utils.CollectiveOperation = lambda **kw: "collective"
        import re as _re

        # like tensor_parallel.Config, keys become compiled patterns (utils.py:189 indexes attr_rules with one)
        ref_utils.Config = lambda **kw: types.SimpleNamespace(
            **{name: {_re.compile(k): v for k, v in table.items()} for name, table in kw.items()})
        mcfg = types.SimpleNamespace(model_type="mistral", hidden_size=4096, num_attention_heads=32,
                                     num_key_value_heads=8)
        c = ref_utils.get_mistral_config(mcfg, ["cuda:0", "cuda:1", "cuda:2", "cuda:3"])
        rules = dict(
            state_rules={k.pattern: v for k, v in c.state_rules.items()},
            output_rules={k.pattern: {str(i): (o if isinstance(o, str) else "gather_kv") for i, o in v.items()}
                          for k, v in c.output_rules.items()},
            attr_rules={k.pattern: sorted(v) for k, v in c.attr_rules.items()},
            buffer_rule={r".*full_attention_heads$": dict(kind="Split", dim=0)},  # to_device, utils.py:219-221
        )
        with open(os.path.join(HERE, "tp_rules.json"), "w") as f:
            json.dump(rules, f, indent=1, sort_keys=True)
        print("wrote tp rules", len(rules["state_rules"]))

    # ---------------------------------------------------------------- pattern fixtures
    if ref_utils is not None:
        res = {}
        pat_root = os.path.join(REF, "attn_patterns")
        for model in sorted(os.listdir(pat_root)):
            run = sorted(os.listdir(os.path.join(pat_root, model)))[0]
            d = os.path.join(pat_root, model, run)
            for sparsity in (0.0, 0.25, 0.5, 0.75, 1.0):
                h, sink, recent = ref_utils.load_attn_pattern(d)
                np.random.seed(42)
                mask, true_sp = ref_utils.sparsify_attention_heads(h, None, sparsity)
                res[f"{model}|{sparsity}"] = dict(
                    dir=os.path.join("attn_patterns", model, run), sink=sink, recent=recent,
                    shape=list(mask.shape), per_layer_full=mask.sum(1).astype(int).tolist(),
                    mask_rows=["".join(str(int(v)) for v in row) for row in mask], true_sparsity=float(true_sp),
                    clipped_sum=float(np.clip(np.loadtxt(os.path.join(d, "full_attention_heads.tsv")), 0, 1).sum()),
                )
        with open(os.path.join(HERE, "patterns.json"), "w") as f:
            json.dump(res, f, indent=1, sort_keys=True)
        print("wrote patterns", len(res))


if __name__ == "__main__":
    with torch.no_grad():
        main()
