"""Same-box GPU baseline: the reference's static-cache DuoAttention forward restated with the libraries it calls.

What the reference runs on a GPU for its efficiency numbers (eval/efficiency/benchmark_static.py:58-103) is

  * the static driver loop                    duo_attn/patch/static_kv_cache.py:318-567
  * the static attention forward              duo_attn/patch/llama.py:309-434  (q/k/v projections as three GEMMs,
    flashinfer RoPE in place, append to token-major caches, TWO flash_attn_func calls + torch.cat, o_proj)
  * DuoAttentionStaticKVCache                 duo_attn/patch/static_kv_cache.py:18-315 (token-major [B, S, H, D] buffers,
    put_full_kv copy, compress_and_replace_streaming_kv compaction copies)
  * flashinfer RMSNorm                        duo_attn/patch/flashinfer_utils.py:9-16

The reference package itself does not import under the installed transformers (SURVEY.md §8c), so this file restates
that algorithm — same tensor layouts, same library calls (the INSTALLED flash_attn_func / flashinfer), same number of
copies — on the weights of an already patched model (the retrieval-first reorder is the reference's own,
patch/utils.py:6-45).  It exists ONLY as the baseline arm of bench.py (`reference_gpu_same_box` in the bench line): none
of it is on the product path, and none of our kernels is on its path.  Timed with the reference's bench protocol
(eval/efficiency/utils.py:7-30: warm-up, CUDA events around N calls; decode step + evict_last(1))."""
from __future__ import annotations

import torch


class RefStaticCache:
    """Token-major static cache with the reference's put / compaction semantics."""

    def __init__(self, n_full_list, n_kv, head_dim, max_size, sink, recent, dtype, device):
        self.sink, self.recent, self.max_size = sink, recent, max_size
        self.n_full = list(n_full_list)
        W = sink + recent
        self.fk = [torch.zeros(1, max_size, nf, head_dim, dtype=dtype, device=device) for nf in self.n_full]
        self.fv = [torch.zeros(1, max_size, nf, head_dim, dtype=dtype, device=device) for nf in self.n_full]
        self.sk = [torch.zeros(1, W, n_kv - nf, head_dim, dtype=dtype, device=device) for nf in self.n_full]
        self.sv = [torch.zeros(1, W, n_kv - nf, head_dim, dtype=dtype, device=device) for nf in self.n_full]
        self.full_len = [0] * len(self.n_full)
        self.stream_len = [0] * len(self.n_full)

    @property
    def kv_seq_len(self):
        return self.full_len[-1]

    def clear(self):
        self.full_len = [0] * len(self.n_full)
        self.stream_len = [0] * len(self.n_full)

    def evict_last(self, n):
        self.full_len = [max(0, x - n) for x in self.full_len]
        self.stream_len = [max(0, x - n) for x in self.stream_len]

    def put_full(self, l, k, v):
        n, cur = k.shape[1], self.full_len[l]
        if n + cur > self.max_size:
            raise ValueError(f"Trying to put {n} KVs into a cache with max size {self.max_size}, current size: {cur}.")
        self.fk[l][:, cur : cur + n].copy_(k)
        self.fv[l][:, cur : cur + n].copy_(v)
        self.full_len[l] = cur + n
        return self.fk[l][:, : cur + n], self.fv[l][:, : cur + n]

    def streaming(self, l):
        n = self.stream_len[l]
        return self.sk[l][:, :n], self.sv[l][:, :n]

    def compress(self, l, k, v):
        """Keep sinks + the last `recent` rows of [cached | new] (static_kv_cache.py:127-167)."""
        n, W = k.shape[1], self.sink + self.recent
        if n <= W:
            self.sk[l][:, :n].copy_(k)
            self.sv[l][:, :n].copy_(v)
            self.stream_len[l] = n
        else:
            self.sk[l][:, : self.sink].copy_(k[:, : self.sink])
            self.sv[l][:, : self.sink].copy_(v[:, : self.sink])
            self.sk[l][:, self.sink :].copy_(k[:, n - self.recent :])
            self.sv[l][:, self.sink :].copy_(v[:, n - self.recent :])
            self.stream_len[l] = W


class RefRunner:
    def __init__(self, model, n_full_list, sink, recent, max_size):
        from flash_attn import flash_attn_func

        self.fa = flash_attn_func
        self.model = model
        cfg = model.config
        self.Hq, self.Hkv = cfg.num_attention_heads, cfg.num_key_value_heads
        self.D = getattr(cfg, "head_dim", None) or cfg.hidden_size // cfg.num_attention_heads
        self.G = self.Hq // self.Hkv
        p = next(model.parameters())
        self.dev = p.device
        self.cache = RefStaticCache(n_full_list, self.Hkv, self.D, max_size, sink, recent, p.dtype, p.device)
        self.theta = float(getattr(cfg, "rope_theta", None) or cfg.rope_parameters["rope_theta"])
        self.rope = "flashinfer.rope.apply_rope_inplace"
        self.norm = "flashinfer.norm.rmsnorm"
        try:
            import flashinfer

            self.fi = flashinfer
            q = torch.zeros(1, self.Hq, self.D, dtype=p.dtype, device=p.device)
            k = torch.zeros(1, self.Hkv, self.D, dtype=p.dtype, device=p.device)
            flashinfer.rope.apply_rope_inplace(q, k, torch.tensor([0, 1], dtype=torch.int32, device=p.device),
                                               torch.zeros(1, dtype=torch.int32, device=p.device), interleave=False,
                                               rope_scale=1.0, rope_theta=self.theta)
        except Exception:  # JIT compile unavailable on the box: HF table RoPE in torch (same cost class)
            self.fi, self.rope = None, "torch (HF tables)"
        try:
            if self.fi is None:
                raise RuntimeError
            self.fi.norm.rmsnorm(torch.zeros(1, cfg.hidden_size, dtype=p.dtype, device=p.device),
                                 model.model.norm.weight, 1e-5)
        except Exception:
            self.norm = "HF LlamaRMSNorm (torch)"

    def _rms(self, mod, x):
        if self.norm.startswith("flashinfer"):
            s = x.shape
            return self.fi.norm.rmsnorm(x.reshape(-1, s[-1]), mod.weight, mod.variance_epsilon).view(s)
        return mod(x)

    def _attention(self, l, attn, x, pos0):
        B, S, _ = x.shape
        c = self.cache
        q = attn.q_proj(x).view(B, S, self.Hq, self.D)
        k = attn.k_proj(x).view(B, S, self.Hkv, self.D)
        v = attn.v_proj(x).view(B, S, self.Hkv, self.D)
        if self.fi is not None:
            # the reference builds indptr with a host->device torch.tensor on every call (flashinfer_utils.py:42-45)
            indptr = torch.tensor([0, S], dtype=torch.int32, device=x.device)
            off = torch.full((1,), pos0, dtype=torch.int32, device=x.device)
            self.fi.rope.apply_rope_inplace(q.view(S, self.Hq, self.D), k.view(S, self.Hkv, self.D), indptr, off,
                                            interleave=False, rope_scale=1.0, rope_theta=self.theta)
        else:
            from transformers.models.llama.modeling_llama import apply_rotary_pos_emb

            pos = torch.arange(pos0, pos0 + S, device=x.device)[None]
            cos, sin = self.model.model.rotary_emb(x, pos)
            q, k = apply_rotary_pos_emb(q, k, cos, sin, unsqueeze_dim=2)
        nf = c.n_full[l]
        first = c.full_len[l] == 0
        fk, fv = c.put_full(l, k[:, :, :nf], v[:, :, :nf])
        sk, sv = k[:, :, nf:], v[:, :, nf:]
        if first:
            out = self.fa(q, k, v, causal=True, dropout_p=0.0)
        else:
            ck, cv = c.streaming(l)
            sk, sv = torch.cat([ck, sk], dim=1), torch.cat([cv, sv], dim=1)
            parts = []
            if nf > 0:
                parts.append(self.fa(q[:, :, : nf * self.G], fk, fv, causal=True, dropout_p=0.0))
            if nf < self.Hkv:
                parts.append(self.fa(q[:, :, nf * self.G :], sk, sv, causal=True, dropout_p=0.0))
            out = parts[0] if len(parts) == 1 else torch.cat(parts, dim=2)
        c.compress(l, sk, sv)
        return attn.o_proj(out.reshape(B, S, self.Hq * self.D))

    @torch.no_grad()
    def forward(self, ids):
        m = self.model.model
        pos0 = self.cache.kv_seq_len
        h = m.embed_tokens(ids)
        for l, layer in enumerate(m.layers):
            h = h + self._attention(l, layer.self_attn, self._rms(layer.input_layernorm, h), pos0)
            x = self._rms(layer.post_attention_layernorm, h)
            mlp = layer.mlp
            h = h + mlp.down_proj(torch.nn.functional.silu(mlp.gate_proj(x)) * mlp.up_proj(x))
        return self.model.lm_head(self._rms(m.norm, h[:, -1:, :]))


def fill_synthetic(cache: RefStaticCache, ctx):
    g = torch.Generator(device=cache.fk[0].device).manual_seed(7)
    for t in cache.fk + cache.fv + cache.sk + cache.sv:
        if t.numel():
            t.normal_(generator=g)
    cache.full_len = [ctx] * len(cache.n_full)
    cache.stream_len = [cache.sink + cache.recent] * len(cache.n_full)


def run(model, n_full_list, sink, recent, ctx, prefill_ctx, chunk, vocab, decode_steps=10, decode_warmup=3,
        do_prefill=True):
    """-> dict with the reference arm's end-to-end decode tokens/s at `ctx` and prefill tokens/s at `prefill_ctx`."""
    dev = next(model.parameters()).device
    r = RefRunner(model, n_full_list, sink, recent, max(ctx, prefill_ctx) + 8)
    res = {"what": "duo_attn/patch/llama.py:309-434 + static_kv_cache.py restated with the installed flash_attn_func "
                   f"(token-major caches, 2 FA2 calls + cat, compaction copies), eager; rope: {r.rope}; rmsnorm: {r.norm}",
           "protocol": f"eval/efficiency/utils.py bench_func (CUDA events); decode: {decode_warmup} warm-up + "
                       f"{decode_steps} steps with evict_last(1); prefill: 1 rep after a one-chunk warm-up"}
    g = torch.Generator().manual_seed(1)
    if do_prefill:
        ids = torch.randint(0, vocab, (1, prefill_ctx), generator=g).to(dev)
        r.forward(ids[:, :chunk])
        r.cache.clear()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(0, prefill_ctx, chunk):
            out = r.forward(ids[:, i : i + chunk])
        int(out[:, -1].argmax(-1).item())
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        res["prefill"] = {"value": prefill_ctx / (ms / 1e3), "unit": "tokens/s", "ms_per_prefill": ms}
    fill_synthetic(r.cache, ctx)
    tok = torch.randint(0, vocab, (1, 1), generator=g).to(dev)

    def step():
        r.forward(tok)
        r.cache.evict_last(1)

    for _ in range(decode_warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(decode_steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / decode_steps
    res["decode"] = {"value": 1e3 / ms, "unit": "tokens/s", "ms_per_step": ms, "ctx": ctx}
    del r
    torch.cuda.empty_cache()
    return res
