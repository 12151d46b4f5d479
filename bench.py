#!/usr/bin/env python
"""Benchmark of the DuoAttention hot path on B200 (contract: see the task statement / DESIGN.md §Measurement).

Workload (BASELINE.json configs[1] + the metric's 1M-context decode point):
  Llama-3-8B-Instruct-Gradient-1048k architecture, random-init bf16 weights, real head pattern
  attn_patterns/Llama-3-8B-Instruct-Gradient-1048k/... at sparsity 0.5 (128 retrieval + 128 streaming KV heads),
  deploy-time sink=64 / recent=256, batch 1, synthetic random token ids.
    * decode  : one token per step against a synthetically filled 1,048,576-token KV cache (evict_last(1) after
                every step, the reference's benchmark_static.py:96-103 protocol)  -> `value` (tokens/s)
    * prefill : 131,072 tokens in chunks of 32,768 through the same patched model        -> `prefill` object

One process per GPU (`torchrun` for N > 1).  Prefill: KV heads are sharded across ranks (head-parallel TP, the reference's
rule: one all-reduce on the attention output and one on the MLP output per layer).  Decode: retrieval heads are
SEQUENCE-sharded (every rank streams 1/N of every retrieval head; one peer-memory exchange of the (O, lse) partials per
layer, fused one-shot all-reduce for the MLP), reached from the prefill layout by a timed reshard.  Total work is fixed
-> "strong".

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--ctx 1048576] [--prefill-ctx 131072]
                  [--dump-outputs DIR]

--dump-outputs DIR writes the logits the timed prefill and decode returned in their last repetition / step as
DIR/prefill_logits.npy and DIR/decode_logits.npy (float32).  Weights, token ids and the synthetic cache come from fixed
seeds, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

def pattern_dir(name):
    base = os.path.join(ROOT, "attn_patterns", name)
    return os.path.join(base, sorted(os.listdir(base))[0])
L3_8B = dict(hidden_size=4096, num_attention_heads=32, num_key_value_heads=8, head_dim=128, num_hidden_layers=32,
             intermediate_size=14336, vocab_size=128256, rms_norm_eps=1e-5, rope_theta=3580165449.0,
             max_position_embeddings=1048576)
ARCHS = {
    # name: (model-config overrides, default attention pattern)  — dimensions from the public HF configs (SURVEY §8)
    "llama3-8b-1048k": (dict(), "Llama-3-8B-Instruct-Gradient-1048k"),
    "llama3-8b-4194k": (dict(rope_theta=45315059621.0, max_position_embeddings=4194304),
                        "Llama-3-8B-Instruct-Gradient-4194k"),
    "mistral-7b-v0.3": (dict(vocab_size=32768, rope_theta=1000000.0, max_position_embeddings=32768),
                        "Mistral-7B-Instruct-v0.3"),
    "llama2-7b-32k": (dict(num_key_value_heads=32, intermediate_size=11008, vocab_size=32000, rope_theta=10000.0,
                           max_position_embeddings=32768), "Llama-2-7B-32K-Instruct"),
}
SINK, RECENT = 64, 256


def ncu_traffic(kind):
    """DRAM traffic of the dominant kernel from THIS round's `ncu --set full` capture (profiles/r2_traffic.json, written by
    profiles/summarize.py from the .ncu-rep of profiles/capture.sh): {"dram_bytes": read+write of the captured launch,
    "algorithmic_bytes": algorithmic bytes of that same launch}.  None if the capture has not been summarised."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))[kind]
        return d
    except Exception:
        return None

METRIC = "decode tok/s @1M ctx (+ prefill tok/s @128K in `prefill`), Llama-3-8B, DuoAttention 50% retrieval heads"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ctx", type=int, default=1048576)
    ap.add_argument("--prefill-ctx", type=int, default=131072)
    ap.add_argument("--chunk", type=int, default=32768)
    ap.add_argument("--prefill-reps", type=int, default=2)
    ap.add_argument("--layers", type=int, default=32, help="debug only: a run with fewer layers is not a valid number")
    ap.add_argument("--kv-format", default="bf16", choices=["bf16", "int4"],
                    help="int4 = BASELINE configs[3]: fp16 activations, INT4 KV with fused dequant (linears stay 16-bit: "
                         "the reference's W8A8 linears are QServe's, absent here)")
    ap.add_argument("--arch", default="llama3-8b-1048k", choices=sorted(ARCHS),
                    help="other BASELINE configs (parity-test architectures); the headline line is the default")
    ap.add_argument("--pattern", default=None, help="attn_patterns/<name>; default: the architecture's own")
    ap.add_argument("--sparsity", type=float, default=0.5)
    ap.add_argument("--no-prefill", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fa2", action="store_true", help="skip the same-box FlashAttention-2 micro-comparison")
    ap.add_argument("--no-graph", action="store_true", help="drive decode eagerly instead of replaying a CUDA graph")
    ap.add_argument("--prefill-only", action="store_true", help="tuning: stop after the prefill (+ reshard) measurement")
    ap.add_argument("--tp-pipeline-blocks", type=int, default=None,
                    help="N > 1 prefill: row blocks of the pipelined all-reduce (0 = plain NCCL all-reduce per site)")
    ap.add_argument("--profile-step", action="store_true",
                    help="after the timed regions: kernel table (torch.profiler / CUPTI, rank 0) of eager decode steps -> "
                         "gpurun_out/profile_step_n<N>.txt; never used for a bench value")
    ap.add_argument("--head-tp-decode", action="store_true",
                    help="N > 1: decode head-parallel like the reference's TP rule instead of sequence-sharded (A/B)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed regions: write the logits of the last timed prefill and decode step to DIR "
                         "(--impl ours only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours: the reference arm extrapolates timings and returns no outputs")
    if args.pattern is None:
        args.pattern = ARCHS[args.arch][1]
    return args


def head_pattern(name="Llama-3-8B-Instruct-Gradient-1048k", sparsity=0.5):
    import numpy as np

    from duo_attn.utils import load_attn_pattern, sparsify_attention_heads

    gates, _, _ = load_attn_pattern(pattern_dir(name))
    np.random.seed(42)
    mask, sp = sparsify_attention_heads(gates, None, sparsity)
    return mask, float(sp)


def decode_bytes_per_token(mask, ctx, row_bytes=256):
    """Algorithmic K+V bytes one decode step must read (BASELINE.md §4): retrieval heads read ctx+1 rows,
    streaming heads sink+recent+1; a row is 256 B (bf16) or 64+2+2 = 68 B (INT4 + fp16 scale/zero)."""
    n_f = mask.sum(1)
    n_s = mask.shape[1] - n_f
    return float(((n_f * (ctx + 1) + n_s * (SINK + RECENT + 1)) * 2 * row_bytes).sum())


def prefill_flops(mask, n_ctx, chunk, G=4, D=128):  # G = q heads per kv head of the architecture
    """Algorithmic attention FLOPs (4*D per visible (q,k) pair per q-head; masked halves not credited)."""
    W = SINK + RECENT
    full_pairs = n_ctx * (n_ctx + 1) // 2
    stream_pairs = 0
    for cs in range(0, n_ctx, chunk):
        c = min(chunk, n_ctx - cs)
        past = cs if cs <= W else W
        stream_pairs += c * past + c * (c + 1) // 2
    n_f = int(mask.sum())
    n_s = mask.size - n_f
    return 4.0 * D * G * (n_f * full_pairs + n_s * stream_pairs)


# --------------------------------------------------------------------------------------------------
# CPU reference arm (the oracle port of the reference forward, timed on the host cores)
# --------------------------------------------------------------------------------------------------
def cpu_reference_sample(ctx, mask, threads=None):
    """Time a bounded sample of ONE decode step of the reference's forward on the host: the attention of one
    retrieval KV head (its 4 q-heads against ctx keys), one streaming KV head (321 keys) and one layer's
    linear projections + MLP; scale to the whole model (128 + 128 KV heads, 32 layers).  Returns tokens/s."""
    import torch

    from oracle import duo_oracle as O

    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(0)
    D, G = 128, 4
    q = torch.randn(1, 1, G, D, generator=g).to(torch.bfloat16)
    k = torch.randn(1, ctx + 1, 1, D, generator=g).to(torch.bfloat16)
    v = torch.randn(1, ctx + 1, 1, D, generator=g).to(torch.bfloat16)
    samples = []
    for _ in range(3):  # median of three: one cold sample swings 4x between boxes
        t0 = time.perf_counter()
        O.flash_attn_contract(q, k, v, causal=True)
        samples.append(time.perf_counter() - t0)
    t_full = sorted(samples)[1]
    ks, vs = k[:, : SINK + RECENT + 1], v[:, : SINK + RECENT + 1]
    t0 = time.perf_counter()
    for _ in range(10):
        O.flash_attn_contract(q, ks, vs, causal=True)
    t_stream = (time.perf_counter() - t0) / 10
    # one layer of bf16 GEMVs: qkv (6144x4096), o (4096x4096), gate/up (2x14336x4096), down (4096x14336)
    x = torch.randn(1, 4096).to(torch.bfloat16)
    ws = [torch.randn(n, m).to(torch.bfloat16) for n, m in ((6144, 4096), (4096, 4096), (28672, 4096))]
    wd = torch.randn(4096, 14336).to(torch.bfloat16)
    t0 = time.perf_counter()
    for w in ws:
        torch.nn.functional.linear(x, w)
    torch.nn.functional.linear(torch.randn(1, 14336).to(torch.bfloat16), wd)
    t_lin = time.perf_counter() - t0
    n_f, n_s = int(mask.sum()), int(mask.size - mask.sum())
    step_s = n_f * t_full + n_s * t_stream + mask.shape[0] * t_lin
    return dict(tok_s=1.0 / step_s, t_full_head_s=t_full, t_stream_head_s=t_stream, t_layer_linear_s=t_lin,
                step_s_extrapolated=step_s, cores=threads)


def run_reference(args):
    """`--impl reference`: the reference's CPU path (oracle port; the reference package has no CPU attention of
    its own and no tests — SURVEY.md §0/§4) on all host threads, same metric/config as our arm."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    mask, sp = head_pattern(args.pattern, args.sparsity)
    for _ in range(args.warmup):
        cpu_reference_sample(args.ctx, mask)
    vals = []
    for _ in range(args.steps):  # one sample = one extrapolated decode step
        vals.append(cpu_reference_sample(args.ctx, mask))
    best = sorted(vals, key=lambda r: r["tok_s"])[len(vals) // 2]  # median of the samples, not the best
    line = {
        "impl": "reference", "metric": METRIC, "value": best["tok_s"], "unit": "tokens/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / best["tok_s"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args, sp),
        "cpu_baseline": {"value": best["tok_s"], "unit": "tokens/s", "cores": best["cores"], "kind": "port",
                         "sample": "1 retrieval KV head @ctx + 1 streaming KV head + 1 layer of linears, "
                                   "extrapolated to 128+128 heads x 32 layers", **{k: best[k] for k in
                                   ("t_full_head_s", "t_stream_head_s", "t_layer_linear_s")}},
        "e2e": {"value": best["tok_s"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_config(args, sparsity):
    return {
        "workload": f"{args.arch} arch (random init, 16-bit), DuoAttention pattern {args.pattern} sparsity "
                    f"{sparsity:.2f}, sink {SINK}/recent {RECENT}, batch 1: decode @ctx={args.ctx} "
                    f"(evict_last(1) per step) + prefill {args.prefill_ctx} tokens in chunks of {args.chunk}",
        "pattern": args.pattern, "kv_format": args.kv_format, "ctx": args.ctx, "prefill_ctx": args.prefill_ctx, "chunk": args.chunk, "layers": args.layers,
        "parallelism": (f"prefill head-tp{args.gpus}, decode sequence-sharded retrieval heads x{args.gpus} "
                        f"(attention replicated, MLP tp{args.gpus})") if args.gpus > 1 and args.kv_format == "bf16"
                       and not getattr(args, "head_tp_decode", False) else f"head-tp{args.gpus}",
        "l2": "inputs larger than L2: every decode step streams >2 GB of KV per layer (126 MB L2), "
              "prefill chunks stream the whole KV cache",
    }


# --------------------------------------------------------------------------------------------------
# clocks sampling
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, dev_index):
        self.idx = dev_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i",
                 str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], None, set()
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "samples": len(sm),
                "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def build_model(args, mask, rank, world, dev, seq_shard=False):
    """Random-init Llama-3-8B (or this rank's shard of it) directly on the GPU, patched through the drop-in API.
    ``seq_shard=False``: head-parallel shard (KV heads split over the ranks, the reference's TP rule);
    ``seq_shard=True`` : decode-phase shard with sequence-sharded retrieval heads (attention replicated, MLP split)."""
    import torch
    from transformers import LlamaConfig, LlamaForCausalLM
    from transformers.models.llama.modeling_llama import LlamaRotaryEmbedding

    from duo_attention_b200 import tp
    from duo_attn.patch import enable_duo_attention_eval

    cfgd = dict(L3_8B)
    cfgd.update(ARCHS[args.arch][0])
    cfgd["num_hidden_layers"] = args.layers
    plan = tp.plan_heads(mask[: args.layers], world)  # which (reordered) kv heads each rank owns, per layer
    if seq_shard:
        local_mask = mask[: args.layers]
    else:
        local_mask = plan.local_mask(rank)
        cfgd["num_attention_heads"] = cfgd["num_attention_heads"] // world
        cfgd["num_key_value_heads"] = cfgd["num_key_value_heads"] // world
    cfgd["intermediate_size"] = cfgd["intermediate_size"] // world
    cfg = LlamaConfig(**cfgd, attn_implementation="eager")
    with torch.device("meta"):
        model = LlamaForCausalLM(cfg)
    model = model.to(torch.float16 if args.kv_format == "int4" else torch.bfloat16).to_empty(device=dev)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    g_rep = torch.Generator(device=dev).manual_seed(99)  # replicated tensors must be identical on every rank
    with torch.no_grad():
        for name, prm in model.named_parameters():
            if prm.dim() == 1:
                prm.fill_(1.0)
            else:
                split = ".mlp." in name or (".self_attn." in name and not seq_shard)
                prm.normal_(0.0, 0.02, generator=g if split else g_rep)
    model.model.rotary_emb = LlamaRotaryEmbedding(config=cfg, device=dev)
    model.eval()
    enable_duo_attention_eval(model, local_mask, SINK, RECENT)
    if world > 1 and seq_shard:
        tp.install_seq_shard(model)
    elif world > 1:
        tp.install_allreduce(model)
    return model, local_mask, plan


def fill_cache_synthetic(cache, ctx):
    import torch

    g = torch.Generator(device=cache.device).manual_seed(7)
    for t in cache.tensors:
        for name in ("full_k", "full_v", "ring_k", "ring_v"):
            if not t[name].numel():
                continue
            if t[name].dtype == torch.uint8:  # INT4: random codes, scale/zero of a unit-normal row
                t[name].random_(0, 256, generator=g)
                t[name + "_scale"].fill_(0.4)
                t[name + "_zero"].fill_(-3.0)
            else:
                t[name].normal_(generator=g)
    for l in range(cache.num_layers):
        cache.kv_seq_len_list[l] = ctx
        cache.total_list[l] = ctx
        cache.lo_list[l] = max(cache.sink_size, ctx - cache.recent_size)


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node N for --gpus N"
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        # NCCL kernels on a high-priority stream: the prefill overlaps its 256 MiB all-reduces with GEMMs that would
        # otherwise keep every SM busy until they drain
        os.environ.setdefault("TORCH_NCCL_HIGH_PRIORITY", "1")
        dist.init_process_group("nccl", device_id=dev)

    from duo_attention_b200 import _C, ops
    from duo_attn.patch import DuoAttentionStaticKVCache

    _C.load()  # fail loudly if the CUDA extension is missing
    mask, sparsity = head_pattern(args.pattern, args.sparsity)
    mask = mask[: args.layers]
    model, local_mask, head_plan = build_model(args, mask, rank, world, dev)
    if args.tp_pipeline_blocks is not None:
        model._duo_tp_pipeline_blocks = max(1, args.tp_pipeline_blocks)
        if args.tp_pipeline_blocks == 0:
            model._duo_tp_pipeline_rows = 1 << 60
    vocab = {**L3_8B, **ARCHS[args.arch][0]}["vocab_size"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    result = {}
    dumps = {}  # --dump-outputs: name -> host tensor
    launches = 0
    # ------------------------------------------------------------------ prefill @128K
    seq_decode = world > 1 and args.kv_format == "bf16" and not args.head_tp_decode
    cache = DuoAttentionStaticKVCache(model, local_mask, 1, (args.prefill_ctx if seq_decode else args.ctx) + 8, SINK, RECENT,
                                      prefilling_chunk_size=args.chunk if not args.no_prefill else 64,
                                      kv_format="int4" if args.kv_format == "int4" else "same")
    gcpu = torch.Generator().manual_seed(1)
    if not args.no_prefill:
        ids_host = torch.randint(0, vocab, (1, args.prefill_ctx), generator=gcpu).pin_memory()

        def prefill_once(e2e):
            cache.clear()
            out = None
            for i in range(0, args.prefill_ctx, args.chunk):
                chunk = ids_host[:, i : i + args.chunk].to(dev, non_blocking=True)
                out = model(input_ids=chunk, past_key_values=cache, use_cache=True)
            tok = out.logits[:, -1, :].argmax(-1)
            return (int(tok.item()) if e2e else tok), out.logits

        with torch.no_grad():
            prefill_once(False)  # warm-up (cuBLAS heuristics, TMA descriptors, allocator)
            barrier()
            c0 = cache.launch_count + ops.LAUNCHES
            times, attn_times = [], []
            for _ in range(args.prefill_reps):
                cache.profile_events = []
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.nvtx.range_push("timed_prefill")
                e0.record()
                _, logits = prefill_once(True)  # host ids in, host token out: this IS the end-to-end call
                e1.record()
                barrier()
                torch.cuda.nvtx.range_pop()
                times.append(max_over_ranks(e0.elapsed_time(e1)))
                attn_times.append(sum(a.elapsed_time(b) for a, b in cache.profile_events))
            cache.profile_events = None
            launches_prefill = cache.launch_count + ops.LAUNCHES - c0
            if args.dump_outputs:
                dumps["prefill_logits"] = logits.float().cpu()
        best = min(range(len(times)), key=lambda i: times[i])
        ms = times[best]
        fl = prefill_flops(mask, args.prefill_ctx, args.chunk, G=32 // mask.shape[1])
        peaks = load_peaks()
        attn_ms = max_over_ranks(attn_times[best])  # attention launches of the SAME repetition `ms` comes from
        result["prefill"] = {
            "value": args.prefill_ctx / (ms / 1e3), "unit": "tokens/s", "ms_per_prefill": ms, "reps": args.prefill_reps,
            "e2e": True, "h2d_bytes": int(args.prefill_ctx * 8), "d2h_bytes": 8,
            "roofline": {"bound": "tensor", "achieved": fl / world / (attn_ms / 1e3) / 1e12 if attn_ms else None,
                         "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                         "frac": (fl / world / (attn_ms / 1e3) / 1e12 / peaks["bf16_tflops_sustained"]) if attn_ms else None,
                         "traffic": (ncu_traffic("prefill") or {}).get("dram_bytes"),
                         "traffic_note": "dram__bytes_read+write of ONE ncu-captured launch of duo_attn_tc_kernel (last 32K "
                                         "chunk over 96K past, n_full=4: profiles/r2_prefill.md); compute-bound kernel",
                         "attn_ms": attn_ms, "algorithmic_flops": fl,
                         "peak_source": peaks["source"] + " (sustained bf16: kernel timed inside a long step)"},
            "gpu_launches": launches_prefill,
        }

    # ------------------------------------------------------------------ decode @1M
    decode_mask = local_mask
    if seq_decode:
        # N > 1: the decode phase runs with SEQUENCE-SHARDED retrieval heads (tp.install_seq_shard): every rank streams
        # 1/N of every retrieval head, attention weights and streaming heads replicated, MLP tensor-parallel.  The
        # head-parallel caches the prefill just filled are moved over by point-to-point resharding (timed), then the
        # cache is filled synthetically to the decode context like at N = 1.
        from duo_attention_b200.kv_cache import DuoSeqShardKVCache

        model_sp, decode_mask, _ = build_model(args, mask, rank, world, dev, seq_shard=True)
        cache_sp = DuoSeqShardKVCache(model_sp, decode_mask, 1, (args.prefill_ctx if args.prefill_only else args.ctx) + 8,
                                      SINK, RECENT)
        if not args.no_prefill:
            for key in ("reshard_first_call_ms", "reshard_to_sequence_sharded_ms"):
                # first call: includes NCCL's lazy point-to-point connection set-up between every pair of ranks
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                cache_sp.load_from_head_parallel(cache, head_plan)
                e1.record()
                barrier()
                result["prefill"][key] = max_over_ranks(e0.elapsed_time(e1))
        if args.prefill_only:
            if rank == 0:
                if args.dump_outputs:
                    write_dumps(args.dump_outputs, dumps)
                print(json.dumps({"prefill_only": True, "n_gpus": world, "tp_pipeline_blocks": args.tp_pipeline_blocks,
                                  **result}), flush=True)
            dist.barrier()
            torch.cuda.synchronize()
            sys.stdout.flush()
            os._exit(0)
        del cache, model
        torch.cuda.empty_cache()
        model, cache = model_sp, cache_sp
    fill_cache_synthetic(cache, args.ctx)
    tok_dev = torch.randint(0, vocab, (1, 1), generator=gcpu).to(dev)
    tok_host = torch.randint(0, vocab, (1, 1), generator=gcpu).pin_memory()

    graph = None

    def decode_step_resident():
        if graph is not None:
            logits = graph.step(tok_dev)
        else:
            logits = model(input_ids=tok_dev, past_key_values=cache, use_cache=True).logits
        cache.evict_last(1)
        if graph is not None:
            graph.resync()
        return logits

    def decode_step_e2e():
        if graph is not None:
            logits = graph.step(tok_host)  # pinned host token -> device inside the step
        else:
            logits = model(input_ids=tok_host.to(dev, non_blocking=True), past_key_values=cache, use_cache=True).logits
        nxt = int(logits[:, -1, :].argmax(-1).item())  # D2H of the step's result
        cache.evict_last(1)
        if graph is not None:
            graph.resync()
        return nxt

    sampler = ClockSampler(local_rank)
    sampler.start()  # 200 ms period: spans warm-up, the timed decode steps and the e2e steps
    with torch.no_grad():
        # --- kernel timing pass (eager, CUDA events around every duo_attention launch on its stream) -> roofline
        for _ in range(max(3, args.warmup)):
            decode_step_resident()
        barrier()
        cache.profile_events = []
        for _ in range(args.steps):
            decode_step_resident()
        torch.cuda.synchronize()
        attn_ms = sum(a.elapsed_time(b) for a, b in cache.profile_events) / args.steps
        n_attn = len(cache.profile_events) // args.steps
        cache.profile_events = None
        if not args.no_graph:
            from duo_attention_b200.graph import DuoDecodeGraph

            graph = DuoDecodeGraph(model, cache)
        for _ in range(max(3, args.warmup)):
            decode_step_resident()
        barrier()
        # --- value: inputs resident in HBM
        c0 = cache.launch_count + ops.LAUNCHES
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.nvtx.range_push("timed_decode")
        e0.record()
        for _ in range(args.steps):
            logits = decode_step_resident()
        e1.record()
        barrier()
        torch.cuda.nvtx.range_pop()
        ms_total = max_over_ranks(e0.elapsed_time(e1))
        if args.dump_outputs:  # copied now: the graph's output buffer is overwritten by the next replay
            dumps["decode_logits"] = logits.float().cpu()
        launches = cache.launch_count + ops.LAUNCHES - c0
        # --- e2e: host token in, host token out, every step
        for _ in range(2):
            decode_step_e2e()
        barrier()
        e0.record()
        for _ in range(args.steps):
            decode_step_e2e()
        e1.record()
        barrier()
        ms_e2e = max_over_ranks(e0.elapsed_time(e1))
        for _ in range(int(0.6 / max(ms_step_guess(ms_total, args.steps), 1e-3)) + 1):  # keep the GPU busy >= 3 samples
            decode_step_resident()
        torch.cuda.synchronize()
    clocks = sampler.stop()
    if args.profile_step:
        profile_decode_steps(model, cache, tok_dev, rank, world)
    if graph is not None:  # a replayed step launches the same kernels as the captured one
        launches = args.steps * per_step_launches(cache, ops, model, tok_dev)

    ms_step = ms_total / args.steps
    peaks = load_peaks()
    if seq_decode:  # this rank's slice of every retrieval head + all (replicated) streaming heads
        from duo_attention_b200.seqshard import SeqShardPlan

        n_loc = SeqShardPlan(world, model._duo_seq.block).local_len(rank, args.ctx + 1)
        n_f = decode_mask.sum(1)
        by = float(((n_f * n_loc + (decode_mask.shape[1] - n_f) * (SINK + RECENT + 1)) * 2 * 256).sum())
    else:
        by = decode_bytes_per_token(local_mask, args.ctx, 68 if args.kv_format == "int4" else 256)  # this rank's bytes
    attn_ms_max = max_over_ranks(attn_ms)
    achieved = by / (attn_ms / 1e3) / 1e9
    cap = ncu_traffic("decode_int4" if args.kv_format == "int4" else "decode")
    traffic, traffic_note = None, "no ncu capture summarised for this round (profiles/r2_traffic.json missing)"
    if cap:
        # per average launch of THIS run: algorithmic bytes per launch x (DRAM bytes / algorithmic bytes) of the launch
        # ncu captured this round — a run whose kernel re-read data would show up in the capture, not here
        traffic = by / max(n_attn, 1) * cap["dram_bytes"] / cap["algorithmic_bytes"]
        traffic_note = (f"algorithmic bytes per average launch x DRAM/algorithmic ratio "
                        f"{cap['dram_bytes'] / cap['algorithmic_bytes']:.4f} of this round's ncu --set full capture "
                        f"({cap.get('source', 'profiles/r2_decode.md')})")
    line = {
        "metric": METRIC, "value": 1e3 / ms_step, "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "fp16 (INT4 KV)" if args.kv_format == "int4" else "bf16", "data": "synthetic",
        "config": workload_config(args, sparsity),
        "e2e": {"value": 1e3 / (ms_e2e / args.steps), "unit": "tokens/s", "h2d_bytes_per_step": 8,
                "d2h_bytes_per_step": 8},
        "gpu_launches": launches, "decode_driver": "cuda-graph replay (DuoDecodeGraph)" if graph is not None else "eager",
        "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": achieved / peaks["hbm_gbs"],
                     "traffic": traffic, "traffic_note": traffic_note,
                     "achieved_note": "algorithmic bytes of the 32 attention launches of a step / sum of their "
                                      "CUDA-event durations (eager pass on the launching stream)",
                     "kernel": ("duo_attn_int4_dec8_kernel" if args.kv_format == "int4" else "duo_attn_mma_kernel")
                               + " (decode, all layers of one step)",
                     "attn_ms_per_step": attn_ms, "attn_ms_per_step_max_rank": attn_ms_max,
                     "launches_per_step": n_attn, "algorithmic_bytes_per_step": by,
                     "peak_source": peaks["source"]},
        "a100_published": {"decode_ms_per_tok_1M": 55.0, "note": "reference figure, 1xA100-80G, other hardware"},
    }
    line.update(result)
    if world == 1 and args.kv_format == "bf16" and not args.no_fa2:
        graph = None
        del cache
        torch.cuda.empty_cache()
        try:  # end to end: the reference's static forward + cache on its own libraries, same weights, same protocol
            from baseline import fa2_restated

            ref = fa2_restated.run(model, [int(x) for x in mask.sum(1)], SINK, RECENT, args.ctx, args.prefill_ctx,
                                   args.chunk, vocab, decode_steps=args.steps, decode_warmup=max(3, args.warmup),
                                   do_prefill=not args.no_prefill)
            ref["decode"]["ours_over_reference"] = line["e2e"]["value"] / ref["decode"]["value"]
            if "prefill" in ref and "prefill" in line:
                ref["prefill"]["ours_over_reference"] = line["prefill"]["value"] / ref["prefill"]["value"]
            line["reference_gpu_same_box"] = ref
        except Exception as e:  # the comparison is informative, never fatal
            line["reference_gpu_same_box"] = {"error": repr(e)}
        torch.cuda.empty_cache()
        if args.arch == "llama3-8b-1048k":
            try:
                line["fa2_same_box"] = fa2_same_box(dev, args.ctx, args.chunk, args.prefill_ctx)
            except Exception as e:
                line["fa2_same_box"] = {"error": repr(e)}
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        cb = cpu_reference_sample(args.ctx, mask)
        line["cpu_baseline"] = {"value": cb["tok_s"], "unit": "tokens/s", "cores": cb["cores"], "kind": "port",
                                "sample": "oracle port of the reference forward: 1 retrieval KV head @ctx + 1 streaming "
                                          "KV head + 1 layer of linears, extrapolated to 128+128 heads x 32 layers",
                                "t_full_head_s": cb["t_full_head_s"]}
    if rank == 0:
        if args.dump_outputs:
            write_dumps(args.dump_outputs, dumps)
        print(json.dumps(line), flush=True)
    if world > 1:
        # NCCL communicators captured inside the CUDA graph make destroy_process_group() hang: synchronise,
        # release the graph and leave without the collective teardown.
        dist.barrier()
        torch.cuda.synchronize()
        graph = None
        sys.stdout.flush()
        os._exit(0)


def fa2_same_box(dev, ctx, chunk, prefill_ctx):
    """The reference's own GPU attention on this box: llama.py:374-421 restated with the INSTALLED flash_attn_func
    (FA2 recompiled for sm_100, mma.sync; SURVEY.md §0 fact 10) on token-major caches, timed per layer with the
    reference's bench protocol (CUDA events), next to our fused launch on the same shapes.  Micro-benchmark of
    the attention op only (one layer, n_full = 4 of 8 KV heads)."""
    import ctypes as C

    import torch

    from duo_attention_b200 import _C
    from duo_attention_b200.kv_cache import DuoKVCache

    try:
        from flash_attn import flash_attn_func
    except Exception as e:  # pragma: no cover
        return {"unavailable": repr(e)}
    Hq, Hkv, nf, D, G = 32, 8, 4, 128, 4
    W = SINK + RECENT
    res = {}
    g = torch.Generator(device=dev).manual_seed(3)

    def timeit(fn, reps):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    # ---- decode at ctx: reference = FA2(full q-heads, token-major full cache) + FA2(streaming) + cat
    fk = torch.randn(1, ctx + 1, nf, D, device=dev, dtype=torch.bfloat16, generator=g)
    fv = torch.randn(1, ctx + 1, nf, D, device=dev, dtype=torch.bfloat16, generator=g)
    sk = torch.randn(1, W + 1, Hkv - nf, D, device=dev, dtype=torch.bfloat16, generator=g)
    sv = torch.randn(1, W + 1, Hkv - nf, D, device=dev, dtype=torch.bfloat16, generator=g)
    q = torch.randn(1, 1, Hq, D, device=dev, dtype=torch.bfloat16, generator=g)

    def ref_decode():
        a = flash_attn_func(q[:, :, : nf * G], fk, fv, causal=True)
        b = flash_attn_func(q[:, :, nf * G :], sk, sv, causal=True)
        return torch.cat([a, b], dim=2)

    t_ref = timeit(ref_decode, 10)
    del fk, fv
    cache = DuoKVCache(1, Hq, Hkv, D, [nf], 1, ctx + 8, SINK, RECENT, torch.bfloat16, dev)
    for n in ("full_k", "full_v", "ring_k", "ring_v"):
        cache.tensors[0][n].normal_(generator=g)
    qkv = torch.randn(1, 1, (Hq + 2 * Hkv) * D, device=dev, dtype=torch.bfloat16, generator=g)
    out = torch.empty(1, 1, Hq, D, device=dev, dtype=torch.bfloat16)
    st = _C.CacheState(ctx, ctx, ctx - RECENT)
    stream = torch.cuda.current_stream().cuda_stream
    lib, h = cache.lib, cache.handles[0]
    _C.check(lib.duo_rope_append(h, C.byref(st), qkv.data_ptr(), qkv.stride(1), None, None, 0, 1, stream))

    def ours_decode():
        _C.check(lib.duo_attention(h, C.byref(st), qkv.data_ptr(), qkv.stride(1), out.data_ptr(), 1, D ** -0.5,
                                   cache.workspace.data_ptr(), cache.workspace.numel(), stream))

    t_ours = timeit(ours_decode, 10)
    res["decode_layer_nfull4"] = {"ctx": ctx, "fa2_ms": t_ref, "ours_ms": t_ours, "speedup": t_ref / t_ours}
    del cache
    # ---- prefill: last chunk of the 128K prefill (chunk tokens against prefill_ctx keys)
    past = prefill_ctx - chunk
    fk = torch.randn(1, prefill_ctx, nf, D, device=dev, dtype=torch.bfloat16, generator=g)
    fv = torch.randn(1, prefill_ctx, nf, D, device=dev, dtype=torch.bfloat16, generator=g)
    sk = torch.randn(1, W + chunk, Hkv - nf, D, device=dev, dtype=torch.bfloat16, generator=g)
    sv = torch.randn(1, W + chunk, Hkv - nf, D, device=dev, dtype=torch.bfloat16, generator=g)
    q = torch.randn(1, chunk, Hq, D, device=dev, dtype=torch.bfloat16, generator=g)

    def ref_prefill():
        a = flash_attn_func(q[:, :, : nf * G], fk, fv, causal=True)
        b = flash_attn_func(q[:, :, nf * G :], sk, sv, causal=True)
        return torch.cat([a, b], dim=2)

    t_ref = timeit(ref_prefill, 3)
    del fk, fv, sk, sv
    cache = DuoKVCache(1, Hq, Hkv, D, [nf], 1, prefill_ctx + 8, SINK, RECENT, torch.bfloat16, dev, stage_cap=chunk)
    for n in ("full_k", "full_v", "ring_k", "ring_v"):
        cache.tensors[0][n].normal_(generator=g)
    qkv = torch.randn(1, chunk, (Hq + 2 * Hkv) * D, device=dev, dtype=torch.bfloat16, generator=g)
    out = torch.empty(1, chunk, Hq, D, device=dev, dtype=torch.bfloat16)
    st = _C.CacheState(past, past, past - RECENT)
    lib, h = cache.lib, cache.handles[0]
    _C.check(lib.duo_rope_append(h, C.byref(st), qkv.data_ptr(), qkv.stride(1), None, None, 0, chunk, stream))

    def ours_prefill():
        _C.check(lib.duo_attention(h, C.byref(st), qkv.data_ptr(), qkv.stride(1), out.data_ptr(), chunk, D ** -0.5,
                                   cache.workspace.data_ptr(), cache.workspace.numel(), stream))

    t_ours = timeit(ours_prefill, 3)
    pairs_full = chunk * past + chunk * (chunk + 1) // 2
    pairs_stream = chunk * W + chunk * (chunk + 1) // 2
    fl = 4.0 * D * G * (nf * pairs_full + (Hkv - nf) * pairs_stream)
    res["prefill_layer_nfull4_last_chunk"] = {
        "chunk": chunk, "past": past, "fa2_ms": t_ref, "ours_ms": t_ours, "speedup": t_ref / t_ours,
        "fa2_tflops": fl / t_ref / 1e9, "ours_tflops": fl / t_ours / 1e9}
    del cache
    torch.cuda.empty_cache()
    return res


def profile_decode_steps(model, cache, tok_dev, rank, world, steps=3):
    """Kernel-level table of `steps` EAGER decode steps on rank 0 (every rank runs the steps: they contain the
    exchanges).  Evidence for which kernel / exchange limits a multi-GPU step; kept under profiles/."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    ds, cache.dev_state = cache.dev_state, None

    def run():
        with torch.no_grad():
            for _ in range(steps):
                model(input_ids=tok_dev, past_key_values=cache, use_cache=True)
                cache.evict_last(1)
        torch.cuda.synchronize()

    run()
    if rank == 0:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run()
        os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
        with open(os.path.join(ROOT, "gpurun_out", f"profile_step_n{world}.txt"), "w") as f:
            f.write(f"{steps} eager decode steps, rank 0 of {world} (torch.profiler, CUDA activities)\n")
            f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=25, max_name_column_width=90))
    else:
        run()
    cache.dev_state = ds
    cache.sync_device_state()


def per_step_launches(cache, ops, model, tok_dev):
    """Kernels of OUR library in one decode step (counted on one eager step)."""
    import torch

    c0 = cache.launch_count + ops.LAUNCHES
    ds, cache.dev_state = cache.dev_state, None  # eager step without touching the graph's device state
    with torch.no_grad():
        model(input_ids=tok_dev, past_key_values=cache, use_cache=True)
    cache.evict_last(1)
    cache.dev_state = ds
    cache.sync_device_state()
    return cache.launch_count + ops.LAUNCHES - c0


def write_dumps(out_dir, dumps):
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, t in dumps.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.numpy().astype(np.float32))


def ms_step_guess(ms_total, steps):
    return ms_total / max(steps, 1) / 1e3


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "MEASURED_PEAKS.json (of measured)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0,
            "source": "B200_PROFILING.md fallback (of fallback)"}


if __name__ == "__main__":
    main()
