"""RoPE + append + ring commit + INT4 quantise kernels vs torch / the oracles / the reference's own
kernels (demo/quantize_int4.cu; their outputs are stored in tests/golden/int4_ref_kernels.npz)."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest
import torch

import golden_cases as GC
from duo_attention_b200 import _C
from duo_attention_b200.kv_cache import DuoKVCache, ring_slot
from oracle import duo_oracle as O
from oracle import int4_oracle as Q

pytestmark = pytest.mark.gpu
D = 128
dev = torch.device("cuda:0") if torch.cuda.is_available() else None


def _rope_case(dtype, mode, B=2, S=37, Hq=8, Hkv=4, n_full=3, pos0=1000, theta=10000.0):
    g = torch.Generator().manual_seed(4)
    qkv = torch.randn(B, S, (Hq + 2 * Hkv) * D, generator=g).to(dtype)
    pos = torch.arange(pos0, pos0 + S)[None]
    cache = DuoKVCache(1, Hq, Hkv, D, [n_full], B, 64, 4, 8, dtype, dev, stage_cap=S)
    q = qkv[..., : Hq * D].reshape(B, S, Hq, D)
    k = qkv[..., Hq * D : (Hq + Hkv) * D].reshape(B, S, Hkv, D)
    v = qkv[..., (Hq + Hkv) * D :].reshape(B, S, Hkv, D)
    if mode == _C.ROPE_HF:
        cos, sin = O.hf_cos_sin(pos, D, theta, dtype)
        q_ref, k_ref = O.apply_rotary_pos_emb_hf(q, k, cos, sin, unsqueeze_dim=2)
        cos_d, sin_d = cos[0].contiguous().to(dev), sin[0].contiguous().to(dev)
    else:
        q_ref, k_ref = O.rope_flashinfer(q, k, pos0, 1.0, theta)
        idx = torch.arange(D // 2, dtype=torch.float32)
        freq = torch.pow(torch.tensor(theta), -2.0 * idx / D)
        ang = pos[0].float()[:, None] * freq[None]
        cos_d = torch.cat([ang.cos(), ang.cos()], -1).contiguous().to(dev)
        sin_d = torch.cat([ang.sin(), ang.sin()], -1).contiguous().to(dev)
    qkv_d = qkv.to(dev)
    st = cache.state(0)
    stream = torch.cuda.current_stream().cuda_stream
    _C.check(cache.lib.duo_rope_append(cache.handles[0], C.byref(st), qkv_d.data_ptr(), qkv_d.stride(1),
                                       cos_d.data_ptr(), sin_d.data_ptr(), mode, S, stream))
    torch.cuda.synchronize()
    t = cache.tensors[0]
    q_got = qkv_d[..., : Hq * D].reshape(B, S, Hq, D).cpu()
    # caches are head-major: [B, heads, slot, D]
    fk = t["full_k"][:, :, :S].permute(0, 2, 1, 3).cpu()
    fv = t["full_v"][:, :, :S].permute(0, 2, 1, 3).cpu()
    W = 12
    rk = t["ring_k"][:, :, W : W + S].permute(0, 2, 1, 3).cpu()
    rv = t["ring_v"][:, :, W : W + S].permute(0, 2, 1, 3).cpu()
    return (q_got, q_ref), (fk, k_ref[:, :, :n_full]), (rk, k_ref[:, :, n_full:]), (fv, v[:, :, :n_full]), \
        (rv, v[:, :, n_full:]), qkv_d, qkv


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_rope_hf_mode_is_bit_exact_with_torch(dtype):
    *pairs, qkv_d, qkv = _rope_case(dtype, _C.ROPE_HF)
    for got, ref in pairs:
        assert torch.equal(got, ref)
    # k / v columns of the fused buffer are left untouched
    assert torch.equal(qkv_d[..., 8 * D :].cpu(), qkv[..., 8 * D :])


def test_rope_fp32_mode_matches_flashinfer_restatement():
    *pairs, _, _ = _rope_case(torch.bfloat16, _C.ROPE_FP32, pos0=123456)
    for got, ref in pairs:
        torch.testing.assert_close(got.float(), ref.float(), rtol=8e-3, atol=8e-3)


def test_rope_restatement_vs_installed_flashinfer():
    """Pins oracle.rope_flashinfer against the library the reference's static path calls."""
    flashinfer = pytest.importorskip("flashinfer")
    g = torch.Generator().manual_seed(1)
    S, Hq, Hkv = 50, 8, 2
    q = torch.randn(1, S, Hq, D, generator=g).to(torch.bfloat16)
    k = torch.randn(1, S, Hkv, D, generator=g).to(torch.bfloat16)
    q_ref, k_ref = O.rope_flashinfer(q, k, 777, 1.0, 10000.0)
    qd, kd = q.to(dev).view(S, Hq, D).clone(), k.to(dev).view(S, Hkv, D).clone()
    indptr = torch.tensor([0, S], dtype=torch.int32, device=dev)
    offsets = torch.tensor([777], dtype=torch.int32, device=dev)
    try:
        flashinfer.rope.apply_rope_inplace(qd, kd, indptr, offsets, interleave=False, rope_scale=1.0,
                                           rope_theta=10000.0)
    except Exception as e:  # JIT compile needs a toolchain/network on some boxes
        pytest.skip(f"flashinfer rope unavailable here: {e!r}")
    torch.testing.assert_close(qd.cpu().float().view(1, S, Hq, D), q_ref.float(), rtol=2e-2, atol=2e-2)
    torch.testing.assert_close(kd.cpu().float().view(1, S, Hkv, D), k_ref.float(), rtol=2e-2, atol=2e-2)


def test_commit_places_rows_in_sink_and_ring_slots():
    Hq, Hkv, n_full, sink, recent = 4, 2, 0, 3, 5
    W = sink + recent
    cache = DuoKVCache(1, Hq, Hkv, D, [n_full], 1, 64, sink, recent, torch.bfloat16, dev, stage_cap=16)
    g = torch.Generator().manual_seed(2)
    pos = 0
    where = {}
    for S in [2, 4, 1, 16, 1, 1, 7]:
        qkv = torch.randn(1, S, (Hq + 2 * Hkv) * D, generator=g).to(torch.bfloat16)
        # tag: K row of token p has p in element 0 (bf16 exact for small ints)
        kpart = qkv[..., Hq * D : (Hq + Hkv) * D].view(1, S, Hkv, D)
        for i in range(S):
            kpart[0, i, :, 0] = float(pos + i)
        out = torch.empty(1, S, Hq, D, dtype=torch.bfloat16, device=dev)
        cache.attend(0, qkv.to(dev), None, None, _C.ROPE_NONE, out)
        pos += S
        torch.cuda.synchronize()
        rk = cache.tensors[0]["ring_k"][0, :, :W, 0].float().cpu()
        live = list(range(0, min(pos, sink))) + list(range(max(sink, pos - recent), pos))
        for p in live:
            assert (rk[:, ring_slot(p, sink, recent)] == p).all(), (pos, p)


# ------------------------------------------------------------------------------------------------ INT4
def _quant_gpu(x16):
    rows = x16.numel() // 128
    xd = x16.to(dev).contiguous()
    packed = torch.empty(rows, 64, dtype=torch.uint8, device=dev)
    scale = torch.empty(rows, dtype=torch.float16, device=dev)
    zero = torch.empty(rows, dtype=torch.float16, device=dev)
    lib = _C.load()
    _C.check(lib.duo_quant_int4(xd.data_ptr(), 128, rows, packed.data_ptr(), scale.data_ptr(), zero.data_ptr(),
                                torch.cuda.current_stream().cuda_stream))
    return packed, scale, zero


def test_quant_matches_numpy_oracle_bit_exact():
    rng = np.random.RandomState(0)
    x = (rng.randn(3000, 128) * rng.uniform(0.01, 8, size=(3000, 1))).astype(np.float16)
    x[5] = 0.25  # constant group
    x[6, :] = 0
    p, s, z = _quant_gpu(torch.from_numpy(x))
    po, so, zo = Q.quantize_int4(x)
    assert np.array_equal(s.cpu().numpy(), so[:, 0]) and np.array_equal(z.cpu().numpy(), zo[:, 0])
    assert np.array_equal(p.cpu().numpy(), po)  # IEEE division on both sides: bit exact


def test_dequant_matches_numpy_oracle_bit_exact():
    rng = np.random.RandomState(1)
    x = (rng.randn(2000, 128) * 2).astype(np.float16)
    po, so, zo = Q.quantize_int4(x)
    out = torch.empty(2000, 128, dtype=torch.float16, device=dev)
    lib = _C.load()
    pd, sd, zd = (torch.from_numpy(a).to(dev).contiguous() for a in (po, so[:, 0].copy(), zo[:, 0].copy()))
    _C.check(lib.duo_dequant_int4(pd.data_ptr(), sd.data_ptr(), zd.data_ptr(), 2000, out.data_ptr(),
                                  torch.cuda.current_stream().cuda_stream))
    assert np.array_equal(out.cpu().numpy(), Q.dequantize_int4(po, so, zo))


def test_quant_dequant_vs_reference_kernels_compiled_from_source():
    """The reference's demo/quantize_int4.cu built with its own flags (--use_fast_math); its outputs on this input
    are the fixture (tests/golden/make_golden.py int4-kernels): codes, scales and zeros of every row, and the SHA-256
    of its dequantisation of them.
    scale/zero must be bit-exact; codes may differ by one only on (near-)exact .5 ties because the
    reference's fast-math division is approximate; dequantise is bit-exact."""
    fx = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "int4_ref_kernels.npz"))
    x = GC.make_int4_kernel_input()
    assert abs(np.abs(x.astype(np.float64)).sum() - float(fx["checksum"])) < 1e-9 * float(fx["checksum"]), "RNG drift"
    p, s, z = _quant_gpu(torch.from_numpy(x))
    assert np.array_equal(s.cpu().numpy(), fx["scale"]) and np.array_equal(z.cpu().numpy(), fx["zero"])
    mine = Q.unpack_codes(p.cpu().numpy()).astype(np.int32).reshape(-1)
    theirs = Q.unpack_codes(fx["packed"]).astype(np.int32).reshape(-1)
    diff = np.abs(mine - theirs)
    assert diff.max() <= 1 and (diff != 0).mean() < 2e-3, (diff.max(), (diff != 0).mean())
    # where they differ the true quotient sits on a rounding tie
    po, so, zo = Q.quantize_int4(x.reshape(-1, 128))
    assert np.array_equal(Q.unpack_codes(po).reshape(-1), mine)
    # K2: dequantise their packed data with both
    n = fx["packed"].shape[0]
    qp, sc, zp = (torch.from_numpy(fx[k]).to(dev).contiguous() for k in ("packed", "scale", "zero"))
    mine_d = torch.empty(n, 128, dtype=torch.float16, device=dev)
    lib = _C.load()
    _C.check(lib.duo_dequant_int4(qp.data_ptr(), sc.data_ptr(), zp.data_ptr(), n, mine_d.data_ptr(),
                                  torch.cuda.current_stream().cuda_stream))
    oracle_d = Q.dequantize_int4(fx["packed"], fx["scale"].reshape(-1, 1), fx["zero"].reshape(-1, 1))
    assert np.array_equal(mine_d.cpu().numpy(), oracle_d)
    assert hashlib.sha256(oracle_d.tobytes()).hexdigest() == str(fx["dequant_sha256"])
