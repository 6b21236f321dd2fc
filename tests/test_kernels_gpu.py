"""GPU: every kernel behind its C-ABI test entry point against a plain torch fp64/fp32 reference of the same op
(operands pre-rounded to the kernel's operand dtype, so the comparison isolates the kernel's own arithmetic)."""

import math

import pytest
import torch

from gpu_util import BF16, CODE, F16, F32, check, gelu_tanh, gemm, ptr, quick_gelu, rel_err, stream

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _tf32(x):
    import jimm_oracle as O

    return O.round_operand(x.cpu(), "tf32").to(x.device)


def _mk(M, N, K, dtype, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    A = torch.randn(M, K, generator=g).to(DEV)
    B = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(DEV)
    if dtype == torch.float32:
        A, B = _tf32(A), _tf32(B)  # low 13 mantissa bits zero: exact whether the MMA truncates or rounds to tf32
        return A, B, A.double(), B.double()
    A, B = A.to(dtype), B.to(dtype)
    return A, B, A.double(), B.double()


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float32])
@pytest.mark.parametrize("M,N,K", [(128, 256, 64), (256, 512, 768), (197 * 4, 2304, 768), (1000, 1000, 512), (5, 24, 128), (300, 768, 3072)])
def test_gemm_plain(lib, dtype, M, N, K):
    A, B, Ad, Bd = _mk(M, N, K, dtype)
    ref = Ad @ Bd.T
    for mode in (0, 1, 2):
        out = gemm(lib, A, B, mode=mode)
        assert rel_err(out, ref) < 2e-5, (mode, rel_err(out, ref))
    simt = gemm(lib, A, B, impl=1)
    assert rel_err(simt, ref) < 2e-5


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("act", [0, 1, 2])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_gemm_bias_act_16bit_out(lib, dtype, act, mode):
    M, N, K = 777, 1536, 512
    A, B, Ad, Bd = _mk(M, N, K, dtype, seed=1)
    bias = torch.randn(N, device=DEV)
    ref = Ad @ Bd.T + bias.double()
    ref = [ref, gelu_tanh(ref), quick_gelu(ref)][act]
    out = gemm(lib, A, B, bias=bias, act=act, out_dtype=dtype, mode=mode)
    tol = 2e-3 if dtype == torch.float16 else 1.2e-2  # one output rounding
    assert rel_err(out, ref) < tol
    # and in fp32 to check the activation math itself
    out32 = gemm(lib, A, B, bias=bias, act=act, out_dtype=torch.float32, mode=mode)
    assert rel_err(out32, ref) < 3e-5


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_gemm_residual_inplace(lib, dtype, mode):
    M, N, K = 650, 768, 256
    A, B, Ad, Bd = _mk(M, N, K, dtype, seed=2)
    bias = torch.randn(N, device=DEV)
    x = torch.randn(M, N, device=DEV)
    ref = x.double() + Ad @ Bd.T + bias.double()
    out = gemm(lib, A, B, bias=bias, residual=x, mode=mode)  # in place on x
    assert out.data_ptr() == x.data_ptr()
    assert rel_err(out, ref) < 2e-5


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_gemm_patch_epilogue(lib, mode):
    """Row remap + position-embedding add used by the patch-embed GEMM (common/vit.py:231-236)."""
    Bn, n, S, D, K = 3, 16, 17, 128, 192
    A, B, Ad, Bd = _mk(Bn * n, D, K, torch.float16, seed=3)
    bias = torch.randn(D, device=DEV)
    pos = torch.randn(S, D, device=DEV)
    out = torch.full((Bn * S, D), -7.0, device=DEV)
    gemm(lib, A, B, bias=bias, rowadd=pos, rows=(n, S, 1), out=out, mode=mode)
    ref = (Ad @ Bd.T + bias.double()).reshape(Bn, n, D) + pos[1:].double()
    got = out.reshape(Bn, S, D)
    assert rel_err(got[:, 1:], ref) < 2e-5
    assert torch.all(got[:, 0] == -7.0)  # CLS rows untouched


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.float16])
def test_gemm_unaligned_n_scalar_epilogue(lib, mode, out_dtype):
    """N not a multiple of 4 (e.g. 10 classes): scalar epilogue path, bias + residual."""
    M, N, K = 37, 10, 128
    A, B, Ad, Bd = _mk(M, N, K, torch.float16, seed=5)
    bias = torch.randn(N, device=DEV)
    ref = Ad @ Bd.T + bias.double()
    out = gemm(lib, A, B, bias=bias, out_dtype=out_dtype, mode=mode)
    assert rel_err(out, ref) < (2e-5 if out_dtype == torch.float32 else 2e-3)


def test_gemm_strided_and_m_override_tail(lib):
    M, N, K = 130, 264, 200  # N not a multiple of 256/32-chunks-of-8, K tail (200 = 3*64 + 8)
    A, B, Ad, Bd = _mk(M, N, K, torch.float16, seed=4)
    ref = Ad @ Bd.T
    for mode in (0, 1, 2):
        assert rel_err(gemm(lib, A, B, mode=mode), ref) < 2e-5
    big = torch.randn(M, 3 * K, device=DEV).half()
    Av = big[:, K:2 * K]  # row stride 3K
    assert rel_err(gemm(lib, Av, B), Av.double() @ Bd.T) < 2e-5


@pytest.mark.parametrize("out_dtype", [torch.float16, torch.bfloat16, torch.float32])
@pytest.mark.parametrize("D", [128, 512, 768, 1024, 1152])
def test_layernorm(lib, out_dtype, D):
    rows = 333
    x = (torch.randn(rows, D, device=DEV) * 3 + 1.5)
    scale, bias = torch.randn(D, device=DEV), torch.randn(D, device=DEV)
    out = torch.empty(rows, D, dtype=out_dtype, device=DEV)
    eps = 1e-6
    check(lib, lib.jimm_k_layernorm(ptr(x), D, 1, 0, None, ptr(scale), ptr(bias), eps, ptr(out), CODE[out_dtype], D, rows, D, stream()))
    xd = x.double()
    mean = xd.mean(-1, keepdim=True)
    var = ((xd * xd).mean(-1, keepdim=True) - mean * mean).clamp_min(0)
    ref = (xd - mean) * torch.rsqrt(var + eps) * scale.double() + bias.double()
    tol = {torch.float32: 2e-5, torch.float16: 1e-3, torch.bfloat16: 8e-3}[out_dtype]
    assert rel_err(out, ref) < tol


def test_layernorm_gather_rows_and_eps(lib):
    """Pooled-row LayerNorm: CLS row (offset 0), last row, and per-sample index (CLIP EOT)."""
    B, S, D = 7, 11, 256
    x = torch.randn(B, S, D, device=DEV)
    scale, bias = torch.ones(D, device=DEV), torch.zeros(D, device=DEV)
    idx = torch.randint(0, S, (B,), device=DEV, dtype=torch.int32)
    for off, index in ((0, None), (S - 1, None), (0, idx)):
        out = torch.empty(B, D, device=DEV)
        check(lib, lib.jimm_k_layernorm(ptr(x), D, S, off, ptr(index), ptr(scale), ptr(bias), 1e-12, ptr(out), F32, D, B, D, stream()))
        rows = x[torch.arange(B), index.long()] if index is not None else x[:, off]
        ref = torch.nn.functional.layer_norm(rows.double(), (D,), eps=1e-12)
        assert rel_err(out, ref) < 2e-5
    # constant rows: fast-variance clamps at 0 -> output == bias exactly
    xc = torch.full((4, D), 2.5, device=DEV)
    out = torch.empty(4, D, device=DEV)
    check(lib, lib.jimm_k_layernorm(ptr(xc), D, 1, 0, None, ptr(scale), ptr(bias), 1e-6, ptr(out), F32, D, 4, D, stream()))
    assert torch.all(out == 0)


def _attn_ref(qkv, B, S, H, causal):
    D = H * 64
    q, k, v = qkv.double().reshape(B, S, 3, H, 64).permute(2, 0, 3, 1, 4)
    w = (q / 8.0) @ k.transpose(-1, -2)
    if causal:
        w = w.masked_fill(~torch.tril(torch.ones(S, S, dtype=torch.bool, device=qkv.device)), float("-inf"))
    return (torch.softmax(w, -1) @ v).permute(0, 2, 1, 3).reshape(B * S, D)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("S", [1, 16, 50, 64, 77, 128, 129, 144, 197, 200, 256, 257, 384, 385, 577, 700, 1024])
@pytest.mark.parametrize("causal", [0, 1])
def test_attention(lib, dtype, S, causal):
    B, H = 3, 2
    qkv = (torch.randn(B * S, 3 * H * 64, device=DEV) * 1.5).to(dtype)
    ref = _attn_ref(qkv, B, S, H, causal)
    for out_dtype in (dtype, torch.float32):
        out = torch.empty(B * S, H * 64, dtype=out_dtype, device=DEV)
        check(lib, lib.jimm_k_attention(ptr(qkv), CODE[dtype], ptr(out), CODE[out_dtype], B, S, H, causal, stream()))
        # P is rounded to the operand dtype before P.V (as in any tensor-core flash kernel)
        tol = 3e-3 if dtype == torch.float16 else 2e-2
        assert rel_err(out, ref) < tol, (S, causal, out_dtype, rel_err(out, ref))


@pytest.mark.parametrize("S,causal", [(130, 1), (197, 0), (256, 1), (577, 0)])
def test_attention_flash_kernel_forced(lib, monkeypatch, S, causal):
    """S <= 256 normally takes the tcgen05 kernel; JIMM_ATTN_IMPL=flash keeps the mma.sync kernel covered there too."""
    monkeypatch.setenv("JIMM_ATTN_IMPL", "flash")
    B, H = 2, 3
    qkv = (torch.randn(B * S, 3 * H * 64, device=DEV) * 1.5).half()
    out = torch.empty(B * S, H * 64, dtype=torch.float16, device=DEV)
    check(lib, lib.jimm_k_attention(ptr(qkv), F16, ptr(out), F16, B, S, H, causal, stream()))
    assert rel_err(out, _attn_ref(qkv, B, S, H, causal)) < 3e-3


def test_attention_many_items_persistent(lib):
    """More (sample, head) items than SMs: exercises the persistent loop, the 2-deep smem ring and TMEM slot reuse."""
    B, S, H = 40, 197, 12
    qkv = (torch.randn(B * S, 3 * H * 64, device=DEV)).half()
    out = torch.empty(B * S, H * 64, dtype=torch.float16, device=DEV)
    check(lib, lib.jimm_k_attention(ptr(qkv), F16, ptr(out), F16, B, S, H, 0, stream()))
    assert rel_err(out, _attn_ref(qkv, B, S, H, 0)) < 3e-3


def test_attention_long_many_units_persistent(lib):
    """S > 256: key-block tcgen05 kernel; more units than SMs, partial last key block and single-tile last query pair."""
    B, S, H = 24, 576, 4
    qkv = (torch.randn(B * S, 3 * H * 64, device=DEV)).half()
    out = torch.empty(B * S, H * 64, dtype=torch.float16, device=DEV)
    check(lib, lib.jimm_k_attention(ptr(qkv), F16, ptr(out), F16, B, S, H, 0, stream()))
    assert rel_err(out, _attn_ref(qkv, B, S, H, 0)) < 3e-3


@pytest.mark.parametrize("S", [197, 256, 300, 576, 1024])
def test_attention_lazy_rescale_path(lib, S):
    """Scores that keep growing along the key axis force the lazily raised reference maximum (and the rescale of the P chunks
    already written to tensor memory -- for S > 256 also of the O accumulator, across key blocks) at every 32-key chunk of the
    single-pass softmax."""
    B, H = 2, 2
    g = torch.Generator(device="cpu").manual_seed(3)
    q = torch.randn(B, S, H, 64, generator=g)
    ramp = torch.linspace(0.0, 40.0, S).reshape(1, S, 1, 1)  # key j gets a bias direction scaled by j
    u = torch.nn.functional.normalize(torch.randn(1, 1, H, 64, generator=g), dim=-1)
    k = torch.randn(B, S, H, 64, generator=g) * 0.3 + ramp * u * 3.0
    q = q * 0.3 + u * 8.0
    v = torch.randn(B, S, H, 64, generator=g)
    qkv = torch.stack([q, k, v], dim=2).reshape(B * S, 3 * H * 64).to(DEV).half()
    out = torch.empty(B * S, H * 64, dtype=torch.float32, device=DEV)
    check(lib, lib.jimm_k_attention(ptr(qkv), F16, ptr(out), F32, B, S, H, 0, stream()))
    ref = _attn_ref(qkv, B, S, H, 0)
    assert torch.isfinite(out).all()
    assert rel_err(out, ref) < 5e-3, rel_err(out, ref)


def test_attention_large_scores_stable(lib):
    B, S, H = 1, 230, 1
    qkv = (torch.randn(B * S, 3 * 64, device=DEV) * 12).half()
    out = torch.empty(B * S, 64, dtype=torch.float32, device=DEV)
    check(lib, lib.jimm_k_attention(ptr(qkv), F16, ptr(out), F32, B, S, H, 0, stream()))
    assert torch.isfinite(out).all()
    assert rel_err(out, _attn_ref(qkv, B, S, H, 0)) < 5e-3


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("S", [4, 196, 1024])
def test_map_attention(lib, dtype, S):
    B, H = 5, 3
    D = H * 64
    q = torch.randn(D, device=DEV)
    kv = torch.randn(B * S, 2 * D, device=DEV).to(dtype)
    out = torch.empty(B, D, dtype=torch.float32, device=DEV)
    check(lib, lib.jimm_k_map_attention(ptr(q), ptr(kv), CODE[dtype], ptr(out), F32, B, S, H, stream()))
    k, v = kv.double().reshape(B, S, 2, H, 64).permute(2, 0, 3, 1, 4)
    w = torch.softmax((q.double().reshape(1, H, 1, 64) / 8.0) @ k.transpose(-1, -2), -1)
    ref = (w @ v).reshape(B, D)
    assert rel_err(out, ref) < 2e-5


@pytest.mark.parametrize("in_dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("img,P", [(32, 8), (224, 16), (36, 16)])
def test_patchify(lib, in_dtype, img, P):
    B, C = 3, 3
    x = torch.randn(B, img, img, C, device=DEV).to(in_dtype)
    g = img // P
    out = torch.full((B * g * g, P * P * C), 9.0, dtype=torch.float16, device=DEV)
    check(lib, lib.jimm_k_patchify(ptr(x), CODE[in_dtype], B, img, img, C, P, ptr(out), F16, stream()))
    ref = x[:, : g * P, : g * P].reshape(B, g, P, g, P, C).permute(0, 1, 3, 2, 4, 5).reshape(B * g * g, P * P * C).half()
    assert torch.equal(out, ref)


def test_embed_l2_logits(lib):
    B, T, D, V = 4, 9, 128, 50
    ids = torch.randint(0, V, (B, T), device=DEV, dtype=torch.int32)
    table, pos = torch.randn(V, D, device=DEV), torch.randn(T, D, device=DEV)
    x = torch.empty(B * T, D, device=DEV)
    check(lib, lib.jimm_k_embed(ptr(ids), ptr(table), ptr(pos), ptr(x), B, T, D, V, stream()))
    assert torch.equal(x.reshape(B, T, D), table[ids.long()] + pos)
    Bi, Bt, E = 70, 133, 96
    ie, te = torch.randn(Bi, E, device=DEV), torch.randn(Bt, E, device=DEV)
    i_n, t_n = torch.empty_like(ie), torch.empty_like(te)
    check(lib, lib.jimm_k_l2_normalize(ptr(ie), ptr(i_n), E, Bi, E, stream()))
    check(lib, lib.jimm_k_l2_normalize(ptr(te), ptr(t_n), E, Bt, E, stream()))
    assert rel_err(i_n, ie.double() / ie.double().norm(dim=-1, keepdim=True)) < 1e-6
    sc, bs = torch.tensor([2.3], device=DEV), torch.tensor([-1.7], device=DEV)
    out = torch.empty(Bi, Bt, device=DEV)
    check(lib, lib.jimm_k_logits(ptr(i_n), ptr(t_n), ptr(sc), ptr(bs), ptr(out), Bi, Bt, E, Bt, stream()))
    ref = math.exp(2.3) * (i_n.double() @ t_n.double().T) - 1.7
    assert rel_err(out, ref) < 1e-6
    check(lib, lib.jimm_k_logits(ptr(i_n), ptr(t_n), ptr(sc), None, ptr(out), Bi, Bt, E, Bt, stream()))
    assert rel_err(out, ref + 1.7) < 1e-6


@pytest.mark.parametrize("Bi,Bt,E", [(70, 133, 100), (5, 300, 50), (64, 64, 7), (129, 65, 1024)])
def test_logits_tile_shapes(lib, Bi, Bt, E):
    """logits_tile.cuh: E % 16 != 0 on the 128-bit path (100), the scalar fallback for E % 4 != 0 (50, 7), ragged row / column tiles and a
    strided (sliced) text operand."""
    a = torch.nn.functional.normalize(torch.randn(Bi, E, device=DEV), dim=-1)
    b = torch.nn.functional.normalize(torch.randn(Bt, E, device=DEV), dim=-1)
    sc, bs = torch.tensor([1.1], device=DEV), torch.tensor([0.4], device=DEV)
    out = torch.full((Bi, Bt + 3), 7.0, device=DEV)  # row stride larger than Bt: the columns beyond Bt must stay untouched
    check(lib, lib.jimm_k_logits(ptr(a), ptr(b), ptr(sc), ptr(bs), ptr(out), Bi, Bt, E, Bt + 3, stream()))
    ref = math.exp(1.1) * (a.double() @ b.double().T) + 0.4
    assert rel_err(out[:, :Bt], ref) < 1e-6
    assert torch.all(out[:, Bt:] == 7.0)


def test_bad_arguments_return_errors(lib):
    A = torch.zeros(8, 8, device=DEV).half()
    out = torch.zeros(8, 6, device=DEV)
    rc = lib.jimm_k_gemm(0, F16, ptr(A), 8, ptr(A), 8, 8, 6, 8, None, 0, None, None, 0, ptr(out), F32, 4, 0, 0, 0, 0, stream())
    assert rc == -1 and b"ldo" in lib.jimm_last_error()
    A7 = torch.zeros(8, 7, device=DEV).half()
    rc = lib.jimm_k_gemm(0, F16, ptr(A7), 7, ptr(A7), 7, 8, 8, 7, None, 0, None, None, 0, ptr(out), F32, 8, 0, 0, 0, 0, stream())
    assert rc == -1 and b"16-byte aligned" in lib.jimm_last_error()
    for bad in (-1, 4, 7):  # out_type codes are 0..3 (3 = fp32 rounded to tf32)
        rc = lib.jimm_k_gemm(0, F16, ptr(A), 8, ptr(A), 8, 8, 8, 8, None, 0, None, None, 0, ptr(out), bad, 8, 0, 0, 0, 0, stream())
        assert rc == -1 and b"out_type" in lib.jimm_last_error()
        rc = lib.jimm_k_gemm(1, F16, ptr(A), 8, ptr(A), 8, 8, 8, 8, None, 0, None, None, 0, ptr(out), bad, 8, 0, 0, 0, 0, stream())
        assert rc == -1 and b"out_type" in lib.jimm_last_error()
        y = torch.zeros(2, 8, device=DEV)
        rc = lib.jimm_k_layernorm(ptr(y), 8, 1, 0, None, ptr(y), ptr(y), 1e-6, ptr(y), bad, 8, 2, 8, stream())
        assert rc == -1 and b"out_type" in lib.jimm_last_error()
    x = torch.zeros(2, 6, device=DEV)
    rc = lib.jimm_k_layernorm(ptr(x), 6, 1, 0, None, ptr(x), ptr(x), 1e-6, ptr(x), F32, 6, 2, 6, stream())
    assert rc == -1

