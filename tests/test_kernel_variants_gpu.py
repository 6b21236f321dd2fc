"""The kernel variants the model forward runs but the plain per-kernel entries do not reach: reversed walks, every schedule regime of
the tcgen05 GEMM, the token-scatter patch GEMM, tf32-rounded outputs and plans run on fewer rows than they were built for.

References are fp64 on the GPU with the operands pre-rounded to the kernel's operand type.  Every element is checked on its own: it may
differ from the fp64 reference, rounded to the output type, by one ulp of that type plus an fp32-accumulation allowance of
2e-5 * max|ref|.  Plain stores go into NaN-filled outputs (a tile never stored stays NaN); residual variants add into a random x0 (a
tile added twice or never is off by a whole A . B^T).

The one test without a GPU checks the shape chooser: for several SM counts, every GEMM regime below is actually reached."""

import math
import os
from collections import namedtuple

import pytest
import torch

from gpu_util import BF16, CODE, F16, F32, check, gelu_tanh, ptr, quick_gelu, rel_err, stream

DEV = "cuda"
TF32 = 3  # out_type code of the per-kernel entries: fp32 rounded to tf32
BM, BN = 128, 256  # GEMM tile: 128 rows per CTA (256 per CTA pair) x 256 columns

# ---------------------------------------------------------------------------------------------------------------------------------
# The GEMM schedule (gemm.cu, launch_one), restated.
Sched = namedtuple("Sched", "mode tiles tail parts full rounds")


def _env_flag(name):
    try:
        return int(os.environ.get(name, "1")) != 0
    except ValueError:
        return False


def schedule(M, N, sms, out16, tma=True, pair=None, split=None):
    """mode 'pair' (256 x 256 tiles on CTA pairs) or 'single' (128 x 256 tiles), tiles, tail (tiles of the last round), parts (column
    slices per tail tile), full (whole tiles), rounds.  out16: 16-bit output (64-column store boxes, so at most 2 slices); tma: the
    TMA epilogue (mode 2) -- the LSU epilogues always run single CTAs."""
    pair = _env_flag("JIMM_GEMM_PAIR") if pair is None else pair
    split = _env_flag("JIMM_GEMM_TAIL_SPLIT") if split is None else split
    n_tiles = -(-N // BN)
    if tma and pair and M >= 512:
        tiles = -(-M // (2 * BM)) * n_tiles
        max_pairs = sms // 2
        tail, parts = tiles % max_pairs, 1
        max_parts = 2 if out16 else 4
        if split and tail > 0:
            while parts * 2 <= max_parts and tail * parts * 2 <= max_pairs:
                parts *= 2
        full = tiles - tail if parts > 1 else tiles
        vtiles = full + (tiles - full) * parts
        return Sched("pair", tiles, tail, parts, full, -(-vtiles // min(vtiles, max_pairs)))
    tiles = -(-M // BM) * n_tiles
    return Sched("single", tiles, 0, 1, tiles, -(-tiles // min(tiles, sms)))


REGIMES = {
    "single_many": lambda s, sms: s.mode == "single" and s.tiles > sms,
    "pair_sliced2": lambda s, sms: s.mode == "pair" and s.full == 0 and s.parts == 2,
    "pair_sliced4": lambda s, sms: s.mode == "pair" and s.full == 0 and s.parts == 4,
    "pair_mixed2": lambda s, sms: s.mode == "pair" and s.full > 0 and s.parts == 2,
    "pair_mixed4": lambda s, sms: s.mode == "pair" and s.full > 0 and s.parts == 4,
    "pair_tail_unsplit": lambda s, sms: s.mode == "pair" and s.tiles > sms // 2 and s.tail > 0 and s.parts == 1,
    "pair_tail0": lambda s, sms: s.mode == "pair" and s.tail == 0,
    "pair_rounds3": lambda s, sms: s.mode == "pair" and s.rounds >= 3,
}
ONLY_32BIT = {"pair_sliced4", "pair_mixed4"}  # 16-bit outputs never cut a tile into 4 slices
# rows in the last 256-row block (97 / 128: the second CTA of the last pair has no rows), N % 256, K (not a multiple of the k-block)
SHAPE = {
    "pair_sliced2": (97, 64, 592),
    "pair_sliced4": (200, 128, 200),
    "pair_mixed2": (256, 192, 592),
    "pair_mixed4": (97, 64, 200),
    "pair_tail_unsplit": (200, 128, 592),
    "pair_tail0": (128, 64, 200),
    "pair_rounds3": (97, 192, 592),
}


def choose_shape(regime, sms, out16):
    """(M, N, K) whose schedule on `sms` SMs is in `regime` (the smallest tile count that gets there)."""
    if regime == "single_many":  # fewer than 512 rows: single CTAs; 4 row blocks x (sms / 4 + 1) column tiles
        return 500, (sms // 4 + 1) * BN - 64, 200
    rem, nmod, K = SHAPE[regime]
    for t in range(1, 64 * sms):
        for mp in range(2, t + 1):
            if t % mp:
                continue
            M, N = (mp - 1) * 2 * BM + rem, (t // mp - 1) * BN + nmod
            if M >= 512 and REGIMES[regime](schedule(M, N, sms, out16, pair=True, split=True), sms):
                return M, N, K
    return None


def _cases():
    for regime in REGIMES:
        for out in OUTS:
            if regime in ONLY_32BIT and out[0] in ("f16", "bf16"):
                continue
            yield regime, out


OUTS = [("f16", 0), ("f16", 1), ("f16", 2), ("bf16", 0), ("bf16", 1), ("bf16", 2), ("f32", 0), ("tf32", 0), ("tf32", 1), ("res", 0)]


@pytest.mark.parametrize("sms", [148, 132, 160])
def test_shape_chooser_reaches_every_regime(sms):
    for regime in REGIMES:
        for out16 in (True, False):
            if out16 and regime in ONLY_32BIT:
                continue
            shape = choose_shape(regime, sms, out16)
            assert shape is not None, (regime, sms, out16)
            M, N, K = shape
            s = schedule(M, N, sms, out16, pair=True, split=True)
            assert REGIMES[regime](s, sms), (regime, sms, out16, shape, s)
            assert N % BN in (64, 128, 192) and K % 32 != 0
    # the pair regimes the 16-bit outputs cannot reach
    for regime in ONLY_32BIT:
        M, N, _ = choose_shape(regime, sms, False)
        assert schedule(M, N, sms, True, pair=True, split=True).parts == 2


# ---------------------------------------------------------------------------------------------------------------------------------
# per-element comparison
KIND_DTYPE = {"f16": torch.float16, "bf16": torch.bfloat16, "f32": torch.float32, "tf32": torch.float32, "res": torch.float32}
KIND_CODE = {"f16": F16, "bf16": BF16, "f32": F32, "tf32": TF32, "res": F32}
MANT = {"f16": 10, "bf16": 7, "tf32": 10, "f32": 23, "res": 23}
MIN_EXP = {"f16": -14, "bf16": -126, "tf32": -126, "f32": -126, "res": -126}


def round_tf32(x):
    """fp32 -> nearest tf32 (ties to even), still stored as fp32"""
    b = x.float().contiguous().view(torch.int32)
    b = (b + 0xFFF + ((b >> 13) & 1)) & ~0x1FFF
    return b.view(torch.float32)


def round_to(ref, kind):
    if kind == "tf32":
        return round_tf32(ref).double()
    return ref.to(KIND_DTYPE[kind]).double()


def ulp(a, kind):
    """one unit in the last place of |a| (fp64) in the format `kind`"""
    _, e = torch.frexp(a)
    e = torch.where(a > 0, e - 1, torch.full_like(e, MIN_EXP[kind])).clamp_min(MIN_EXP[kind])
    return torch.ldexp(torch.ones_like(a), e - MANT[kind])


def assert_ulp_close(out, ref, kind, what=""):
    """every element of `out` within one ulp of round(ref) (plus 2e-5 * max|ref|); NaN anywhere fails"""
    ref = ref.double()
    r = round_to(ref, kind)
    tol = ulp(torch.maximum(r.abs(), ref.abs()), kind) + 2e-5 * float(ref.abs().max())
    err = (out.double() - r).abs()
    bad = ~(err <= tol)
    if bool(bad.any()):
        idx = bad.nonzero()[0].tolist()
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements off (first at {idx}: got {out[tuple(idx)].item()!r}, "
                             f"ref {ref[tuple(idx)].item()!r}, tol {tol[tuple(idx)].item():.3g})")


def assert_tf32_bits(out, what=""):
    low = out.contiguous().view(torch.int32) & 0x1FFF
    assert int((low != 0).sum()) == 0, f"{what}: {int((low != 0).sum())} stored values are not tf32 (low 13 mantissa bits set)"


def bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


def same_bits(a, b):
    return torch.equal(bits(a), bits(b))


def _operands(M, N, K, dtype, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    A = torch.randn(M, K, device=DEV, generator=g)
    Bw = torch.randn(N, K, device=DEV, generator=g) / math.sqrt(K)
    if dtype == torch.float32:
        A, Bw = round_tf32(A), round_tf32(Bw)
    else:
        A, Bw = A.to(dtype), Bw.to(dtype)
    bias = torch.randn(N, device=DEV, generator=g)
    return A, Bw, bias


def gemm_ex(lib, A, Bw, out, out_type, *, bias=None, act=0, residual=None, tok=(0, 0, 0), run_M=0, reverse=0, mode=2, M=None):
    M = A.shape[0] if M is None else M
    N, K = Bw.shape
    ldo = out.stride(-2)
    check(lib, lib.jimm_k_gemm_ex(CODE[A.dtype], ptr(A), A.stride(0), ptr(Bw), Bw.stride(0), M, N, K, ptr(bias), act, None, ptr(residual),
                                  0 if residual is None else ldo, ptr(out), out_type, ldo, 0, 0, 0, tok[0], tok[1], tok[2], run_M, reverse,
                                  mode, stream()))
    return out


def _act(ref, act):
    return [ref, gelu_tanh(ref), quick_gelu(ref)][act]


def sm_count():
    env = os.environ.get("JIMM_NUM_SMS", "")
    if env.strip().lstrip("-").isdigit() and int(env) > 0:
        return int(env)
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float32], ids=["a16", "abf16", "a32"])
@pytest.mark.parametrize("regime,out", list(_cases()), ids=[f"{r}-{o}{a}" for r, (o, a) in _cases()])
def test_gemm_regime(lib, regime, out, dtype):
    """One schedule regime of the tcgen05 GEMM x one epilogue; reverse = 1 gives the same bits as reverse = 0."""
    kind, act = out
    sms = sm_count()
    M, N, K = choose_shape(regime, sms, kind in ("f16", "bf16"))
    s = schedule(M, N, sms, kind in ("f16", "bf16"))
    print(f"{regime}: M={M} N={N} K={K} sms={sms} {s}")
    assert REGIMES[regime](s, sms), (regime, s)
    A, Bw, bias = _operands(M, N, K, dtype, seed=M * 7 + N)
    ref = A.double() @ Bw.double().T + bias.double()
    runs = []
    for reverse in (0, 1):
        if kind == "res":
            x0 = torch.randn(M, N, device=DEV, generator=torch.Generator(device=DEV).manual_seed(5))
            o = x0.clone()
            gemm_ex(lib, A, Bw, o, F32, bias=bias, residual=o, reverse=reverse)
            expect = x0.double() + ref
        else:
            o = torch.full((M, N), float("nan"), dtype=KIND_DTYPE[kind], device=DEV)
            gemm_ex(lib, A, Bw, o, KIND_CODE[kind], bias=bias, act=act, reverse=reverse)
            expect = _act(ref, act)
        torch.cuda.synchronize()
        runs.append(o)
    assert_ulp_close(runs[0], expect, kind, f"{regime} {kind} act={act}")
    if kind == "tf32":
        assert_tf32_bits(runs[0], regime)
    assert same_bits(runs[0], runs[1]), f"{regime}: reverse = 1 differs from reverse = 0"


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,K", [(777, 1536, 512), (600, 264, 200), (37, 10, 128)])
@pytest.mark.parametrize("act", [0, 1])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_gemm_tf32_output(lib, M, N, K, act, mode):
    """out code 3 through every epilogue: the TMA store (mode 2; N = 10 falls back to mode 0) and both LSU forms, vector and scalar."""
    A, Bw, bias = _operands(M, N, K, torch.float32, seed=M + N + K)
    o = torch.full((M, N), float("nan"), device=DEV)
    gemm_ex(lib, A, Bw, o, TF32, bias=bias, act=act, mode=mode)
    torch.cuda.synchronize()
    assert_tf32_bits(o, "gemm")
    assert_ulp_close(o, _act(A.double() @ Bw.double().T + bias.double(), act), "tf32", f"gemm mode {mode}")


# ---------------------------------------------------------------------------------------------------------------------------------
SCATTER = [(16, 4), (16, 20), (49, 2), (49, 9), (196, 2), (196, 3), (576, 1)]  # (patches per sample n, samples B): B * n_pad < and >= 512


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float32], ids=["a16", "abf16", "a32"])
@pytest.mark.parametrize("K", [768, 592, 3072])
@pytest.mark.parametrize("off", [0, 1])
@pytest.mark.parametrize("n,B", SCATTER)
def test_token_scatter_patch_gemm(lib, n, B, off, K, dtype):
    """The default patch embedding: rows (b, p < n_pad) of A, reduce-added into x[b, p + off] of the position-initialised residual stream
    [B, S = n + off, D]; pad rows (p >= n) are dropped at S, the CLS rows (off = 1) are not touched."""
    D = 768
    n_pad = -(-n // 32) * 32
    S = n + off
    M = B * n_pad
    A, Bw, bias = _operands(M, D, K, dtype, seed=n * 100 + B + K)
    pad = (torch.arange(M, device=DEV) % n_pad) >= n
    A[pad] = float("nan")  # a pad row that leaks into the stream leaves NaN there
    x0 = torch.randn(B, S, D, device=DEV, generator=torch.Generator(device=DEV).manual_seed(n + K))
    sched = schedule(M, D, sm_count(), False)
    outs = []
    for reverse in (0, 1):
        x = x0.clone()
        gemm_ex(lib, A, Bw, x, F32, bias=bias, residual=x, tok=(n_pad, off, S), reverse=reverse)
        torch.cuda.synchronize()
        outs.append(x)
    x = outs[0]
    assert not torch.isnan(x).any(), f"pad rows leaked into the residual stream ({sched})"
    valid = A.reshape(B, n_pad, K)[:, :n].double()
    ref = x0[:, off:].double() + valid @ Bw.double().T + bias.double()
    assert_ulp_close(x[:, off:], ref, "f32", f"token scatter n={n} B={B} off={off} ({sched})")
    if off:
        assert same_bits(x[:, 0], x0[:, 0]), "CLS rows changed"
    assert same_bits(outs[0], outs[1]), "reverse = 1 differs from reverse = 0"


@pytest.mark.gpu
def test_token_scatter_rejects_bad_arguments(lib):
    A = torch.zeros(64, 64, device=DEV).half()
    x = torch.zeros(2, 33, 64, device=DEV)
    y = torch.zeros(2, 33, 64, device=DEV)
    common = (F16, ptr(A), 64, ptr(A), 64, 64, 64, 64, None, 0, None)
    # residual != out
    assert lib.jimm_k_gemm_ex(*common, ptr(y), 64, ptr(x), F32, 64, 0, 0, 0, 32, 1, 33, 0, 0, 2, stream()) == -1
    # 16-bit output
    assert lib.jimm_k_gemm_ex(*common, ptr(x), 64, ptr(x), F16, 64, 0, 0, 0, 32, 1, 33, 0, 0, 2, stream()) == -1
    # pad not a multiple of 32
    assert lib.jimm_k_gemm_ex(*common, ptr(x), 64, ptr(x), F32, 64, 0, 0, 0, 16, 1, 33, 0, 0, 2, stream()) == -1
    # run_M above the planned M
    assert lib.jimm_k_gemm_ex(*common, None, 0, ptr(x), F32, 64, 0, 0, 0, 0, 0, 0, 65, 0, 2, stream()) == -1


# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("res", [False, True], ids=["store16", "residual"])
@pytest.mark.parametrize("plan_M,N,K", [(788, 768, 256), (50432, 256, 256)])
def test_gemm_plan_run_on_fewer_rows(lib, plan_M, N, K, res):
    """A plan built for plan_M rows, run on run_M: rows < run_M are right; the TMA epilogue also writes rows [run_M, ceil32(run_M))
    (whole 32-row boxes, from the A rows there; gemm.cuh, gemm_plan_run); rows >= ceil32(run_M) keep their bits."""
    A, Bw, bias = _operands(plan_M, N, K, torch.float16, seed=plan_M + N)
    ref = A.double() @ Bw.double().T + bias.double()
    x0 = torch.randn(plan_M, N, device=DEV, generator=torch.Generator(device=DEV).manual_seed(9))
    sms = sm_count()
    for run_M in (plan_M, plan_M - 1, 591, 511, 33, 1):
        if res:
            o = x0.clone()
            gemm_ex(lib, A, Bw, o, F32, bias=bias, residual=o, run_M=run_M)
            before, expect, kind = x0, x0.double() + ref, "f32"
        else:
            o = torch.full((plan_M, N), float("nan"), dtype=torch.float16, device=DEV)
            before = o.clone()
            gemm_ex(lib, A, Bw, o, F16, bias=bias, run_M=run_M)
            expect, kind = ref, "f16"
        torch.cuda.synchronize()
        hi = min(plan_M, -(-run_M // 32) * 32)
        what = f"plan {plan_M} run {run_M} ({schedule(run_M, N, sms, not res)})"
        assert_ulp_close(o[:hi], expect[:hi], kind, what)
        assert same_bits(o[hi:], before[hi:]), f"{what}: rows >= ceil32(run_M) were written"
        if not res:  # the LSU epilogue stops at run_M exactly
            o2 = torch.full((plan_M, N), float("nan"), dtype=torch.float16, device=DEV)
            gemm_ex(lib, A, Bw, o2, F16, bias=bias, run_M=run_M, mode=0)
            torch.cuda.synchronize()
            assert same_bits(o2[:run_M], o[:run_M]), f"{what}: LSU and TMA epilogues differ"
            assert torch.isnan(o2[run_M:].float()).all(), f"{what}: LSU epilogue wrote rows >= run_M"


# ---------------------------------------------------------------------------------------------------------------------------------
def _attn_ref(qkv, B, S, H, causal):
    q, k, v = qkv.double().reshape(B, S, 3, H, 64).permute(2, 0, 3, 1, 4)
    w = (q / 8.0) @ k.transpose(-1, -2)
    if causal:
        w = w.masked_fill(~torch.tril(torch.ones(S, S, dtype=torch.bool, device=qkv.device)), float("-inf"))
    return (torch.softmax(w, -1) @ v).permute(0, 2, 1, 3).reshape(B * S, H * 64)


def _attn_cases():
    for S, causal in ((1, 0), (77, 1), (197, 0), (256, 0), (577, 0), (1024, 0)):
        for impl in ("default", "flash"):
            yield S, causal, impl


@pytest.mark.gpu
@pytest.mark.parametrize("S,causal,impl", list(_attn_cases()))
def test_attention_reverse_and_tf32(lib, monkeypatch, S, causal, impl):
    """Every attention kernel (tcgen05 S <= 256, the long-sequence kernel, the mma.sync flash kernel) with more
    (sample, head) items than SMs: reverse = 1 gives the bits of reverse = 0; fp16 in / tf32 out stores tf32 values within one tf32 ulp
    of the same kernel's fp32 output, which is within the attention bound of the fp64 reference."""
    if impl != "default":
        monkeypatch.setenv("JIMM_ATTN_IMPL", impl)
    H = 2
    B = sm_count() // H + 3
    g = torch.Generator(device=DEV).manual_seed(S)
    for io, out_dtypes in ((torch.float16, (torch.float16, torch.float32, "tf32")), (torch.bfloat16, (torch.bfloat16,))):
        qkv = (torch.randn(B * S, 3 * H * 64, device=DEV, generator=g) * 1.5).to(io)
        outs = {}
        for od in out_dtypes:
            code, dt = (TF32, torch.float32) if od == "tf32" else (CODE[od], od)
            pair = []
            for reverse in (0, 1):
                o = torch.full((B * S, H * 64), float("nan"), dtype=dt, device=DEV)
                check(lib, lib.jimm_k_attention_ex(ptr(qkv), CODE[io], ptr(o), code, B, S, H, causal, reverse, stream()))
                pair.append(o)
            torch.cuda.synchronize()
            assert same_bits(pair[0], pair[1]), f"{impl} S={S} {io}->{od}: reverse = 1 differs from reverse = 0"
            outs[od] = pair[0]
        ref = _attn_ref(qkv, B, S, H, causal)
        tol = 3e-3 if io == torch.float16 else 2e-2
        for od, o in outs.items():
            assert not torch.isnan(o.float()).any()
            assert rel_err(o, ref) < tol, (impl, S, od, rel_err(o, ref))
        if "tf32" in outs:
            assert_tf32_bits(outs["tf32"], f"attention {impl}")
            f32 = outs[torch.float32].double()
            err = (outs["tf32"].double() - round_tf32(outs[torch.float32]).double()).abs()
            assert bool((err <= ulp(f32.abs(), "tf32")).all()), f"{impl} S={S}: tf32 output not the tf32 rounding of the fp32 output"


# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["f32", "f16", "bf16", "tf32"])
@pytest.mark.parametrize("D", [768, 1024])
@pytest.mark.parametrize("many", [False, True], ids=["rows333", "rows_gt_32sms"])
def test_layernorm_reverse_and_out_types(lib, kind, D, many):
    rows = 32 * sm_count() + 77 if many else 333
    g = torch.Generator(device=DEV).manual_seed(D + rows)
    x = torch.randn(rows, D, device=DEV, generator=g) * 3 + 1.5
    scale, bias = torch.randn(D, device=DEV, generator=g), torch.randn(D, device=DEV, generator=g)
    outs = []
    for reverse in (0, 1):
        o = torch.full((rows, D), float("nan"), dtype=KIND_DTYPE[kind], device=DEV)
        check(lib, lib.jimm_k_layernorm_ex(ptr(x), D, 1, 0, None, ptr(scale), ptr(bias), 1e-6, ptr(o), KIND_CODE[kind], D, rows, D, reverse,
                                           stream()))
        outs.append(o)
    torch.cuda.synchronize()
    xd = x.double()
    mean = xd.mean(-1, keepdim=True)
    var = ((xd * xd).mean(-1, keepdim=True) - mean * mean).clamp_min(0)
    ref = (xd - mean) * torch.rsqrt(var + 1e-6) * scale.double() + bias.double()
    assert_ulp_close(outs[0], ref, kind, f"layernorm D={D} rows={rows}")
    if kind == "tf32":
        assert_tf32_bits(outs[0], "layernorm")
    assert same_bits(outs[0], outs[1]), "reverse = 1 differs from reverse = 0"


@pytest.mark.gpu
@pytest.mark.parametrize("img,P", [(224, 16), (32, 8), (42, 14)])
def test_patchify_tf32_output(lib, img, P):
    """fp32 image -> tf32 patches (the fp32 compute mode's patch operand), vectorised kernel and generic (patch 14) kernel."""
    B, C = 3, 3
    x = torch.randn(B, img, img, C, device=DEV)
    gsz = img // P
    out = torch.full((B * gsz * gsz, P * P * C), float("nan"), device=DEV)
    check(lib, lib.jimm_k_patchify(ptr(x), F32, B, img, img, C, P, ptr(out), TF32, stream()))
    torch.cuda.synchronize()
    ref = x[:, : gsz * P, : gsz * P].reshape(B, gsz, P, gsz, P, C).permute(0, 1, 3, 2, 4, 5).reshape(B * gsz * gsz, P * P * C)
    assert_tf32_bits(out, "patchify")
    assert_ulp_close(out, ref.double(), "tf32", "patchify")


# ---------------------------------------------------------------------------------------------------------------------------------
# model level: the switches that only change the order of the work or the epilogue that stores it give the same bits
def _vit(dtype, p):
    from jimm_b200.models import VisionTransformer

    m = VisionTransformer(dtype=dtype).eval()
    for k, v in p.items():
        m.set_flat_param(k, v.to(torch.float32))
    return m


def _unset(monkeypatch):
    for name in ("JIMM_L2_ALTERNATE", "JIMM_EPI_MODE_RES", "JIMM_EPI_MODE_16"):
        monkeypatch.delenv(name, raising=False)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
def test_vit_b16_walk_direction_and_epilogues_same_bits(monkeypatch, dtype):
    """ViT-B/16 @224 at B = 4 and 64: JIMM_L2_ALTERNATE=0 (every kernel walks forward) and JIMM_EPI_MODE_RES=0 + JIMM_EPI_MODE_16=0
    (LSU epilogues instead of TMA stores / reduce-adds, row-add patch GEMM instead of the token scatter) give the default's bits."""
    import jimm_oracle as O

    cfg = O.ViTCfg()
    p = O.random_vit_params(cfg, seed=0)
    imgs = {B: O.synthetic_images(B, 224, seed=B).cuda() for B in (4, 64)}
    variants = {"default": {}, "l2_alternate=0": {"JIMM_L2_ALTERNATE": "0"}, "epi_mode=0": {"JIMM_EPI_MODE_RES": "0", "JIMM_EPI_MODE_16": "0"}}
    got = {}
    for name, env in variants.items():
        _unset(monkeypatch)
        for k, v in env.items():
            monkeypatch.setenv(k, v)  # read when the native model is created (first call)
        m = _vit(dtype, p)
        got[name] = {B: m(img) for B, img in imgs.items()}
        got[name]["4, replayed"] = m(imgs[4])  # the second call of a small batch replays a captured graph
        del m
    assert torch.equal(got["default"]["4, replayed"], got["default"][4])
    for name in variants:
        for B in got[name]:
            assert torch.equal(got[name][B], got["default"][B]), f"{name} B={B}: max |diff| {(got[name][B] - got['default'][B]).abs().max().item():.3g}"


@pytest.mark.gpu
def test_clip_medium_walk_direction_and_epilogues_same_bits(monkeypatch):
    import jimm_oracle as O
    from jimm_b200.models import CLIP

    cfg = O.DualCfg(image_resolution=64, vision_layers=2, vision_width=256, vision_patch_size=16, context_length=20, vocab_size=300,
                    transformer_width=128, transformer_heads=2, transformer_layers=2)
    p = O.random_dual_params(cfg, "clip", seed=11)
    img, txt = O.synthetic_images(6, 64).cuda(), O.synthetic_tokens(9, 20, 300, "clip").cuda()
    got = {}
    for name, env in {"default": {}, "l2_alternate=0": {"JIMM_L2_ALTERNATE": "0"},
                      "epi_mode=0": {"JIMM_EPI_MODE_RES": "0", "JIMM_EPI_MODE_16": "0"}}.items():
        _unset(monkeypatch)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        m = CLIP(64, 2, 256, 16, 20, 300, 128, 2, 2, dtype=torch.float16)
        for k, v in p.items():
            m.set_flat_param(k, v.to(torch.float32))
        got[name] = (m.encode_image(img), m.encode_text(txt), m(img, txt))
        del m
    for name, outs in got.items():
        for what, a, b in zip(("image", "text", "logits"), outs, got["default"]):
            assert torch.equal(a, b), f"{name} {what}: max |diff| {(a - b).abs().max().item():.3g}"
