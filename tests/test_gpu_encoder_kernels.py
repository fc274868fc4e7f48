"""Each encoder kernel on its own against a float64 reference computed from the same fp16 inputs, with an error bound
per element, at the shapes and edges where the kernels change behaviour; the whole forward at the benchmark's scale.

Bounds (ulp(x): spacing of fp16 numbers at |x|, 2^-24 below the normal range).  A kernel rounds an fp32 value y to
fp16 once, so |out - ref| <= ulp(ref) + |y - ref| (one ulp, not half, because y may sit in the binade above ref):

* GEMM:      ulp(ref) + C_GEMM (|A| |W|^T)_ij.  GELU: 2 ulp(ref) (the epilogue's GELU is <= 1 ulp from the erf form,
             tests/test_gelu_restatement.py) + 1.13 C_GEMM (|A| |W|^T)_ij (max |GELU'| = 1.13).  Residual: + ulp(dense),
             because the pair kernel (gemm_tn_pair_kernel, every N % 256 == 0 up to 4096) rounds the dense part to fp16
             before it adds the residual (HF BertSelfOutput / BertOutput order); gemm_tn_kernel adds it in fp32, which
             the same bound covers.
* LayerNorm: ulp(ref) + C_LN (|gamma| rstd mean_j|x_j| + |ref - beta|): the fp32 mean is off by at most a multiple of
             mean|x|, and the fp32 variance / rsqrt give a relative error of the normalised value.
* Attention: ulp(ref) + 2^-11 sum_j p_j |v_j| (probabilities are rounded to fp16 before P V).

C_GEMM and C_LN are set from errors measured on a B200 (1000 W power limit): the largest (|out - ref| - the bound's
rounding terms at half their size) / scale over every case and every epilogue of this file, rounded up to a power of
two.  The "MEASURED" lines of profiles/r03_encoder_kernels.log hold the per-case values.  For attention the same
measurement found no error beyond ulp(ref) / 2 + 0.97 x 2^-11 sum_j p_j |v_j|, so it has no such constant -- and its
margin is thin: in the NQ mix (rows whose ref is near 0, where ulp(ref) is small) the probability-rounding term is
used to 97 %.  The kernels are deterministic, so this does not flake, but a change in how the attention kernels round
(for example normalising the probabilities after P V instead of before rounding them) may fail that case without a
real bug; look at the MEASURED line before concluding either way.
The CPU tests at the end check that the bounds still reject a kernel that is wrong in the ways kernels go wrong.

Guards: every output is a view into a buffer filled with a sentinel (an fp16 NaN pattern).  The kernels take no row
stride, so what lies past the declared shape is the trailing rows; they and a lead-in before the output must come back
unchanged.  Inputs are followed by rows of large values that a kernel reading past its rows would pick up."""
import ctypes
import json
import os

import numpy as np
import pytest
import torch

from oracle import bert_oracle as BO

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
EPI_BIAS, EPI_GELU, EPI_RESIDUAL = 0, 1, 2
ROWS_REVERSED = 0x100                       # RSB_GEMM_ROWS_REVERSED (include/rsb.h)

C_GEMM = 2.0 ** -20     # measured 5.0e-7 over both kernels and all epilogues (bias, M = 9473, N = 768, K = 3072; GELU
                        # 1.0e-7, residual 4.3e-7): the tensor cores' fp32 accumulation
C_LN = 2.0 ** -22       # measured 1.4e-7 (T = 41990)

SENTINEL = 0x7E5A                           # fp16 NaN bit pattern
LEAD = 256                                  # sentinel elements before an output (512 bytes keep its alignment)


# ---- bounds and guards (pure torch, checked on the CPU at the end of this file) --------------------------------------

def ulp16(x):
    return torch.exp2(torch.floor(torch.log2(x.abs().clamp_min(2.0 ** -14))) - 10)


def gemm_bound(ref, dense, absprod, epi):
    if epi == EPI_GELU:
        return 2 * ulp16(ref) + 1.13 * C_GEMM * absprod
    b = ulp16(ref) + C_GEMM * absprod
    return b + ulp16(dense) if epi == EPI_RESIDUAL else b


def ln_bound(ref, rstd, mean_abs, gamma, beta):
    return ulp16(ref) + C_LN * (gamma.double().abs() * rstd * mean_abs + (ref - beta.double()).abs())


def ln_violations(out, x, ref, rstd, mean_abs, gamma, beta):
    """Elements outside ln_bound, and every element of a constant row that is not beta exactly.  (The bound's mean
    term is loose for such rows -- rstd is 1 / sqrt(eps) -- but the fp32 sum of 768 copies of an fp16 value is exact,
    and so is the mean.)"""
    bad = violations(out, ref, ln_bound(ref, rstd, mean_abs, gamma, beta))
    const = (x == x[:, :1]).all(dim=1, keepdim=True)
    return bad | (const & (out != beta))


def attention_bound(ref, pv_abs):
    return ulp16(ref) + 2.0 ** -11 * pv_abs


def violations(out, ref, bound):
    return ~((out.double() - ref).abs() <= bound)          # NaN counts as a violation


def assert_within(out, ref, bound, what, bad=None):
    bad = violations(out, ref, bound) if bad is None else bad
    if bool(bad.any()):
        err = (out.double() - ref).abs()
        over = torch.where(bad, (err - bound).nan_to_num(float("inf")), torch.full_like(err, -float("inf")))
        i = int(over.argmax())
        idx = np.unravel_index(i, tuple(out.shape))
        raise AssertionError(f"{what}: {int(bad.sum())} of {out.numel()} elements outside the bound; worst at {idx}: "
                             f"out {out.reshape(-1)[i].item()!r} ref {ref.reshape(-1)[i].item()!r} "
                             f"bound {bound.reshape(-1)[i].item()!r}")


class Guarded:
    """fp16 [rows, cols] output inside a sentinel-filled buffer: LEAD elements before it, tail_rows rows after it."""

    def __init__(self, rows, cols, device, tail_rows=256):
        self.n = rows * cols
        self.buf = torch.full((LEAD + self.n + tail_rows * cols,), SENTINEL, dtype=torch.int16, device=device)
        self.out = self.buf[LEAD:LEAD + self.n].view(torch.float16).view(rows, cols)

    def untouched(self):
        return bool((self.buf[:LEAD] == SENTINEL).all()) and bool((self.buf[LEAD + self.n:] == SENTINEL).all())


def with_garbage_rows(x, rows=128, value=300.0):
    """x as the leading rows of a larger tensor whose remaining rows hold `value`."""
    buf = torch.full((x.shape[0] + rows, x.shape[1]), value, dtype=x.dtype, device=x.device)
    buf[: x.shape[0]] = x
    return buf[: x.shape[0]]


def measured(kind, case, **vals):
    """One line of the measurement log (run with -s to see it)."""
    print("MEASURED " + json.dumps({"kind": kind, "case": case, **{k: float(v) for k, v in vals.items()}}))


def _excess(out, ref, minus, scale):
    """max over elements of (|out - ref| - minus) / scale, elements with scale 0 left out."""
    e = ((out.double() - ref).abs() - minus).clamp_min(0.0)
    m = scale > 0
    return float((e[m] / scale[m]).max()) if bool(m.any()) else 0.0


# ---- GPU side --------------------------------------------------------------------------------------------------------

def _lib():
    from retrieval_scaling_b200 import _lib as lib_mod
    return lib_mod.lib()


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return ctypes.c_void_p(t.data_ptr() if t is not None else 0)


def run_gemm(A, W, bias, res, epi, rev, C):
    L = _lib()
    M, K = A.shape
    rc = L.rsb_gemm_f16(_p(A), _p(W), _p(bias), _p(res), _p(C), M, W.shape[0], K, epi | (ROWS_REVERSED if rev else 0),
                        _stream())
    assert rc == 0, L.rsb_bert_last_error()
    torch.cuda.synchronize()


@pytest.fixture(scope="module")
def bert():
    """An encoder handle for the attention / LayerNorm entries (eps 1e-12 as BERT; the weights are not used)."""
    from retrieval_scaling_b200.encoder import B200Contriever
    return B200Contriever(dict(num_hidden_layers=1, vocab_size=16, layer_norm_eps=1e-12))


GEMM_M = [1, 127, 129, 255, 257, 9473, 41984 + 37]
GEMM_NK = [(768, 768), (2304, 768), (3072, 768), (768, 3072), (4096, 64), (4352, 768), (1152, 768)]


def pair_kernel_expected(N):
    """gemm_tn_pair_kernel takes N % 256 == 0 up to 4096 (its fp32 bias lives in shared memory); gemm_tn_kernel the
    rest -- here (4352, 768) and (1152, 768)."""
    return N % 256 == 0 and N <= 4096


@pytest.mark.gpu
@pytest.mark.parametrize("N,K", GEMM_NK, ids=[f"N{n}_K{k}" for n, k in GEMM_NK])
def test_gemm_takes_the_expected_kernel(N, K):
    """rsb_gemm_f16 runs the kernel the forward runs for the same N, so the parity cases below cover both GEMM kernels.
    Both give results within the same bounds, so no parity case would notice calls routed to the other kernel."""
    A = torch.randn(300, K, device="cuda").half()
    W = torch.randn(N, K, device="cuda").half()
    bias = torch.zeros(N, device="cuda").half()
    C = torch.empty(300, N, device="cuda", dtype=torch.float16)
    run_gemm(A, W, bias, None, EPI_BIAS, True, C)                    # module attributes set outside the trace
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run_gemm(A, W, bias, None, EPI_BIAS, True, C)
    names = [e.name for e in prof.events() if "gemm_tn" in e.name]
    want, other = ("gemm_tn_pair_kernel", "gemm_tn_kernel") if pair_kernel_expected(N) else ("gemm_tn_kernel", "gemm_tn_pair_kernel")
    assert any(want in n for n in names) and not any(other in n for n in names), names


@pytest.mark.gpu
@pytest.mark.parametrize("rev", [False, True], ids=["rows_fwd", "rows_rev"])
@pytest.mark.parametrize("N,K", GEMM_NK, ids=[f"N{n}_K{k}" for n, k in GEMM_NK])
@pytest.mark.parametrize("M", GEMM_M, ids=[f"M{m}" for m in GEMM_M])
def test_gemm_matches_f64(M, N, K, rev):
    """All three epilogues.  For the pair kernel (74 clusters on 148 SMs), M = 9473 and 42021 give every cluster
    several tiles, so the tile loop, the TMEM accumulator double buffer and the barrier phases across tiles all run, in
    both row orders.  gemm_tn_kernel (one tile per CTA, no order) ignores RSB_GEMM_ROWS_REVERSED: its rows_rev cases
    only check that the flag is accepted and changes nothing.  Row invariance: each row of C is computed from its own
    row of A with the same instructions wherever its tile falls and in whichever order the tiles are visited, so C[:m2]
    of A[:m2] in the other row order is bit-identical."""
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(M * 7 + N * 3 + K)
    A = with_garbage_rows(torch.randn(M, K, generator=g, device=dev).half())
    W = (torch.randn(N, K, generator=g, device=dev) * 0.04).half()
    bias = (torch.randn(N, generator=g, device=dev) * 0.1).half()
    R = with_garbage_rows(torch.randn(M, N, generator=g, device=dev).half())
    m2 = M // 2 + 1
    for epi in (EPI_BIAS, EPI_GELU, EPI_RESIDUAL):
        res = R if epi == EPI_RESIDUAL else None
        C = Guarded(M, N, dev)
        run_gemm(A, W, bias, res, epi, rev, C.out)
        assert C.untouched(), f"epilogue {epi}: a store landed outside C[{M}, {N}]"
        ref, dense, absprod = BO.gemm_f64(A, W, bias, res, gelu=epi == EPI_GELU)
        # the bound's rounding terms at half size; the GELU's 1-ulp approximation term at full size
        if epi == EPI_GELU:
            minus, scale = 1.5 * ulp16(ref), 1.13 * absprod
        elif epi == EPI_RESIDUAL:
            minus, scale = 0.5 * (ulp16(ref) + ulp16(dense)), absprod
        else:
            minus, scale = 0.5 * ulp16(ref), absprod
        measured("gemm", f"M{M}_N{N}_K{K}_rev{int(rev)}_epi{epi}", c=_excess(C.out, ref, minus, scale),
                 max_err_ulp=float(((C.out.double() - ref).abs() / ulp16(ref)).max()))
        del minus, scale
        assert_within(C.out, ref, gemm_bound(ref, dense, absprod, epi), f"gemm epilogue {epi}")
        del ref, dense, absprod
        C2 = Guarded(m2, N, dev)
        run_gemm(A[:m2], W, bias, res[:m2] if res is not None else None, epi, not rev, C2.out)
        assert C2.untouched()
        assert torch.equal(C2.out.view(torch.int16), C.out[:m2].view(torch.int16)), \
            f"epilogue {epi}: rows of C depend on M or on the row order"


LN_T = [1, 8, 3552, 3553, 41990]


def _ln_rows(T, rng):
    """Rows of four kinds: ordinary, constant, around +-1000 with small noise (fp16 spacing 0.5 there), near +-65504."""
    kind = rng.choice(4, size=T, p=[0.7, 0.1, 0.1, 0.1])
    if T > 1:
        kind[-1] = 1
    if T > 3552:
        kind[3552] = 3                                     # the first row that is some warp's second row
    x = rng.normal(rng.normal(0, 3, (T, 1)), rng.uniform(0.05, 5, (T, 1)), (T, 768))
    sign = np.where(rng.random((T, 1)) < 0.5, -1.0, 1.0)
    x = np.where(kind[:, None] == 1, rng.uniform(-100, 100, (T, 1)), x)
    x = np.where(kind[:, None] == 2, sign * (1000 + rng.normal(0, 2, (T, 768))), x)
    x = np.where(kind[:, None] == 3, sign * (65504 - 32 * rng.integers(0, 64, (T, 768))), x)
    return torch.from_numpy(x).half(), kind


@pytest.mark.gpu
@pytest.mark.parametrize("T", LN_T, ids=[f"T{t}" for t in LN_T])
def test_layernorm_matches_f64(T, bert):
    """layernorm_rows_kernel runs min(ceil(T / 8), 3 x SMs) blocks of 8 warps: 3552 warps on 148 SMs.  T <= 3552 gives
    each warp at most one row; T = 3553 gives one warp a second row, T = 41990 about 12 rows per warp, so the
    prefetch of the next row is exercised.  Constant rows must give beta exactly."""
    rng = np.random.default_rng(T)
    x, _ = _ln_rows(T, rng)
    x = with_garbage_rows(x.cuda(), value=-3000.0)
    gamma = (1 + 0.1 * torch.randn(768, generator=torch.Generator().manual_seed(T))).half().cuda()
    beta = (0.1 * torch.randn(768, generator=torch.Generator().manual_seed(T + 1))).half().cuda()
    out = Guarded(T, 768, "cuda")
    L = _lib()
    rc = L.rsb_bert_layernorm(bert._h, _p(x), T, _p(gamma), _p(beta), _p(out.out), _stream())
    assert rc == 0, L.rsb_bert_last_error()
    torch.cuda.synchronize()
    assert out.untouched(), "a store landed outside out[T, 768]"
    ref, rstd, mean_abs = BO.layernorm_f64(x, gamma, beta, 1e-12)
    scale = gamma.double().abs() * rstd * mean_abs + (ref - beta.double()).abs()
    measured("layernorm", f"T{T}", c=_excess(out.out, ref, 0.5 * ulp16(ref), scale),
             max_err_ulp=float(((out.out.double() - ref).abs() / ulp16(ref)).max()))
    bound = ln_bound(ref, rstd, mean_abs, gamma, beta)
    assert_within(out.out, ref, bound, "layernorm (constant rows must give beta exactly)",
                  bad=ln_violations(out.out, x, ref, rstd, mean_abs, gamma, beta))


ATT_LENGTHS = [1, 8, 9, 16, 17, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 511, 512]


def _nq_lengths(n):
    return [int(v) for v in np.resize(np.load(os.path.join(GOLD, "nq_open_token_lengths.npy")), n)]


ATT_CASES = {f"S{s}": [s, 3, s] for s in ATT_LENGTHS}
# one 512-token sequence and many 33-token ones: the flash grid (2 blocks per SM) is smaller than the 121 x 12 x 4 work
# items, so blocks walk several items and skip those whose query block starts past the sequence end
ATT_CASES["flash_grid_smaller_than_work"] = [512] + [33] * 120
ATT_CASES["nq_mix_2048"] = "nq"


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(ATT_CASES))
def test_attention_matches_f64(case, bert):
    """Sequences of up to 32 tokens take attention_mma32_kernel (one warp, key tiles of 8 and 16-key P V steps), longer
    ones attention_flash_kernel (blocks of 128 queries, key blocks of 32); the lengths sit on both kernels' tile edges.
    Each length appears twice, once in the middle of the batch and once at its end, next to a 3-token sequence."""
    lens = _nq_lengths(2048) if ATT_CASES[case] == "nq" else ATT_CASES[case]
    cu = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    T = int(cu[-1])
    g = torch.Generator(device="cuda").manual_seed(len(lens) * 1000 + max(lens))
    qkv = with_garbage_rows((torch.randn(T, 3 * 768, generator=g, device="cuda") * 1.5).half(), value=40.0)
    cu_d = torch.from_numpy(cu).cuda()
    ctx = Guarded(T, 768, "cuda")
    L = _lib()
    rc = L.rsb_bert_attention(bert._h, _p(qkv), _p(cu_d), len(lens), T, max(lens), _p(ctx.out), _stream())
    assert rc == 0, L.rsb_bert_last_error()
    torch.cuda.synchronize()
    assert ctx.untouched(), "a store landed outside ctx[T, 768]"
    ref, pv_abs = BO.attention_f64(qkv, cu)
    # share of the 2^-11 term used beyond half an ulp (<= 1 means the bound holds with half an ulp to spare)
    measured("attention", case, p_term_share=_excess(ctx.out, ref, 0.5 * ulp16(ref), 2.0 ** -11 * pv_abs),
             max_err_ulp=float(((ctx.out.double() - ref).abs() / ulp16(ref)).max()))
    assert_within(ctx.out, ref, attention_bound(ref, pv_abs), f"attention {case}")


def _forward_batch(kind, vocab, rng):
    if kind == "nq2048":
        lens = np.array(_nq_lengths(2048))
    else:
        lens = rng.integers(33, 513, 64)
        lens[0] = 512
    S = int(lens.max())
    ids = torch.from_numpy(rng.integers(1, vocab, (len(lens), S)))
    mask = (torch.arange(S)[None, :] < torch.from_numpy(lens)[:, None]).long()
    return (ids * mask).cuda(), mask.cuda(), lens


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["nq2048", "passages64"])
def test_forward_at_bench_scale(kind):
    """The benchmark's query batch (2048 NQ-length sequences, about 41k tokens) and 64 passages of 33..512 tokens
    through a 2-layer model, mean and CLS pooling, against the fp32 and fp16 torch oracles with the bound of
    test_gpu_encoder.py::test_encoder_matches_reference_golden_and_fp16_oracle.  Two runs are bit-identical, and 32
    sequences encoded alone give the rows they get in the big batch bit for bit: every kernel computes a row or a
    (sequence, head) from its own data only, in an order that does not depend on the rest of the batch."""
    from retrieval_scaling_b200.encoder import BERT_BASE, B200Contriever, random_state_dict
    cfg = dict(BERT_BASE, num_hidden_layers=2)
    sd = random_state_dict(cfg, 11)
    rng = np.random.default_rng(0 if kind == "nq2048" else 1)
    ids, mask, lens = _forward_batch(kind, cfg["vocab_size"], rng)
    sample = rng.choice(len(lens), 32, replace=False)
    for pooling in ("average", "cls"):
        model = B200Contriever(cfg, pooling)
        model.load_state_dict(sd)
        out = model(input_ids=ids, attention_mask=mask)
        again = model(input_ids=ids, attention_mask=mask)
        assert torch.equal(out.view(torch.int16), again.view(torch.int16)), "two runs of the same batch differ"
        for i in sample:
            n = int(lens[i])
            alone = model(input_ids=ids[i:i + 1, :n], attention_mask=mask[i:i + 1, :n])
            assert torch.equal(alone[0].view(torch.int16), out[i].view(torch.int16)), f"sequence {i} alone differs"
        out = out.float().cpu()
        with torch.no_grad():
            gold = BO.bert_forward(sd, cfg, ids, mask, None, pooling, dtype=torch.float32).float().cpu()
            half = BO.bert_forward(sd, cfg, ids, mask, None, pooling, dtype=torch.float16).float().cpu()
        cos_gold = torch.nn.functional.cosine_similarity(out, gold, dim=1).min().item()
        cos_half = torch.nn.functional.cosine_similarity(out, half, dim=1).min().item()
        err_gold = (out - gold).abs().max().item()
        err_half_ref = (half - gold).abs().max().item()
        measured("forward", f"{kind}_{pooling}", cos_gold=cos_gold, cos_half=cos_half, err_gold=err_gold,
                 err_half_ref=err_half_ref)
        assert cos_gold >= 0.9999 and cos_half >= 0.9999, (cos_gold, cos_half)
        assert err_gold <= max(2.0 * err_half_ref, 2e-2), (err_gold, err_half_ref)


# ---- the bounds tell a wrong kernel apart (CPU) ------------------------------------------------------------------------

def test_gemm_bound_rejects_wrong_results():
    g = torch.Generator().manual_seed(0)
    M, N, K = 256, 256, 256
    A = torch.randn(M, K, generator=g).half()
    W = (torch.randn(N, K, generator=g) * 0.04).half()
    bias = (torch.randn(N, generator=g) * 0.1).half()
    R = torch.randn(M, N, generator=g).half()

    def kernel_like(A_, bias_, epi):                       # fp16 rounding in the kernel's order
        res = R if epi == EPI_RESIDUAL else None
        ref, dense, _ = BO.gemm_f64(A_, W, bias_, res, gelu=epi == EPI_GELU)
        if epi == EPI_RESIDUAL:
            return (dense.half().double() + R.double()).half()
        return ref.half()

    for epi in (EPI_BIAS, EPI_GELU, EPI_RESIDUAL):
        ref, dense, absprod = BO.gemm_f64(A, W, bias, R if epi == EPI_RESIDUAL else None, gelu=epi == EPI_GELU)
        bound = gemm_bound(ref, dense, absprod, epi)
        good = kernel_like(A, bias, epi)
        assert not bool(violations(good, ref, bound).any()), epi
        swapped = good.clone()
        swapped[[5, 100]] = swapped[[100, 5]]               # two rows of the first 128-row tile
        assert bool(violations(swapped, ref, bound).any()), epi
        A_gap = A.clone()
        A_gap[:, 64:128] = 0                               # one 64-wide K block left out
        assert bool(violations(kernel_like(A_gap, bias, epi), ref, bound).any()), epi
        assert bool(violations(kernel_like(A, torch.roll(bias, 1), epi), ref, bound).any()), epi


def _attention_probs_in_half(qkv, cu, drop_last_key_of=None):
    """Attention with the probabilities rounded to fp16 before P V (as the kernels do), optionally without the last
    key of one sequence."""
    x = qkv.double()
    ctx = torch.zeros((x.shape[0], 768), dtype=torch.float64)
    for b in range(len(cu) - 1):
        s = x[cu[b]:cu[b + 1]].view(-1, 3, 12, 64).permute(1, 2, 0, 3)
        q, k, v = s[0], s[1], s[2]
        if b == drop_last_key_of:
            k, v = k[:, :-1], v[:, :-1]
        p = torch.softmax(q @ k.transpose(-1, -2) * 0.125, dim=-1).half().double()
        ctx[cu[b]:cu[b + 1]] = (p @ v).permute(1, 0, 2).reshape(-1, 768)
    return ctx.half()


def test_attention_bound_rejects_wrong_results():
    g = torch.Generator().manual_seed(1)
    cu = [0, 9, 49, 66]
    qkv = (torch.randn(66, 3 * 768, generator=g) * 1.5).half()
    ref, pv_abs = BO.attention_f64(qkv, cu)
    bound = attention_bound(ref, pv_abs)
    assert not bool(violations(ref.half(), ref, bound).any())
    assert not bool(violations(_attention_probs_in_half(qkv, cu), ref, bound).any())
    for b in range(3):
        assert bool(violations(_attention_probs_in_half(qkv, cu, drop_last_key_of=b), ref, bound).any()), b


def test_layernorm_bound_rejects_wrong_results():
    x, kind = _ln_rows(64, np.random.default_rng(2))
    gamma = (1 + 0.1 * torch.randn(768, generator=torch.Generator().manual_seed(3))).half()
    beta = (0.1 * torch.randn(768, generator=torch.Generator().manual_seed(4))).half()
    ref, rstd, mean_abs = BO.layernorm_f64(x, gamma, beta, 1e-12)
    good = ref.half()
    assert not bool(ln_violations(good, x, ref, rstd, mean_abs, gamma, beta).any())
    assert (kind == 1).sum() >= 2
    x64 = x.double()
    mean = x64.mean(dim=1, keepdim=True)
    for r in range(63):                                    # row r normalised with row r + 1's statistics
        if kind[r] == 1 and kind[r + 1] == 1:
            continue                                       # two constant rows: both give beta, nothing to see
        bad = good.clone()
        bad[r] = ((x64[r] - mean[r + 1]) * rstd[r + 1] * gamma.double() + beta.double()).half()
        assert bool(ln_violations(bad, x, ref, rstd, mean_abs, gamma, beta).any()), r


def test_guard_detects_one_stray_store():
    for pos in (0, LEAD - 1, LEAD + 12 * 8, LEAD + 12 * 8 + 999):
        G = Guarded(12, 8, "cpu", tail_rows=128)
        G.out.fill_(1.0)
        assert G.untouched()
        G.buf[pos] = 0
        assert G.untouched() == (LEAD <= pos < LEAD + 96), pos
