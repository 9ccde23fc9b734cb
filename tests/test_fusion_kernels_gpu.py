"""GPU: the fusion-path kernels through the C ABI against oracle/fusion_oracle.py (float64, fed the same inputs):
attention forward and backward (csrc/attention.cu), the unfused softmax, the resample, the bias column sums and the CTC
head's log-softmax (csrc/fusion_kernels.cu), and the public modes of the tcgen05 GEMM (csrc/gemm_tcgen05.cu).

The cases sit where these kernels go wrong: attention at every tile edge of T (1, 16/17, 32/33, 63-65, 127-129, 191,
192: the 16- and 32-row MMA and TMA extents, the 64-column panels, the second 128-row tile), H = 1, 2, 3, 8 and B up to
64, on random, peaky, near-uniform, tied and large-magnitude score rows; the softmax at T around the 32-lane warp width
with pad columns; the resample when down-sampling, at Tv = Tp, 2 Tp and 1, at Tp = 1, with an empty sample and an empty
batch, for B > 32 (the batch maximum loops over lanes), Ta > 256 (the compaction carries its count across 256-frame
chunks) and D % 8 != 0; column sums over 1 to 64 row chunks with ld > N; log-softmax over V up to 5000 with every
dtype pair; the GEMM with either bias, alpha != 1, accumulate, ragged M, N and K, the element-wise epilogue forced by an
odd ldc or a C one element off alignment, and 3-D operands.

Errors are measured per output against the oracle: for bf16 outputs the max error in bf16 ulps of max(|ref|, RMS/64);
for fp32 outputs the max error over the output's RMS, for column sums over sum |x| of the column; for both the fraction
of elements off by more than one bf16 ulp and the relative norm error.  Output buffers start as NaN or a sentinel, and
every element outside the region an entry point writes must come back bit-identical.

The bounds (BOUNDS) are the worst values over the cases measured on one NVIDIA B200 (1000 W power limit) with at most
2x headroom; the measured worst values are listed next to each bound.  Mutants of the oracle's output, each a plausible
kernel bug, must fall outside the bounds in every case where they change anything, and each must show in some case."""
import ctypes
import math

import pytest
import torch

from oracle import fusion_oracle as fo

gpu = pytest.mark.gpu

bf16, f32, f64, i64 = torch.bfloat16, torch.float32, torch.float64, torch.int64
OK, BAD_ARG, UNSUPPORTED, WORKSPACE, ALIGNMENT = 0, -1, -2, -3, -4
F32, BF16 = 0, 1
_DT = {F32: f32, BF16: bf16}
_BITS = {f32: torch.int32, bf16: torch.int16, i64: i64, torch.uint8: torch.uint8}

# name: (max error, fraction above 1 ulp, relative norm error).  Max is in bf16 ulps for the "ulp" outputs, in RMS for
# "rms", in sum |x| for "sum".  Measured worst over the cases on one NVIDIA B200 at a 1000 W power limit in the comment.
# Every output but the attention gradients is within half an ulp of the float64 value: only the final rounding
# separates them.  The attention gradients' large max-ulp figures are elements that cancel to a small value (the
# "large" score rows, where dS = P (dP - D) subtracts near-equal terms in fp32).  The resample is compared with the
# weights ATen computes for float32 and bf16 tensors (fp32 scale and source index), which the kernel reproduces.
KIND = {"attn.o": "ulp", "attn.lse2": "rms", "attn.dq": "ulp", "attn.dk": "ulp", "attn.dv": "ulp",
        "softmax.P": "ulp", "softmax.dS": "ulp", "resample.out": "ulp", "resample.da_f32": "rms",
        "resample.da_bf16": "ulp", "colsum.out": "sum", "logsm.y_f32": "rms", "logsm.y_bf16": "ulp",
        "logsm.dx": "ulp", "gemm.c_f32": "rms", "gemm.c_bf16": "ulp"}
BOUNDS = {
    "attn.o": (50, 0.00025, 0.0002),          # worst 23.5, 0.000107, 8.13e-05
    "attn.lse2": (1e-06, 0, 2.5e-07),         # worst 4.27e-07, 0, 1.22e-07
    "attn.dq": (640, 0.014, 0.0014),          # worst 319, 0.00687, 0.000719
    "attn.dk": (550, 0.015, 0.0013),          # worst 276, 0.00745, 0.000654
    "attn.dv": (100, 0.0017, 0.0012),         # worst 50.3, 0.000868, 0.000629
    "softmax.P": (1, 0, 0.004),               # worst 0.5, 0, 0.002
    "softmax.dS": (1.15, 0, 0.0048),          # worst 0.577, 0, 0.00241
    "resample.out": (1, 0, 0.0039),           # worst 0.5, 0, 0.00197
    "resample.da_f32": (1e-06, 0, 7e-08),     # worst 5.01e-07, 0, 3.65e-08
    "resample.da_bf16": (1, 0, 0.0033),       # worst 0.5, 0, 0.00166
    "colsum.out": (2.7e-07, 0, 2.3e-07),      # worst 1.37e-07, 0, 1.18e-07
    "logsm.y_f32": (1.4e-05, 0, 3.4e-06),     # worst 7.39e-06, 0, 1.72e-06
    "logsm.y_bf16": (1, 0, 0.0033),           # worst 0.5, 0, 0.00167
    "logsm.dx": (1, 0, 0.0035),               # worst 0.5, 0, 0.00178
    "gemm.c_f32": (2.1e-06, 0, 2.8e-07),      # worst 1.06e-06, 0, 1.42e-07
    "gemm.c_bf16": (1, 0, 0.0033),            # worst 0.5, 0, 0.00167
}


def _lib():
    import multimodal_av_model_b200 as pkg
    return pkg._lib


def _L():
    return _lib().lib()


def _st():
    return _lib().stream_ptr(torch.device("cuda"))


def _cdiv(a, b):
    return -(-a // b)


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _randn(g, *shape, dtype=f32):
    return torch.randn(*shape, generator=g, device="cuda").to(dtype)


def _bits(t):
    return t.view(_BITS[t.dtype])


class Guarded:
    """A device tensor of `shape` filled with `fill` inside a buffer with 64 guard elements on each side (the tensor
    stays 16-byte aligned).  untouched(written) -> True when every element outside `written` (a bool mask of the
    tensor, or None for the whole tensor written) and every guard element still has its old bits."""

    def __init__(self, shape, dtype, fill, pad=64):
        n = math.prod(shape)
        self.buf = torch.full((n + 2 * pad,), fill, dtype=dtype, device="cuda")
        self.t = self.buf[pad:pad + n].view(shape)
        self.pad = pad
        self.snap = None

    def seal(self):
        self.snap = self.buf.clone()
        return self

    def untouched(self, written=None):
        p = self.pad
        b, s = _bits(self.buf), _bits(self.snap)
        ok = torch.equal(b[:p], s[:p]) and torch.equal(b[-p:], s[-p:])
        if written is not None:
            inner, old = _bits(self.t), _bits(self.snap[p:p + self.t.numel()].view(self.t.shape))
            ok = ok and torch.equal(inner[~written], old[~written])
        return ok


# ----------------------------------------------------------------------------------------------------- measures
def errors(out, ref, kind, scale=None):
    """-> (max error, fraction of elements above one bf16 ulp, relative norm error); see the module docstring."""
    d = (out.to(f64) - ref).abs()
    rms = ref.pow(2).mean().sqrt().item()
    ulp = torch.exp2(torch.floor(torch.log2(torch.clamp(ref.abs(), min=rms / 64 + 1e-300))) - 7)
    if kind == "ulp":
        mx = (d / ulp).max().item()
    elif kind == "rms":
        mx = d.max().item() / rms if rms > 0 else (0.0 if d.max().item() == 0 else math.inf)
    else:
        mx = (d / scale).max().item()
    rn = ref.norm().item()
    rel = d.norm().item() / rn if rn > 0 else (0.0 if d.max().item() == 0 else math.inf)
    return mx, (d > ulp).double().mean().item(), rel


def rejecting(errs, name):
    """The measures of `errs` outside BOUNDS[name]."""
    return [m for m, v, lim in zip(("max", "share", "rel"), errs, BOUNDS[name]) if not v <= lim]


def judge(label, outs, refs, mutants, scales=None):
    """Print the measures of each output and which bound rejects each mutant; assert the outputs are within bounds and
    every mutant that changes an output by more than one ulp somewhere is rejected.  outs/refs: {bound name: tensor};
    mutants: {mutant: {bound name: mutated reference} or None}.  -> the names of the mutants that changed something."""
    scales = scales or {}
    print(f"\n{label}")
    bad = []
    for n in outs:
        assert torch.isfinite(outs[n].to(f64)).all(), n
        e = errors(outs[n], refs[n], KIND[n], scales.get(n))
        print(f"  {n:16s} max {e[0]:10.4g} {KIND[n]:3s}  >1ulp {e[1]:9.3g}  rel {e[2]:9.3g}")
        if rejecting(e, n):
            bad.append((n, e, BOUNDS[n]))
    assert not bad, bad
    shown = []
    for mname, m in mutants.items():
        changed = {n: mm for n, mm in (m or {}).items() if errors(mm, refs[n], "ulp")[1] > 0}
        if not changed:
            print(f"  mutant {mname}: changes nothing here")
            continue
        caught = {n: rejecting(errors(outs[n], mm, KIND[n], scales.get(n)), n) for n, mm in changed.items()}
        caught = {n: r for n, r in caught.items() if r}
        print(f"  mutant {mname}: rejected by {caught}")
        assert caught, mname
        shown.append(mname)
    return shown


# ----------------------------------------------------------------------------------------------------- attention
# (B, T, H, score rows)
ATTN_CASES = [
    (1, 1, 1, "random"), (3, 2, 2, "random"), (1, 16, 1, "peaky"), (3, 17, 3, "random"), (1, 32, 8, "uniform"),
    (3, 33, 1, "tied"), (1, 63, 2, "large"), (64, 64, 1, "random"), (3, 65, 3, "peaky"), (1, 127, 8, "random"),
    (3, 128, 2, "uniform"), (1, 129, 1, "large"), (64, 150, 8, "random"), (3, 191, 3, "tied"), (1, 192, 1, "peaky"),
    (3, 192, 8, "large"), (64, 192, 2, "uniform"), (3, 129, 2, "tied"),
]
ATTN_MUTANTS = ("drop_last_key", "last_tile_from_wrong_tile", "lse_natural_log", "D_zero")


def attention_inputs(B, T, H, kind, seed):
    E = 128 * H
    g = _gen(seed)
    q, kv, dout = _randn(g, B, T, E), _randn(g, B, T, 2 * E), _randn(g, B, T, E)
    if kind == "peaky":
        q *= 8
    elif kind == "uniform":
        q *= 0.01
    elif kind == "tied":                                     # keys repeated in groups of 4: tied scores in every row
        kv[:, :, :E] = kv[:, (torch.arange(T, device="cuda") // 4) * 4, :E]
    elif kind == "large":                                    # |s| ~ 64 sigma: exp without the max subtraction overflows
        q *= 8
        kv[:, :, :E] *= 8
    return q.to(bf16), kv.to(bf16), dout.to(bf16)


def _last_tile_wrong(x, T, rows_dim):
    """Rows [128, T) of the last 128-row tile replaced by rows [0, T - 128)."""
    y = x.clone()
    idx = torch.arange(128, T, device=x.device)
    y.index_copy_(rows_dim, idx, x.index_select(rows_dim, idx - 128))
    return y


@gpu
@pytest.mark.parametrize("case", ATTN_CASES, ids=[f"B{c[0]}-T{c[1]}-H{c[2]}-{c[3]}" for c in ATTN_CASES])
def test_attention_matches_oracle(case):
    B, T, H, kind = case
    E = 128 * H
    L, st = _L(), _st()
    q, kv, dout = attention_inputs(B, T, H, kind, seed=ATTN_CASES.index(case))
    o, lse2 = Guarded((B, T, E), bf16, float("nan")).seal(), Guarded((B * H, T), f32, float("nan")).seal()
    assert L.avctc_attention_forward(q.data_ptr(), kv.data_ptr(), o.t.data_ptr(), lse2.t.data_ptr(), B, T, H, E,
                                     st) == OK
    dq, dkv = Guarded((B, T, E), bf16, float("nan")).seal(), Guarded((B, T, 2 * E), bf16, float("nan")).seal()
    assert L.avctc_attention_backward(q.data_ptr(), kv.data_ptr(), dout.data_ptr(), o.t.data_ptr(), lse2.t.data_ptr(),
                                      dq.t.data_ptr(), dkv.t.data_ptr(), B, T, H, E, st) == OK
    torch.cuda.synchronize()
    assert all(x.untouched() for x in (o, lse2, dq, dkv))
    ref_o, ref_l = fo.attention_forward(q, kv, H)
    ref_dq, ref_dk, ref_dv = fo.attention_backward(q, kv, dout, ref_o, ref_l, H)
    outs = {"attn.o": o.t, "attn.lse2": lse2.t, "attn.dq": dq.t, "attn.dk": dkv.t[..., :E], "attn.dv": dkv.t[..., E:]}
    refs = {"attn.o": ref_o, "attn.lse2": ref_l, "attn.dq": ref_dq, "attn.dk": ref_dk, "attn.dv": ref_dv}
    mut = dict.fromkeys(ATTN_MUTANTS)
    names = list(refs)
    if T > 1:
        km = torch.arange(T, device="cuda") < T - 1
        mo, ml = fo.attention_forward(q, kv, H, key_mask=km)
        mut["drop_last_key"] = dict(zip(names, (mo, ml) + fo.attention_backward(q, kv, dout, mo, ml, H, key_mask=km)))
    if T > 128:
        mut["last_tile_from_wrong_tile"] = {n: _last_tile_wrong(r, T, 1) for n, r in refs.items()}
    mut["lse_natural_log"] = {"attn.lse2": ref_l * fo.LN2}
    mut["D_zero"] = dict(zip(names[2:], fo.attention_backward(q, kv, dout, ref_o, ref_l, H, zero_D=True)))
    judge(f"attention B={B} T={T} H={H} {kind}", outs, refs, mut)


# ----------------------------------------------------------------------------------------------------- softmax
# (rows, T, Tp)
SOFTMAX_CASES = [(1, 1, 8), (9, 1, 25), (7, 31, 32), (9, 31, 55), (4800, 32, 32), (1, 32, 56), (7, 33, 40),
                 (4800, 33, 57), (9, 150, 152), (4800, 150, 174), (1, 193, 200), (7, 193, 217), (9, 257, 264),
                 (4800, 257, 281), (7, 1000, 1000), (4800, 1000, 1024)]


@gpu
@pytest.mark.parametrize("case", SOFTMAX_CASES, ids=[f"rows{c[0]}-T{c[1]}-Tp{c[2]}" for c in SOFTMAX_CASES])
def test_softmax_matches_oracle(case):
    rows, T, Tp = case
    L, st = _L(), _st()
    g = _gen(100 + SOFTMAX_CASES.index(case))
    S = _randn(g, rows, Tp) * 3
    S[1::3] *= 10          # peaky rows, among ordinary ones: a one-hot row's dS cancels to fp32 rounding of its sum
    S[:, T:] = float("nan")                                   # pad columns are never read
    dP = _randn(g, rows, Tp)
    dP[:, T:] = float("nan")
    P = Guarded((rows, Tp), bf16, float("nan")).seal()
    assert L.avctc_softmax_forward(S.data_ptr(), P.t.data_ptr(), rows, T, Tp, st) == OK
    dS = Guarded((rows, Tp), bf16, float("nan")).seal()
    assert L.avctc_softmax_backward(P.t.data_ptr(), dP.data_ptr(), dS.t.data_ptr(), rows, T, Tp, st) == OK
    torch.cuda.synchronize()
    assert P.untouched() and dS.untouched()
    assert (P.t[:, T:] == 0).all() and (dS.t[:, T:] == 0).all()    # the following P.V / dS.K GEMMs read them
    refs = {"softmax.P": fo.softmax_forward(S, T), "softmax.dS": fo.softmax_backward(P.t, dP, T)}
    mut = {"pad_column_nonzero": None}
    if Tp > T:
        m = {}
        for n, r in refs.items():
            m[n] = r.clone()
            m[n][:, T] = r[:, T - 1]
        mut["pad_column_nonzero"] = m
    judge(f"softmax rows={rows} T={T} Tp={Tp}", {"softmax.P": P.t, "softmax.dS": dS.t}, refs, mut)


# ----------------------------------------------------------------------------------------------------- resample
# (audio dtype, D, B, Ta, Tv rule, mask pattern).  Tv rule: "lt" 2 Tp / 3, "eq" Tp, "2x" 2 Tp, "one" 1, "seven" 7.
RESAMPLE_CASES = [
    (F32, 8, 1, 9, "eq", "mixed"), (BF16, 12, 5, 249, "lt", "one_empty"), (F32, 1024, 5, 600, "lt", "mixed"),
    (BF16, 1024, 1, 249, "2x", "mixed"), (F32, 12, 40, 600, "2x", "one_empty"), (BF16, 8, 40, 249, "one", "mixed"),
    (F32, 8, 5, 9, "seven", "single"), (BF16, 12, 5, 249, "seven", "all_empty"), (BF16, 1024, 40, 600, "eq", "one_empty"),
    (F32, 8, 40, 249, "lt", "mixed"), (BF16, 8, 5, 9, "lt", "mixed"), (F32, 12, 1, 600, "one", "mixed"),
]
RESAMPLE_MUTANTS = ("i1_off_by_one", "w0_w1_swapped", "source_from_unpadded_sample")


def resample_mask(B, Ta, pattern, seed):
    g = torch.Generator().manual_seed(seed)
    m = torch.randint(0, 4, (B, Ta), generator=g)
    m[torch.rand(B, Ta, generator=g) < 0.4] = 1
    if pattern == "one_empty":
        m[B // 2] = torch.randint(0, 2, (Ta,), generator=g) * 3
    elif pattern == "all_empty":
        m = torch.randint(0, 2, (B, Ta), generator=g) * 3
    elif pattern == "single":                                # at most one speech frame per sample: Tp = 1
        m = torch.zeros(B, Ta, dtype=torch.int64)
        for b in range(B - 1):
            m[b, (3 * b + 2) % Ta] = 1 + b % 2
    return m


def resample_tv(Tp, rule):
    return dict(lt=max(1, 2 * Tp // 3), eq=Tp, one=1, seven=7).get(rule, 2 * Tp)


def _resample_mutant(audio, mask, dout, Tv, which):
    src, cnt = fo.speech_index(mask)
    Tp = int(cnt.max())
    if Tp == 0:
        return None
    i0, i1, w0, w1 = fo.lerp_coef(Tp, Tv, audio.device, f32)
    if which == "i1_off_by_one":
        W = fo.lerp_matrix(Tp, Tv, coef=(i0, torch.where(w1 != 0, torch.clamp(i1 + 1, max=Tp - 1), i1), w0, w1))
    elif which == "w0_w1_swapped":
        W = fo.lerp_matrix(Tp, Tv, coef=(i0, i1, w1, w0))
    else:                                                    # frame r of the padded sample read from raw frame r
        W = fo.lerp_matrix(Tp, Tv, audio.device, dtype=f32)
        keep = (torch.arange(Tp, device=audio.device)[None, :] < cnt[:, None]).to(f64)
        out = W @ (audio[:, :Tp].to(f64) * keep[:, :, None])
        da = torch.zeros(audio.shape, dtype=f64, device=audio.device)
        da[:, :Tp] = (W.T @ dout.to(f64)) * keep[:, :, None]
        return out, da
    return fo.resample_forward(audio, mask, Tv, W=W)[0], fo.resample_backward(dout, mask, W=W)


@gpu
@pytest.mark.parametrize("case", RESAMPLE_CASES, ids=[f"{'bf16' if c[0] else 'f32'}-D{c[1]}-B{c[2]}-Ta{c[3]}-{c[4]}-{c[5]}"
                                                      for c in RESAMPLE_CASES])
def test_resample_matches_oracle(case):
    dt, D, B, Ta, rule, pattern = case
    L, st = _L(), _st()
    i = RESAMPLE_CASES.index(case)
    mask = resample_mask(B, Ta, pattern, seed=200 + i).cuda()
    Tp = int(fo.speech_index(mask)[1].max())
    Tv = resample_tv(Tp, rule) if pattern != "all_empty" else 7
    g = _gen(200 + i)
    audio = _randn(g, B, Ta, D, dtype=_DT[dt])
    out, mo, il = (Guarded((B, Tv, D), bf16, float("nan")).seal(), Guarded((B, Tv), i64, -7).seal(),
                   Guarded((B,), i64, -7).seal())
    ws = torch.empty(L.avctc_resample_workspace_bytes(B, Ta), dtype=torch.uint8, device="cuda")
    assert L.avctc_resample_forward(audio.data_ptr(), dt, mask.data_ptr(), B, Ta, D, Tv, out.t.data_ptr(),
                                    mo.t.data_ptr(), il.t.data_ptr(), ws.data_ptr(), ws.numel(), st) == OK
    dout = _randn(g, B, Tv, D, dtype=bf16)
    da = Guarded((B, Ta, D), _DT[dt], float("nan")).seal()
    assert L.avctc_resample_backward(dout.data_ptr(), B, Ta, D, Tv, ws.data_ptr(), da.t.data_ptr(), dt, st) == OK
    torch.cuda.synchronize()
    assert all(x.untouched() for x in (out, mo, il, da))
    ref_out, ref_mo, ref_il = fo.resample_forward(audio, mask, Tv, coef_dtype=f32)   # ATen's weights for float32 / bf16
    ref_da = fo.resample_backward(dout, mask, coef_dtype=f32)
    assert torch.equal(mo.t, ref_mo) and torch.equal(il.t, ref_il)
    speech = (mask != 0) & (mask != 3)
    assert (da.t[~speech] == 0).all()                        # frames that are not speech get exact zeros
    da_name = "resample.da_bf16" if dt == BF16 else "resample.da_f32"
    outs, refs = {"resample.out": out.t, da_name: da.t}, {"resample.out": ref_out, da_name: ref_da}
    mut = {}
    for m in RESAMPLE_MUTANTS:
        r = _resample_mutant(audio, mask, dout, Tv, m)
        mut[m] = None if r is None else {"resample.out": r[0], da_name: r[1]}
    judge(f"resample {'bf16' if dt else 'f32'} D={D} B={B} Ta={Ta} Tp={Tp} Tv={Tv} {pattern}", outs, refs, mut)


# ----------------------------------------------------------------------------------------------------- colsum
K_COLSUM_ROWS, K_COLSUM_CHUNKS = 128, 64                      # fusion_kernels.cu: rows per chunk, chunk cap
# (M, N, ld - N, dtype, accumulate)
COLSUM_CASES = [(1, 1, 0, F32, 0), (7, 33, 8, BF16, 1), (128, 800, 0, F32, 1), (129, 2048, 8, BF16, 0),
                (8193, 33, 0, BF16, 0), (8193, 800, 8, F32, 1), (100000, 33, 8, F32, 0), (100000, 800, 0, BF16, 1),
                (129, 1, 8, F32, 0), (7, 2048, 0, F32, 0), (100000, 2048, 8, BF16, 0), (1, 800, 8, BF16, 1),
                (128, 33, 0, BF16, 0), (8193, 2048, 0, F32, 0)]


def colsum_last_chunk(M):
    chunks = min(_cdiv(M, K_COLSUM_ROWS), K_COLSUM_CHUNKS)
    return (chunks - 1) * _cdiv(M, chunks)


@gpu
@pytest.mark.parametrize("case", COLSUM_CASES, ids=[f"M{c[0]}-N{c[1]}-ld+{c[2]}-{'bf16' if c[3] else 'f32'}-acc{c[4]}"
                                                    for c in COLSUM_CASES])
def test_colsum_matches_oracle(case):
    M, N, extra, dt, acc = case
    L, st = _L(), _st()
    g = _gen(300 + COLSUM_CASES.index(case))
    X = (_randn(g, M, N + extra) + 0.25).to(_DT[dt])
    X[:, N:] = float("nan")                                   # columns past N are never read
    out = Guarded((N,), f32, float("nan"))
    out0 = _randn(g, N) * 10 if acc else None
    if acc:
        out.t.copy_(out0)
    out.seal()
    assert L.avctc_colsum(X.data_ptr(), dt, M, N, N + extra, out.t.data_ptr(), acc, st) == OK
    torch.cuda.synchronize()
    assert out.untouched()
    ref = fo.colsum(X, N) + (out0.to(f64) if acc else 0)
    scale = X[:, :N].to(f64).abs().sum(0) + (out0.to(f64).abs() if acc else 0)
    r0 = colsum_last_chunk(M)
    mut = {"missing_last_row_chunk": {"colsum.out": ref - fo.colsum(X[r0:], N)}}
    judge(f"colsum M={M} N={N} ld={N + extra} {'bf16' if dt else 'f32'} accumulate={acc}", {"colsum.out": out.t},
          {"colsum.out": ref}, mut, scales={"colsum.out": scale})


# ----------------------------------------------------------------------------------------------------- log_softmax
# (rows, V, in dtype, out dtype); the backward runs with Y and dY in the input dtype
LOGSM_CASES = [(5, 1, F32, F32), (37, 2, BF16, F32), (64, 33, F32, BF16), (300, 801, BF16, BF16), (64, 1024, F32, F32),
               (33, 1025, BF16, F32), (20, 5000, F32, BF16), (150, 801, F32, F32), (40, 5000, BF16, BF16),
               (9, 1024, BF16, BF16), (10, 1025, F32, BF16), (7, 2, F32, BF16), (11, 33, BF16, BF16)]


@gpu
@pytest.mark.parametrize("case", LOGSM_CASES, ids=[f"rows{c[0]}-V{c[1]}-{'bf16' if c[2] else 'f32'}-{'bf16' if c[3] else 'f32'}"
                                                   for c in LOGSM_CASES])
def test_log_softmax_matches_oracle(case):
    rows, V, din, dout_ = case
    L, st = _L(), _st()
    g = _gen(400 + LOGSM_CASES.index(case))
    X = _randn(g, rows, V) * 4
    X[1::5] = 3.0                                             # equal logits
    X[2::5] = 5000.0 + 20 * X[2::5]                           # large logits
    X = X.to(_DT[din])
    Y = Guarded((rows, V), _DT[dout_], float("nan")).seal()
    assert L.avctc_log_softmax_forward(X.data_ptr(), din, Y.t.data_ptr(), dout_, rows, V, st) == OK
    ldx = _cdiv(V, 8) * 8
    Yin = fo.log_softmax_forward(X).to(_DT[din])              # the backward's inputs, in its dtype
    dY = _randn(g, rows, V, dtype=_DT[din])
    dX = Guarded((rows, ldx), bf16, float("nan")).seal()
    assert L.avctc_log_softmax_backward(Yin.data_ptr(), dY.data_ptr(), din, dX.t.data_ptr(), rows, V, ldx, st) == OK
    torch.cuda.synchronize()
    cols = torch.zeros(rows, ldx, dtype=torch.bool, device="cuda")
    cols[:, :V] = True
    assert Y.untouched() and dX.untouched(cols)               # dX's pad columns keep their NaN bits
    y_name = "logsm.y_bf16" if dout_ == BF16 else "logsm.y_f32"
    refs = {y_name: fo.log_softmax_forward(X), "logsm.dx": fo.log_softmax_backward(Yin, dY)}
    mut = {"dx_without_expY_sum_term": {"logsm.dx": dY.to(f64)}}
    judge(f"log_softmax rows={rows} V={V} in={'bf16' if din else 'f32'} out={'bf16' if dout_ else 'f32'}",
          {y_name: Y.t, "logsm.dx": dX.t[:, :V]}, refs, mut)


# ----------------------------------------------------------------------------------------------------- gemm
# (M, N, K, out dtype, bias_mode, alpha, accumulate, C layout, batch, inner_count).  C layout: "" ldc = round_up(N, 8)
# + 8, "vec" ldc = N (the 16-byte epilogue when N is a multiple of 128), "ldc" odd ldc, "off" C one element off.
GEMM_CASES = [
    (1, 1, 1, F32, 0, 1.0, 0, "", 1, 1), (8, 63, 65, BF16, 1, 0.37, 0, "", 1, 1), (63, 65, 129, F32, 2, -1.5, 1, "", 1, 1),
    (65, 129, 8, F32, 1, 0.37, 1, "ldc", 1, 1), (129, 8, 63, BF16, 2, 2.0, 0, "", 1, 1),
    (129, 129, 129, F32, 1, 0.37, 0, "off", 1, 1), (128, 128, 129, BF16, 2, 0.37, 0, "ldc", 1, 1),
    (128, 256, 64, F32, 1, 0.37, 1, "off", 1, 1), (128, 256, 192, F32, 2, 0.37, 1, "vec", 1, 1),
    (256, 128, 65, BF16, 1, 0.37, 0, "vec", 1, 1), (65, 63, 129, F32, 2, 0.5, 0, "", 6, 3),
    (129, 128, 65, BF16, 1, 1.25, 0, "vec", 4, 2), (1, 129, 63, F32, 2, 0.37, 1, "", 2, 2),
    (63, 1, 8, F32, 1, -0.75, 0, "", 1, 1), (8, 8, 1, BF16, 2, 0.37, 0, "off", 1, 1),
]
GEMM_MUTANTS = ("bias_row_column_swapped", "missing_last_k_block", "accumulate_ignored")


def _operand(t, rows, K):
    """avctc_gemm_operand of a K-major [Z, rows, ld] bf16 tensor whose first K columns are the operand; batch entry z
    reads slice z (z_outer = inner_count and z_inner = 1 are set by the caller)."""
    op = _lib().GemmOperand()
    op.ptr, op.rows, op.kdim, op.zdim = t.data_ptr(), rows, K, t.shape[0]
    op.ld, op.zstride = t.shape[2], (t.shape[1] * t.shape[2] if t.shape[0] > 1 else 0)
    op.k_outer = op.k_inner = op.r_outer = op.r_inner = 0
    op.z_outer, op.z_inner, op.mn_major = 1, 0, 0
    return op


@gpu
@pytest.mark.parametrize("case", GEMM_CASES, ids=[f"M{c[0]}-N{c[1]}-K{c[2]}-{'bf16' if c[3] else 'f32'}-bias{c[4]}-acc{c[6]}"
                                                  f"-{c[7] or 'pad'}-z{c[8]}x{c[9]}" for c in GEMM_CASES])
def test_gemm_matches_oracle(case):
    M, N, K, dt, bmode, alpha, acc, lay, Z, inner = case
    L, st = _L(), _st()
    g = _gen(500 + GEMM_CASES.index(case))
    ldk = _cdiv(K, 8) * 8
    A, Bm = _randn(g, Z, M, ldk).to(bf16), _randn(g, Z, N, ldk).to(bf16)
    A[..., K:] = float("nan")                                 # columns past K are outside the operand
    Bm[..., K:] = float("nan")
    bias = _randn(g, max(M, N))
    ldc = {"vec": N, "ldc": N + 1}.get(lay, _cdiv(N, 8) * 8 + 8)
    off = 1 if lay == "off" else 0
    C = Guarded((Z * M * ldc + off,), _DT[dt], float("nan"))
    view = C.t[off:].view(Z, M, ldc)
    C0 = (_randn(g, Z, M, N) * 3) if acc else None
    if acc:
        view[..., :N] = C0
    C.seal()
    opa, opb = _operand(A, M, K), _operand(Bm, N, K)
    opa.z_outer = opb.z_outer = inner
    opa.z_inner = opb.z_inner = 1
    rc = L.avctc_gemm_bf16(ctypes.byref(opa), ctypes.byref(opb), M, N, K, Z, inner, view.data_ptr(), dt, ldc,
                           inner * M * ldc, M * ldc, bias.data_ptr() if bmode else None, bmode, alpha, acc, st)
    assert rc == OK
    torch.cuda.synchronize()
    written = torch.zeros(C.t.shape, dtype=torch.bool, device="cuda")
    written[off:].view(Z, M, ldc)[..., :N] = True
    assert C.untouched(written)                               # ldc pad columns, guard rows, the offset element
    Ak, Bk = A[..., :K], Bm[..., :K]
    ref = fo.gemm(Ak, Bk, alpha, bias, bmode, C0)
    name = "gemm.c_bf16" if dt == BF16 else "gemm.c_f32"
    kl = (_cdiv(K, 64) - 1) * 64
    mut = {"bias_row_column_swapped": {name: fo.gemm(Ak, Bk, alpha, bias, 3 - bmode, C0)} if bmode else None,
           "missing_last_k_block": {name: ref - fo.gemm(Ak[..., kl:], Bk[..., kl:], alpha)},
           "accumulate_ignored": {name: ref - C0.to(f64)} if acc else None}
    judge(f"gemm M={M} N={N} K={K} {'bf16' if dt else 'f32'} bias_mode={bmode} alpha={alpha} accumulate={acc} "
          f"ldc={ldc} C+{off} batch={Z}/{inner}", {name: view[..., :N]}, {name: ref}, mut)


# ----------------------------------------------------------------------------------------------------- coverage
def test_cases_reach_every_edge_and_every_mutant():
    """Host-side: the case lists cover the shapes the kernels branch on, and every mutant has a case where it
    changes something (the GPU tests then require it to be rejected there)."""
    T = {c[1] for c in ATTN_CASES}
    assert T >= {1, 2, 16, 17, 32, 33, 63, 64, 65, 127, 128, 129, 150, 191, 192}
    assert {c[2] for c in ATTN_CASES} == {1, 2, 3, 8} and {c[0] for c in ATTN_CASES} == {1, 3, 64}
    assert {c[3] for c in ATTN_CASES} == {"random", "peaky", "uniform", "tied", "large"}
    assert any(t > 128 for t in T) and any(t > 1 for t in T)                 # wrong tile, dropped key
    assert {c[0] for c in SOFTMAX_CASES} == {1, 7, 9, 4800}
    assert {c[1] for c in SOFTMAX_CASES} == {1, 31, 32, 33, 150, 193, 257, 1000}
    for t in {c[1] for c in SOFTMAX_CASES}:
        assert {c[2] for c in SOFTMAX_CASES if c[1] == t} == {_cdiv(t, 8) * 8, t + 24}
    assert {c[0] for c in RESAMPLE_CASES} == {F32, BF16} and {c[1] for c in RESAMPLE_CASES} == {8, 12, 1024}
    assert {c[2] for c in RESAMPLE_CASES} == {1, 5, 40} and {c[3] for c in RESAMPLE_CASES} == {9, 249, 600}
    assert {c[5] for c in RESAMPLE_CASES} >= {"one_empty", "all_empty", "single"}
    seen, shows = set(), set()
    for i, c in enumerate(RESAMPLE_CASES):
        m = resample_mask(c[2], c[3], c[5], seed=200 + i)
        cnt = fo.speech_index(m)[1]
        Tp = int(cnt.max())
        assert (Tp == 1) == (c[5] == "single") and (Tp == 0) == (c[5] == "all_empty")
        assert (c[5] != "one_empty") or (cnt == 0).sum() == 1
        if not Tp:
            continue
        Tv = resample_tv(Tp, c[4])
        seen |= {n for n, hit in (("Tv<Tp", Tv < Tp), ("Tv=Tp", Tv == Tp), ("Tv=2Tp", Tv == 2 * Tp), ("Tv=1", Tv == 1))
                 if hit}
        a, d = torch.randn(c[2], c[3], 1, dtype=f64), torch.randn(c[2], Tv, 1, dtype=f64)
        ref = fo.resample_forward(a, m, Tv)[0], fo.resample_backward(d, m)
        for n in RESAMPLE_MUTANTS:
            r = _resample_mutant(a, m, d, Tv, n)
            if any((x - y).abs().max() > 1e-9 for x, y in zip(r, ref)):
                shows.add(n)
    assert seen == {"Tv<Tp", "Tv=Tp", "Tv=2Tp", "Tv=1"}
    assert shows == set(RESAMPLE_MUTANTS)
    assert {c[0] for c in COLSUM_CASES} == {1, 7, 128, 129, 8193, 100000}
    assert {c[1] for c in COLSUM_CASES} == {1, 33, 800, 2048} and {c[2] for c in COLSUM_CASES} == {0, 8}
    assert {(c[3], c[4]) for c in COLSUM_CASES} == {(F32, 0), (F32, 1), (BF16, 0), (BF16, 1)}
    assert any(_cdiv(c[0], K_COLSUM_ROWS) > K_COLSUM_CHUNKS for c in COLSUM_CASES)
    assert all(colsum_last_chunk(c[0]) < c[0] for c in COLSUM_CASES)      # the last chunk is never empty
    assert {c[1] for c in LOGSM_CASES} == {1, 2, 33, 801, 1024, 1025, 5000}
    assert {(c[2], c[3]) for c in LOGSM_CASES} == {(a, b) for a in (F32, BF16) for b in (F32, BF16)}
    assert any(c[1] % 8 for c in LOGSM_CASES)                              # ldx > V
    for d in range(3):
        assert {c[d] for c in GEMM_CASES} >= {1, 8, 63, 65, 129}
    assert {c[4] for c in GEMM_CASES} == {0, 1, 2} and {c[7] for c in GEMM_CASES} >= {"vec", "ldc", "off"}
    assert any(c[6] and c[3] == F32 for c in GEMM_CASES) and any(c[9] > 1 for c in GEMM_CASES)
    assert any(c[7] in ("ldc", "off") and c[1] % 128 == 0 for c in GEMM_CASES)   # epilogue forced on a full tile


# ----------------------------------------------------------------------------------------------------- error contract
def _rejects(rc_want, bufs, fn, *args, **kw):
    """Call fn(*args, **kw), expect rc_want, and every buffer in `bufs` bit-identical afterwards."""
    snaps = [_bits(b).clone() for b in bufs]
    rc = fn(*args, **kw)
    torch.cuda.synchronize()
    assert rc == rc_want, (fn, rc, rc_want)
    for b, s in zip(bufs, snaps):
        assert torch.equal(_bits(b), s), fn


def _sentinel(*shape, dtype=f32):
    return torch.full(shape, -7 if dtype == i64 else float("nan"), dtype=dtype, device="cuda")


@gpu
def test_resample_error_contract():
    L, st = _L(), _st()
    B, Ta, D, Tv = 2, 16, 8, 10
    audio = torch.randn(B, Ta, D, device="cuda")
    mask = torch.ones(B, Ta, dtype=i64, device="cuda")
    out, mo, il, da = _sentinel(B, Tv, D, dtype=bf16), _sentinel(B, Tv, dtype=i64), _sentinel(B, dtype=i64), \
        _sentinel(B, Ta, D)
    nws = L.avctc_resample_workspace_bytes(B, Ta)
    ws = torch.full((nws,), 0x5A, dtype=torch.uint8, device="cuda")
    dout = torch.randn(B, Tv, D, device="cuda").to(bf16)
    bufs = (out, mo, il, ws)
    a = [audio.data_ptr(), F32, mask.data_ptr(), B, Ta, D, Tv, out.data_ptr(), mo.data_ptr(), il.data_ptr(),
         ws.data_ptr(), nws, st]
    fwd = L.avctc_resample_forward
    for i in (0, 2, 7, 8, 9, 10):
        _rejects(BAD_ARG, bufs, fwd, *a[:i], None, *a[i + 1:])
    for i in (3, 4, 5, 6):
        _rejects(BAD_ARG, bufs, fwd, *a[:i], 0, *a[i + 1:])
    for dt in (2, -1):                                       # fails at the parent: input_lengths zeroed first
        _rejects(BAD_ARG, bufs, fwd, *a[:1], dt, *a[2:])
    _rejects(WORKSPACE, bufs, fwd, *a[:11], nws - 1, a[12])
    _rejects(ALIGNMENT, bufs, fwd, audio.data_ptr() + 4, *a[1:])
    _rejects(ALIGNMENT, bufs, fwd, *a[:7], out.data_ptr() + 2, *a[8:])
    assert fwd(*a) == OK
    torch.cuda.synchronize()
    b = [dout.data_ptr(), B, Ta, D, Tv, ws.data_ptr(), da.data_ptr(), F32, st]
    bwd = L.avctc_resample_backward
    for i in (0, 5, 6):
        _rejects(BAD_ARG, (da,), bwd, *b[:i], None, *b[i + 1:])
    _rejects(BAD_ARG, (da,), bwd, *b[:7], 2, st)
    _rejects(ALIGNMENT, (da,), bwd, dout.data_ptr() + 2, *b[1:])
    _rejects(ALIGNMENT, (da,), bwd, *b[:6], da.data_ptr() + 4, *b[7:])
    assert bwd(*b) == OK


@gpu
def test_softmax_colsum_log_softmax_error_contract():
    L, st = _L(), _st()
    rows, T, Tp = 9, 30, 32
    S, dP = torch.randn(rows, Tp, device="cuda"), torch.randn(rows, Tp, device="cuda")
    P, dS = _sentinel(rows, Tp, dtype=bf16), _sentinel(rows, Tp, dtype=bf16)
    for args in ((None, P.data_ptr(), rows, T, Tp, st), (S.data_ptr(), None, rows, T, Tp, st),
                 (S.data_ptr(), P.data_ptr(), 0, T, Tp, st), (S.data_ptr(), P.data_ptr(), rows, 0, Tp, st),
                 (S.data_ptr(), P.data_ptr(), rows, T, T - 1, st)):
        _rejects(BAD_ARG, (P,), L.avctc_softmax_forward, *args)
    for i in (0, 1, 2):
        a = [P.data_ptr(), dP.data_ptr(), dS.data_ptr(), rows, T, Tp, st]
        a[i] = None
        _rejects(BAD_ARG, (dS,), L.avctc_softmax_backward, *a)
    _rejects(BAD_ARG, (dS,), L.avctc_softmax_backward, P.data_ptr(), dP.data_ptr(), dS.data_ptr(), rows, T, T - 1, st)

    M, N = 300, 40
    X, out = torch.randn(M, N + 8, device="cuda"), _sentinel(N)
    a = [X.data_ptr(), F32, M, N, N + 8, out.data_ptr(), 0, st]
    for i, v in ((0, None), (5, None), (2, 0), (3, 0), (1, 2), (1, -1), (4, N - 1)):   # dtype and ld < N fail at the parent
        _rejects(BAD_ARG, (out,), L.avctc_colsum, *a[:i], v, *a[i + 1:])
    assert L.avctc_colsum(*a) == OK

    V = 30
    x, y, dx = torch.randn(rows, V, device="cuda"), _sentinel(rows, V), _sentinel(rows, 32, dtype=bf16)
    for args in ((None, F32, y.data_ptr(), F32, rows, V, st), (x.data_ptr(), F32, None, F32, rows, V, st),
                 (x.data_ptr(), 2, y.data_ptr(), F32, rows, V, st), (x.data_ptr(), F32, y.data_ptr(), 2, rows, V, st),
                 (x.data_ptr(), F32, y.data_ptr(), F32, 0, V, st), (x.data_ptr(), F32, y.data_ptr(), F32, rows, 0, st)):
        _rejects(BAD_ARG, (y,), L.avctc_log_softmax_forward, *args)
    b = [x.data_ptr(), x.data_ptr(), F32, dx.data_ptr(), rows, V, 32, st]
    for i, v in ((0, None), (1, None), (3, None), (2, 2), (6, V - 1), (4, 0)):
        _rejects(BAD_ARG, (dx,), L.avctc_log_softmax_backward, *b[:i], v, *b[i + 1:])


@gpu
def test_attention_error_contract():
    L, st = _L(), _st()
    B, T, H = 2, 40, 2
    E = 128 * H
    q, kv, dout = (torch.randn(B, T, n, device="cuda").to(bf16) for n in (E, 2 * E, E))
    o, lse2 = _sentinel(B, T, E, dtype=bf16), _sentinel(B * H, T)
    dq, dkv = _sentinel(B, T, E, dtype=bf16), _sentinel(B, T, 2 * E, dtype=bf16)
    f = [q.data_ptr(), kv.data_ptr(), o.data_ptr(), lse2.data_ptr(), B, T, H, E, st]
    fwd, bwd = L.avctc_attention_forward, L.avctc_attention_backward
    for over in ({5: 193}, {5: 0}, {6: 4}, {7: 384}, {6: 0, 7: 0}, {4: 0}):       # T > 192, E != 128 H, empty
        _rejects(UNSUPPORTED, (o, lse2), fwd, *[over.get(i, v) for i, v in enumerate(f)])
    for i in range(4):
        _rejects(BAD_ARG, (o, lse2), fwd, *f[:i], None, *f[i + 1:])
    _rejects(ALIGNMENT, (o, lse2), fwd, q.data_ptr() + 2, *f[1:])
    _rejects(ALIGNMENT, (o, lse2), fwd, q.data_ptr(), kv.data_ptr() + 2, *f[2:])
    assert fwd(*f) == OK
    torch.cuda.synchronize()
    b = [q.data_ptr(), kv.data_ptr(), dout.data_ptr(), o.data_ptr(), lse2.data_ptr(), dq.data_ptr(), dkv.data_ptr(),
         B, T, H, E, st]
    for over in ({8: 193}, {10: 384}):
        _rejects(UNSUPPORTED, (dq, dkv), bwd, *[over.get(i, v) for i, v in enumerate(b)])
    for i in range(7):
        _rejects(BAD_ARG, (dq, dkv), bwd, *b[:i], None, *b[i + 1:])
    _rejects(ALIGNMENT, (dq, dkv), bwd, *b[:2], dout.data_ptr() + 2, *b[3:])
    assert bwd(*b) == OK


@gpu
def test_gemm_error_contract():
    L, st = _L(), _st()
    M, N, K = 70, 40, 48
    A, Bm = torch.randn(1, M, K, device="cuda").to(bf16), torch.randn(1, N, K, device="cuda").to(bf16)
    C, Cb, bias = _sentinel(M, N), _sentinel(M, N, dtype=bf16), torch.randn(max(M, N), device="cuda")
    opa, opb = _operand(A, M, K), _operand(Bm, N, K)

    def call(a=opa, b=opb, M=M, N=N, K=K, batch=1, inner=1, c=C, dt=F32, ldc=N, bias_p=None, bmode=0, acc=0):
        return L.avctc_gemm_bf16(ctypes.byref(a) if a is not None else None, ctypes.byref(b) if b is not None else None,
                                 M, N, K, batch, inner, c.data_ptr() if c is not None else None, dt, ldc, 0, 0, bias_p,
                                 bmode, 1.0, acc, st)

    bufs = (C, Cb)
    for kw in (dict(a=None), dict(b=None), dict(c=None), dict(M=0), dict(N=0), dict(K=0), dict(batch=0), dict(inner=0),
               dict(dt=2), dict(c=Cb, dt=BF16, acc=1), dict(bmode=1), dict(bmode=2), dict(bmode=3, bias_p=bias.data_ptr()),
               dict(bmode=-1, bias_p=bias.data_ptr())):
        _rejects(BAD_ARG, bufs, call, **kw)
    bad = _operand(A, M, K)
    bad.ptr = None
    _rejects(BAD_ARG, bufs, call, a=bad)
    bad = _operand(A, M, K)
    bad.ptr = A.data_ptr() + 2                               # operand pointer not 16-byte aligned
    _rejects(ALIGNMENT, bufs, call, a=bad)
    bad = _operand(Bm, N, K)
    bad.ld = K + 1                                           # ld not a multiple of 8 elements
    _rejects(ALIGNMENT, bufs, call, b=bad)
    bad = _operand(Bm, N, K)
    bad.zdim, bad.zstride = 2, N * K + 4                     # zstride not a multiple of 8 elements
    _rejects(ALIGNMENT, bufs, call, b=bad)
    assert call(bias_p=bias.data_ptr(), bmode=2) == OK
