"""GPU: the four entry points of csrc/wav2vec2_layer.cu through the C ABI against oracle/w2v_oracle.py (float64, bf16
rounding at the module path's points) fed the same bf16 inputs and bf16-rounded weights.

The cases cover every LayerNorm width the kernels are built for (E = 256, 512, 768, 1024, i.e. NC = 1..4), intermediate
widths F = 4E, 4E + 8 and 1032 (the second FFN GEMM's K ragged against its 64-wide k-blocks), and the reduction edges:
M = 1 and 7 (fewer rows than a k-block and than the 32 row chunks of the bias sums), 129, 1200 (a short last split-K
share, and more rows than the 8 x 148 the LayerNorm-backward CTAs cover in one stride), 1992 and 12000.  Inputs include
zero rows (padded frames: variance 0) and rows with mean ~50 and std ~0.1.  Dropout runs at p = 0, p = 0.1, and at
three different p; masks come from ATen's native_dropout at the same (seed, offset).  Every case runs training = 0 or 1
and the backward both with and without the weight-gradient pointers.

Errors are measured per tensor against the oracle: for bf16 outputs the max error in bf16 ulps of the reference, for
fp32 gradients the max error over the tensor's RMS; for both the fraction of elements off by more than one bf16 ulp and
the relative norm error.  The ulp of a reference value is taken at max(|ref|, RMS/64), so that values that cancel to
near zero are not held to an ulp of their own tiny size.

The bounds (BOUNDS) are the worst value over the cases measured on one NVIDIA B200 (1000 W power limit) with at most
2x headroom; the measured worst values are listed next to each bound.  Every relative norm error measured is below
1.6e-3, the size of bf16 rounding flips: these cases found no fault in the kernels.  Six mutants of the oracle's
output, each a plausible kernel bug, must fall outside the bounds in every case where they change anything; that shows
the bounds are tight enough to see a missing split-K share, a missing row chunk of a bias sum, a missing
LayerNorm-backward CTA, a shifted or reused dropout mask and a dropped residual."""
import pytest
import torch

from oracle import w2v_oracle as wo

gpu = pytest.mark.gpu

bf16, f64 = torch.bfloat16, torch.float64
OK, BAD_ARG, UNSUPPORTED, WORKSPACE, ALIGNMENT = 0, -1, -2, -3, -4
EPS = 1e-5
K_COL_PARTS, K_LN_BWD_CTAS, K_ROWS_PER_CTA = 32, 148, 8      # wav2vec2_layer.cu

# (E, F, M, (p_hidden, p_act, p_out), training)
CASES = [
    (256, 1024, 1, (0.1, 0.1, 0.1), 1),
    (256, 1032, 1200, (0.1, 0.1, 0.1), 1),
    (256, 1024, 12000, (0.1, 0.1, 0.1), 1),
    (512, 2048, 129, (0.1, 0.1, 0.1), 1),
    (512, 2056, 1992, (0.05, 0.2, 0.15), 1),
    (512, 1032, 7, (0.0, 0.0, 0.0), 1),
    (768, 3072, 7, (0.1, 0.1, 0.1), 0),
    (768, 3080, 1200, (0.1, 0.1, 0.1), 1),
    (768, 1032, 1992, (0.0, 0.0, 0.0), 1),
    (1024, 4096, 1992, (0.1, 0.1, 0.1), 1),
    (1024, 4104, 129, (0.1, 0.1, 0.1), 0),
    (1024, 1032, 1200, (0.1, 0.1, 0.1), 1),
]

BF16_OUT = ("q", "k", "v", "dx_in", "y", "dattn", "dx_out")
# name: (max error, fraction above 1 ulp, relative norm error); max is in bf16 ulps for BF16_OUT, in RMS otherwise.
# Measured worst over CASES on one NVIDIA B200 at a 1000 W power limit in the comment.  The large max-ulp figures of
# y, dattn and dx_out are elements that cancel to a small value, where one ulp of a bf16 summand (a residual or an
# intermediate gradient rounded one way in the kernel and the other in the oracle) is many ulps of the result.  The bias
# gradients g_bqkv and g_b2 are fixed-order fp32 sums of the kernels' own bf16 inputs, so only fp32 rounding separates
# them from the oracle.
BOUNDS = {
    "q": (40, 0.0006, 0.0004),        # worst 21.7, 0.000372, 0.000241
    "k": (30, 0.0004, 0.00025),       # worst 16, 0.000201, 0.000147
    "v": (40, 0.001, 0.00025),        # worst 20.4, 0.000558, 0.000132
    "dx_in": (12, 0.0005, 0.0004),    # worst 6.12, 0.000279, 0.000227
    "y": (80, 0.01, 0.0006),          # worst 48, 0.00571, 0.000312
    "dattn": (300, 0.04, 0.003),      # worst 189, 0.0237, 0.00157
    "dx_out": (250, 0.008, 0.0015),   # worst 128, 0.00472, 0.000831
    "g_wqkv": (0.004, 0.0012, 6e-05), # worst 0.00211, 0.000731, 3.57e-05
    "g_bqkv": (8e-07, 0, 1.5e-07),    # worst 4.17e-07, 0, 7.56e-08
    "g_lnw1": (0.003, 0.015, 0.00025),# worst 0.00163, 0.00879, 0.000146
    "g_lnb1": (0.006, 0.01, 0.00025), # worst 0.00335, 0.00586, 0.00015
    "g_wo": (0.04, 0.1, 0.001),       # worst 0.0204, 0.0578, 0.000566
    "g_bo": (0.025, 0.08, 0.0015),    # worst 0.0139, 0.0488, 0.000829
    "g_lnw2": (0.015, 0.15, 0.0015),  # worst 0.00972, 0.0947, 0.000855
    "g_lnb2": (0.01, 0.15, 0.0015),   # worst 0.00543, 0.083, 0.000794
    "g_w1": (0.08, 0.04, 0.0008),     # worst 0.0442, 0.023, 0.000428
    "g_b1": (0.015, 0.04, 0.0006),    # worst 0.00896, 0.0242, 0.000386
    "g_w2": (0.05, 0.06, 0.001),      # worst 0.0274, 0.0323, 0.000522
    "g_b2": (8e-07, 0, 1.5e-07),      # worst 4.25e-07, 0, 7.92e-08
}


def _cdiv(a, b):
    return -(-a // b)


def wgrad_splits(M, N, K, other_ctas):
    """The split-K of a weight-gradient job g[N, K] = dy[M, N]^T x[M, K] as wgrad_job (gemm_internal.h) asks for it and
    avctc_gemm_launch_group settles it: -> (splits, k-blocks per split, total k-blocks of 64 rows)."""
    tiles = _cdiv(N, 128) * _cdiv(K, 128)
    s = min(max((296 - other_ctas + tiles - 1) // tiles, 1), 8)
    total = _cdiv(M, 64)
    s = min(s, total)
    per = _cdiv(total, s)
    return _cdiv(total, per), per, total


def _tiles(M, N):
    return _cdiv(M, 128) * _cdiv(N, 128)


def wgrad_jobs(M, E, F):
    """name -> (N, K, splits, k-blocks per split, total k-blocks) for the four weight-gradient GEMMs."""
    jobs = {"g_wqkv": (3 * E, E, _tiles(M, E)), "g_w2": (E, F, _tiles(M, F)), "g_w1": (F, E, _tiles(M, E)),
            "g_wo": (E, E, _tiles(M, E))}
    return {n: (N, K) + wgrad_splits(M, N, K, o) for n, (N, K, o) in jobs.items()}


def _lib():
    import multimodal_av_model_b200 as pkg
    return pkg._lib


# ----------------------------------------------------------------------------------------------------- inputs
def _inputs(E, F, M, seed):
    dev = torch.device("cuda")
    g = torch.Generator(device="cpu").manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g)
    rows = torch.arange(M)
    zero, offs = rows % 97 == 5, rows % 89 == 3                # padded frames; rows with a large mean
    x = r(M, E)
    x[offs] = 50 + 0.1 * x[offs]
    x[zero] = 0
    attn = r(M, E)
    w = dict(wqkv=r(3 * E, E) / E ** 0.5, bqkv=0.1 * r(3 * E), wo=r(E, E) / E ** 0.5, bo=0.1 * r(E),
             w1=r(F, E) / E ** 0.5, b1=0.1 * r(F), w2=r(E, F) / F ** 0.5, b2=0.1 * r(E))
    w = {k: v.to(bf16) for k, v in w.items()}                 # weights in bf16, biases bf16-rounded, as autocast sees them
    attn[zero | offs] = 0
    x2 = x.clone()                                             # residual input of attn_out_ffn: h = 0 on the zero rows
    x2[zero] = -w["bo"].float()
    ln = dict(lnw1=torch.empty(E).uniform_(0.5, 1.5, generator=g), lnb1=torch.empty(E).uniform_(-0.2, 0.2, generator=g),
              lnw2=torch.empty(E).uniform_(0.5, 1.5, generator=g), lnb2=torch.empty(E).uniform_(-0.2, 0.2, generator=g))
    t = dict(x=x.to(bf16), x2=x2.to(bf16), attn=attn.to(bf16), dq=r(M, E).to(bf16), dk=r(M, E).to(bf16),
             dv=r(M, E).to(bf16), dy=r(M, E).to(bf16), **w, **ln)
    t = {k: v.to(dev).contiguous() for k, v in t.items()}
    for k in ("bqkv", "bo", "b1", "b2"):
        t[k + "_f"] = t[k].float()
    return t


def aten_masks(M, E, F, probs, training, seed, offset, late=False):
    """The three dropout masks as native_dropout draws them in module order from the CUDA generator at (seed, offset),
    and the generator offset increment of each.  late: each mask drawn one increment past its own offset."""
    gen = torch.cuda.default_generators[torch.cuda.current_device()]
    gen.manual_seed(seed)
    gen.set_offset(offset)
    masks, incs = [], []
    for n, p in zip((E, F, E), probs):
        if not (training and p > 0):
            masks.append(None)
            incs.append(0)
            continue
        ones = torch.ones(M, n, dtype=bf16, device="cuda")
        o0 = gen.get_offset()
        m = torch.native_dropout(ones, p, True)[1]
        incs.append(gen.get_offset() - o0)
        if late:
            gen.set_offset(o0 + incs[-1])
            m = torch.native_dropout(ones, p, True)[1]
            gen.set_offset(o0 + incs[-1])
        masks.append(m)
    return masks, incs


# ----------------------------------------------------------------------------------------------------- kernels
def run_kernels(t, E, F, M, probs, training, seed, offset, wg=True):
    lib = _lib()
    L = lib.lib()
    dev = t["x"].device
    st = lib.stream_ptr(dev)
    nan = lambda *s, dt=bf16: torch.full(s, float("nan"), dtype=dt, device=dev)
    ws = lambda which: torch.empty(L.avctc_w2v_workspace_bytes(M, E, F if which % 2 else 8, which), dtype=torch.uint8,
                                   device=dev)
    o = {}
    s_in, s_out, sc_in, sc_out = ws(0), ws(1), ws(2), ws(3)
    o["q"], o["k"], o["v"] = nan(M, E), nan(M, E), nan(M, E)
    lib.check(L.avctc_w2v_attn_in_forward(t["x"].data_ptr(), M, E, t["lnw1"].data_ptr(), t["lnb1"].data_ptr(), EPS,
                                          t["wqkv"].data_ptr(), t["bqkv_f"].data_ptr(), o["q"].data_ptr(),
                                          o["k"].data_ptr(), o["v"].data_ptr(), s_in.data_ptr(), s_in.numel(), st),
              "attn_in_forward")
    o["dx_in"] = nan(M, E)
    g = [nan(3 * E, E, dt=torch.float32), nan(3 * E, dt=torch.float32), nan(E, dt=torch.float32),
         nan(E, dt=torch.float32)] if wg else [None] * 4
    lib.check(L.avctc_w2v_attn_in_backward(t["dq"].data_ptr(), t["dk"].data_ptr(), t["dv"].data_ptr(), t["x"].data_ptr(),
                                           M, E, t["lnw1"].data_ptr(), t["wqkv"].data_ptr(), o["dx_in"].data_ptr(),
                                           *[a.data_ptr() if a is not None else None for a in g], s_in.data_ptr(),
                                           s_in.numel(), sc_in.data_ptr(), sc_in.numel(), st), "attn_in_backward")
    if wg:
        o.update(zip(("g_wqkv", "g_bqkv", "g_lnw1", "g_lnb1"), g))
    o["y"] = nan(M, E)
    lib.check(L.avctc_w2v_attn_out_ffn_forward(t["attn"].data_ptr(), t["x2"].data_ptr(), M, E, F, t["wo"].data_ptr(),
                                               t["bo_f"].data_ptr(), t["lnw2"].data_ptr(), t["lnb2"].data_ptr(), EPS,
                                               t["w1"].data_ptr(), t["b1_f"].data_ptr(), t["w2"].data_ptr(),
                                               t["b2_f"].data_ptr(), *probs, training, seed, offset, o["y"].data_ptr(),
                                               s_out.data_ptr(), s_out.numel(), st), "attn_out_ffn_forward")
    o["dattn"], o["dx_out"] = nan(M, E), nan(M, E)
    shapes = ((E, E), (E,), (E,), (E,), (F, E), (F,), (E, F), (E,))
    g = [nan(*s, dt=torch.float32) for s in shapes] if wg else [None] * 8
    lib.check(L.avctc_w2v_attn_out_ffn_backward(t["dy"].data_ptr(), t["attn"].data_ptr(), M, E, F, t["wo"].data_ptr(),
                                                t["lnw2"].data_ptr(), t["w1"].data_ptr(), t["w2"].data_ptr(), *probs,
                                                training, seed, offset, o["dattn"].data_ptr(), o["dx_out"].data_ptr(),
                                                *[a.data_ptr() if a is not None else None for a in g],
                                                s_out.data_ptr(), s_out.numel(), sc_out.data_ptr(), sc_out.numel(), st),
              "attn_out_ffn_backward")
    if wg:
        o.update(zip(("g_wo", "g_bo", "g_lnw2", "g_lnb2", "g_w1", "g_b1", "g_w2", "g_b2"), g))
    torch.cuda.synchronize()
    return o


# ----------------------------------------------------------------------------------------------------- oracle
def run_oracle(t, masks, probs):
    q, k, v, s_in = wo.attn_in_forward(t["x"], t["lnw1"], t["lnb1"], EPS, t["wqkv"], t["bqkv"])
    g_in = wo.attn_in_backward(t["dq"], t["dk"], t["dv"], s_in)
    y, s_out = wo.attn_out_ffn_forward(t["attn"], t["x2"], t["wo"], t["bo"], t["lnw2"], t["lnb2"], EPS, t["w1"], t["b1"],
                                       t["w2"], t["b2"], masks=masks, probs=probs)
    g_out = wo.attn_out_ffn_backward(t["dy"], s_out)
    ref = dict(q=q, k=k, v=v, dx_in=g_in["dx"], g_wqkv=g_in["g_wqkv"], g_bqkv=g_in["g_bqkv"], g_lnw1=g_in["g_lnw"],
               g_lnb1=g_in["g_lnb"], y=y, dattn=g_out["dattn"], dx_out=g_out["dx"])
    ref.update({n: g_out[n] for n in ("g_wo", "g_bo", "g_w1", "g_b1", "g_w2", "g_b2")})
    ref["g_lnw2"], ref["g_lnb2"] = g_out["g_lnw"], g_out["g_lnb"]
    return ref, dict(s_in=s_in, g_in=g_in, s_out=s_out, g_out=g_out)


def errors(out, ref, name):
    """-> (max error, fraction of elements above one bf16 ulp, relative norm error); see the module docstring."""
    d = (out.to(f64) - ref).abs()
    rms = ref.pow(2).mean().sqrt()
    ulp = torch.exp2(torch.floor(torch.log2(torch.clamp(ref.abs(), min=rms.item() / 64 + 1e-300))) - 7)
    e = d / ulp
    mx = e.max() if name in BF16_OUT else d.max() / rms
    return mx.item(), (e > 1).double().mean().item(), (d.norm() / ref.norm()).item()


def within(errs, name):
    b = BOUNDS[name]
    return all(v <= lim for v, lim in zip(errs, b))


# ----------------------------------------------------------------------------------------------------- mutants
def _rows_sum(a, b, rows):
    return a[rows].T @ b[rows]


def mutants(case, t, ref, st, masks_late, masks):
    """name -> mutated copy of the oracle's outputs, or None where the mutant changes nothing in this case."""
    E, F, M, probs, training = case
    gi, go, si, so = st["g_in"], st["g_out"], st["s_in"], st["s_out"]
    out = {}
    # 1. each weight gradient missing its last split's k-blocks (the whole sum when there is one split)
    jobs = wgrad_jobs(M, E, F)
    m = dict(ref)
    for n, dyx in (("g_wqkv", (gi["dqkv"], si["ln"])), ("g_w2", (go["dz"], so["act"])),
                   ("g_w1", (go["dpre"], so["ln"])), ("g_wo", (go["dzo"], so["attn"]))):
        s, per = jobs[n][2], jobs[n][3]
        r0 = (s - 1) * per * 64
        m[n] = ref[n] - _rows_sum(*dyx, slice(r0, M))
    out["wgrad_last_split"] = m
    # 2. each bias gradient missing its last row chunk
    per = _cdiv(M, K_COL_PARTS)
    r0 = (K_COL_PARTS - 1) * per
    if r0 < M:
        m = dict(ref)
        for n, g in (("g_bqkv", gi["dqkv"]), ("g_b2", go["dz"]), ("g_b1", go["dpre"]), ("g_bo", go["dzo"])):
            m[n] = ref[n] - g[r0:].sum(0)
        out["bias_last_chunk"] = m
    else:
        out["bias_last_chunk"] = None
    # 3. both LayerNorms' weight and bias gradients missing the rows of the last LayerNorm-backward CTA
    P = min(_cdiv(M, K_ROWS_PER_CTA), K_LN_BWD_CTAS)
    rows = (torch.arange(M, device=ref["y"].device) // K_ROWS_PER_CTA) % P == K_LN_BWD_CTAS - 1
    if bool(rows.any()):
        m = dict(ref)
        for sfx, dln, s in (("1", gi["dln"], si), ("2", go["dln"], so)):
            m["g_lnw" + sfx] = ref["g_lnw" + sfx] - (dln[rows] * s["xhat"][rows]).sum(0)
            m["g_lnb" + sfx] = ref["g_lnb" + sfx] - dln[rows].sum(0)
        out["ln_last_cta"] = m
    else:
        out["ln_last_cta"] = None
    # 4. masks one increment late; 5. the output dropout reusing the hidden dropout's mask
    dropping = training and any(p > 0 for p in probs)
    out["masks_late"] = run_oracle(t, masks_late, probs)[0] if dropping else None
    if training and probs[0] > 0 and probs[2] > 0:
        out["out_reuses_hidden_mask"] = run_oracle(t, (masks[0], masks[1], masks[0]), probs)[0]
    else:
        out["out_reuses_hidden_mask"] = None
    # 6. attn_out_ffn's dx without the residual branch's dy
    dxn = wo._ln_bwd(go["dln"], so["xhat"], so["rstd"], so["ln_w"])[0]
    out["dx_no_residual"] = dict(ref, dx_out=dxn.to(bf16).to(f64))
    return out


def _masks64(masks):
    return tuple(None if m is None else m.to(f64) for m in masks)


@gpu
@pytest.mark.parametrize("case", CASES, ids=[f"E{c[0]}-F{c[1]}-M{c[2]}-p{'/'.join(map(str, c[3]))}-t{c[4]}" for c in CASES])
def test_entry_points_match_oracle(case):
    E, F, M, probs, training = case
    i = CASES.index(case)
    seed, offset = 1000 + i, 8 * i
    L = _lib().lib()
    t = _inputs(E, F, M, seed=i)
    masks, incs = aten_masks(M, E, F, probs, training, seed, offset)
    assert sum(incs) == L.avctc_w2v_dropout_increment(M, E, F, *probs, training)
    out = run_kernels(t, E, F, M, probs, training, seed, offset)
    lean = run_kernels(t, E, F, M, probs, training, seed, offset, wg=False)
    for n in ("q", "k", "v", "y", "dx_in", "dattn", "dx_out"):      # weight gradients on or off: same input gradients
        assert torch.equal(lean[n], out[n]), n
    ref, st = run_oracle(t, _masks64(masks), probs)
    print(f"\ncase E={E} F={F} M={M} p={probs} training={training}; split-K (splits, k-blocks per split, total, "
          "k-blocks of the last split):", {n: j[2:] + (j[4] - (j[2] - 1) * j[3],) for n, j in wgrad_jobs(M, E, F).items()})
    bad = []
    for n in BOUNDS:
        assert torch.isfinite(out[n]).all(), n
        e = errors(out[n], ref[n], n)
        print(f"  {n:7s} max {e[0]:10.4g} {'ulp' if n in BF16_OUT else 'rms'}  >1ulp {e[1]:9.3g}  rel {e[2]:9.3g}")
        if not within(e, n):
            bad.append((n, e, BOUNDS[n]))
    assert not bad, bad
    late, _ = aten_masks(M, E, F, probs, training, seed, offset, late=True)
    for name, m in mutants(case, t, ref, st, _masks64(late), _masks64(masks)).items():
        if m is None:
            print(f"  mutant {name}: changes nothing here")
            continue
        caught = [n for n in BOUNDS if not within(errors(out[n], m[n], n), n)]
        print(f"  mutant {name}: rejected by {caught}")
        assert caught, name


def test_cases_reach_every_edge_and_every_mutant():
    """Host-side: the case list hits every LayerNorm width, each F tail, a short last split-K share, the LayerNorm
    backward striding over rows, a non-empty last bias row chunk, and gives every mutant a case where it shows."""
    assert {c[0] for c in CASES} == {256, 512, 768, 1024}
    for e in (256, 512, 768, 1024):
        assert {c[1] for c in CASES if c[0] == e} >= {4 * e, 4 * e + 8, 1032}
    short = [(c, n) for c in CASES for n, j in wgrad_jobs(c[2], c[0], c[1]).items() if j[4] % j[3]]
    assert any(c[2] == 1200 and n == "g_w2" and c[0] == 256 for c, n in short)
    assert any(c[2] > K_ROWS_PER_CTA * K_LN_BWD_CTAS for c in CASES)
    assert any(c[2] < 64 for c in CASES) and any(c[2] < K_COL_PARTS for c in CASES)
    assert any(c[2] >= 8 * 1500 for c in CASES)
    assert any((K_COL_PARTS - 1) * _cdiv(c[2], K_COL_PARTS) < c[2] for c in CASES)
    assert any(c[4] == 0 for c in CASES) and any(c[4] and len(set(c[3])) == 3 for c in CASES)
    assert any(c[4] and c[3][0] > 0 and c[3][2] > 0 for c in CASES)


# ----------------------------------------------------------------------------------------------------- error contract
_NAMES = {
    "avctc_w2v_attn_in_forward": "x M E lnw1 lnb1 eps wqkv bqkv_f q k v s_in s_in_n stream",
    "avctc_w2v_attn_in_backward": "dq dk dv x M E lnw1 wqkv dx g_wqkv g_bqkv g_lnw1 g_lnb1 s_in s_in_n sc_in sc_in_n "
                                  "stream",
    "avctc_w2v_attn_out_ffn_forward": "attn x2 M E F wo bo_f lnw2 lnb2 eps w1 b1_f w2 b2_f ph pa po training seed offset y "
                                      "s_out s_out_n stream",
    "avctc_w2v_attn_out_ffn_backward": "dy attn M E F wo lnw2 w1 w2 ph pa po training seed offset dattn dx g_wo g_bo g_lnw2 "
                                       "g_lnb2 g_w1 g_b1 g_w2 g_b2 s_out s_out_n sc_out sc_out_n stream",
}
_WGRADS = {"avctc_w2v_attn_in_backward": ("g_wqkv", "g_bqkv", "g_lnw1", "g_lnb1"),
           "avctc_w2v_attn_out_ffn_backward": ("g_wo", "g_bo", "g_lnw2", "g_lnb2", "g_w1", "g_b1", "g_w2", "g_b2")}


@pytest.fixture(scope="module")
def abi_args():
    """Valid arguments of the four entry points at E = 256, F = 1024, M = 16 (pointers as integers)."""
    E, F, M = 256, 1024, 16
    lib = _lib()
    L = lib.lib()
    t = _inputs(E, F, M, seed=99)
    dev = t["x"].device
    keep = dict(t)
    for name, which in (("s_in", 0), ("s_out", 1), ("sc_in", 2), ("sc_out", 3)):
        n = L.avctc_w2v_workspace_bytes(M, E, F if which % 2 else 8, which)
        keep[name] = torch.empty(n, dtype=torch.uint8, device=dev)
    for n in ("q", "k", "v", "dx", "y", "dattn"):
        keep[n] = torch.empty(M, E, dtype=bf16, device=dev)
    shapes = dict(g_wqkv=(3 * E, E), g_bqkv=(3 * E,), g_lnw1=(E,), g_lnb1=(E,), g_wo=(E, E), g_bo=(E,), g_lnw2=(E,),
                  g_lnb2=(E,), g_w1=(F, E), g_b1=(F,), g_w2=(E, F), g_b2=(E,))
    keep.update({n: torch.empty(s, device=dev) for n, s in shapes.items()})
    a = {n: v.data_ptr() for n, v in keep.items()}
    a.update({n + "_n": keep[n].numel() for n in ("s_in", "s_out", "sc_in", "sc_out")})
    a.update(M=M, E=E, F=F, eps=EPS, ph=0.1, pa=0.1, po=0.1, training=1, seed=5, offset=0, stream=lib.stream_ptr(dev))
    return keep, a


def _call(fn, a, **over):
    L = _lib().lib()
    return getattr(L, fn)(*[over.get(n, a[n]) for n in _NAMES[fn].split()])


@gpu
def test_error_contract(abi_args):
    keep, a = abi_args
    for fn in _NAMES:                                        # the valid call succeeds (forward first: backward reads it)
        assert _call(fn, a) == OK, fn
    torch.cuda.synchronize()
    L = _lib().lib()
    for fn in _NAMES:
        for E in (128, 384, 1280):
            assert _call(fn, a, E=E) == UNSUPPORTED, (fn, E)
        assert _call(fn, a, M=0) == UNSUPPORTED, fn
        if "out_ffn" in fn:
            assert _call(fn, a, F=1028) == UNSUPPORTED, fn
        first = _NAMES[fn].split()[0]
        assert _call(fn, a, **{first: a[first] + 2}) == ALIGNMENT, fn
        for ws in [n for n in _NAMES[fn].split() if n.endswith("_n")]:
            assert _call(fn, a, **{ws: a[ws] - 1}) == WORKSPACE, (fn, ws)
        for i, g in enumerate(_WGRADS.get(fn, ())):          # weight-gradient pointers: all or none
            assert _call(fn, a, **{g: None}) == BAD_ARG, (fn, g)
            others = {o: None for o in _WGRADS[fn] if o != g}
            assert _call(fn, a, **others) == BAD_ARG, (fn, g)
        if fn in _WGRADS:
            assert _call(fn, a, **{g: None for g in _WGRADS[fn]}) == OK, fn
    torch.cuda.synchronize()
    for M, E, F in [(16, 128, 1024), (16, 384, 1024), (16, 1280, 1024), (16, 256, 1028), (0, 256, 1024)]:
        assert all(L.avctc_w2v_workspace_bytes(M, E, F, w) == 0 for w in range(4)), (M, E, F)


def test_native_shape_rule_matches_make_dims():
    """The Python rule that routes a layer to the native path accepts exactly the (M, E, F) the library accepts
    (workspace_bytes > 0).  Host-only: no device needed."""
    from multimodal_av_model_b200 import encoders
    L = _lib().lib()
    for M in (0, 1, 1992):
        for E in range(-256, 1537, 128):
            for F in (-8, 0, 4, 8, 12, 1024, 1028, 1032, 4096, 4100, 4104):
                ok = encoders._w2v_native_shape_ok(M, E, F)
                assert ok == all(L.avctc_w2v_workspace_bytes(M, E, F, w) > 0 for w in range(4)), (M, E, F)
                assert ok == (L.avctc_w2v_workspace_bytes(M, E, F, 1) > 0), (M, E, F)
