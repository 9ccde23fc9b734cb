"""CPU: oracle/fusion_oracle.py (round_bf16=False) is the reference of each fusion-path kernel, in float64: the resample
is oracle/torch_port.select_pad_resample (the reference's F.interpolate calls) and its backward is autograd through it
and the adjoint of the forward; softmax and log-softmax are torch's, with torch's autograd; attention is autograd through
softmax(q k^T / sqrt(128)) v; column sums and the GEMM are plain float64 products."""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import fusion_oracle as fo
from oracle import torch_port as tp

f64 = torch.float64
TOL = 1e-12


def _close(a, b, tol=TOL, floor=1e-300):
    scale = max(b.abs().max().item(), floor)
    assert (a - b).abs().max().item() <= tol * scale, ((a - b).abs().max().item(), scale)


def _mask(B, Ta, g, empty=()):
    m = torch.randint(0, 4, (B, Ta), generator=g)
    m[torch.rand(B, Ta, generator=g) < 0.5] = 1
    for b in empty:
        m[b] = torch.randint(0, 2, (Ta,), generator=g) * 3
    return m


@pytest.mark.parametrize("B,Ta,D,tv", [(3, 9, 8, "eq"), (4, 40, 12, "lt"), (2, 13, 5, "2x"), (5, 30, 8, "one"),
                                       (3, 300, 4, "lt"), (40, 11, 3, "2x")])
def test_resample_matches_torch_port(B, Ta, D, tv):
    g = torch.Generator().manual_seed(B * 100 + Ta)
    mask = _mask(B, Ta, g, empty=(1,) if B > 2 else ())
    Tp = int(((mask != 0) & (mask != 3)).sum(1).max())
    Tv = dict(eq=Tp, lt=max(1, 2 * Tp // 3), one=1).get(tv, 2 * Tp)
    audio = torch.randn(B, Ta, D, generator=g, dtype=f64)
    out, m_out, lens = fo.resample_forward(audio, mask, Tv)
    a = audio.clone().requires_grad_()
    ref, m_ref = tp.select_pad_resample(a, mask, Tv)
    _close(out, ref.detach())
    assert torch.equal(m_out, m_ref)
    assert torch.equal(lens, (m_ref != 0).sum(1))
    dout = torch.randn(B, Tv, D, generator=g, dtype=f64)
    (ref * dout).sum().backward()
    da = fo.resample_backward(dout, mask)
    _close(da, a.grad)
    # adjoint identity <dout, fwd(a)> = <bwd(dout), a>
    assert abs((dout * out).sum().item() - (da * audio).sum().item()) <= TOL * (dout.abs() * out.abs()).sum().item()


def test_resample_nearest_index_is_atens_float32_rule():
    """The mask follows F.interpolate(mode='nearest') on a float tensor, whose index is computed in float32."""
    for Tp in (1, 2, 3, 7, 49, 100, 249, 599):
        for Tv in (1, 2, 3, 5, 50, 75, 150, 199, 1000):
            x = torch.arange(Tp, dtype=torch.float32)[None, None]
            want = F.interpolate(x, size=Tv, mode="nearest")[0, 0].long()
            assert torch.equal(fo.nearest_index(Tp, Tv), want), (Tp, Tv)


@pytest.mark.parametrize("Tp,Tv", [(2, 7), (430, 286), (440, 880), (181, 120), (599, 1), (5, 3)])
def test_resample_float32_weights_are_atens(Tp, Tv):
    """With coef_dtype=float32 the weights are F.interpolate's on a float32 tensor: interpolating the identity gives
    the weight matrix (transposed), to the float32 rounding of w0 + w1 where both land on the last frame."""
    eye = torch.eye(Tp, dtype=torch.float32)[None]
    want = F.interpolate(eye, size=Tv, mode="linear", align_corners=True)[0].T.to(f64)
    got = fo.lerp_matrix(Tp, Tv, dtype=torch.float32)
    assert (got - want).abs().max().item() <= 1e-7
    if Tp >= 100 and Tv > 1:                                 # float64 weights are not
        assert (fo.lerp_matrix(Tp, Tv) - want).abs().max().item() > 1e-7


def test_resample_all_empty_batch_is_zero():
    mask = torch.tensor([[0, 3, 0], [3, 3, 0]])
    out, m_out, lens = fo.resample_forward(torch.randn(2, 3, 4, dtype=f64), mask, 5)
    assert out.abs().max() == 0 and m_out.abs().max() == 0 and lens.tolist() == [0, 0]
    assert fo.resample_backward(torch.randn(2, 5, 4, dtype=f64), mask).abs().max() == 0


@pytest.mark.parametrize("rows,T,Tp", [(1, 1, 8), (7, 33, 57), (9, 150, 152), (5, 1000, 1000)])
def test_softmax_matches_torch(rows, T, Tp):
    g = torch.Generator().manual_seed(T)
    S = torch.randn(rows, Tp, generator=g, dtype=f64) * 3
    P = fo.softmax_forward(S, T)
    s = S[:, :T].clone().requires_grad_()
    ref = torch.softmax(s, -1)
    _close(P[:, :T], ref.detach())
    assert Tp == T or P[:, T:].abs().max().item() == 0
    dP = torch.randn(rows, Tp, generator=g, dtype=f64)
    ref.backward(dP[:, :T])
    dS = fo.softmax_backward(P, dP, T)
    _close(dS[:, :T], s.grad)
    assert Tp == T or dS[:, T:].abs().max().item() == 0


@pytest.mark.parametrize("V", [1, 2, 33, 1025])
def test_log_softmax_matches_torch(V):
    g = torch.Generator().manual_seed(V)
    X = torch.randn(6, V, generator=g, dtype=f64) * 4
    X[1] = 7.0                                       # equal logits
    X[2] += 5000.0                                   # large logits
    x = X.clone().requires_grad_()
    ref = F.log_softmax(x, -1)
    Y = fo.log_softmax_forward(X)
    _close(Y, ref.detach(), 1e-12 * 5000)
    dY = torch.randn(6, V, generator=g, dtype=f64)
    ref.backward(dY)
    _close(fo.log_softmax_backward(ref.detach(), dY), x.grad)


def test_colsum_and_gemm_are_plain_sums():
    g = torch.Generator().manual_seed(0)
    X = torch.randn(37, 12, generator=g, dtype=f64)
    _close(fo.colsum(X, 9), torch.stack([sum(X[m, n] for m in range(37)) for n in range(9)]))
    A, Bm = torch.randn(5, 7, generator=g, dtype=f64), torch.randn(3, 7, generator=g, dtype=f64)
    bias, C0 = torch.randn(6, generator=g, dtype=f64), torch.randn(5, 3, generator=g, dtype=f64)
    loop = torch.tensor([[sum(A[m, k] * Bm[n, k] for k in range(7)) for n in range(3)] for m in range(5)], dtype=f64)
    _close(fo.gemm(A, Bm, 0.5), 0.5 * loop)
    _close(fo.gemm(A, Bm, 0.5, bias, 1, C0), 0.5 * loop + bias[:3] + C0)
    _close(fo.gemm(A, Bm, 0.5, bias, 2), 0.5 * loop + bias[:5, None])


@pytest.mark.parametrize("B,T,H", [(2, 1, 1), (1, 17, 2), (2, 65, 3), (1, 130, 1)])
def test_attention_matches_autograd(B, T, H):
    E = 128 * H
    g = torch.Generator().manual_seed(T * 10 + H)
    q, kv, dout = (torch.randn(B, T, n, generator=g, dtype=f64) for n in (E, 2 * E, E))
    o, lse2 = fo.attention_forward(q, kv, H, round_bf16=False)
    qh = q.view(B, T, H, 128).transpose(1, 2).clone().requires_grad_()
    kh = kv[..., :E].reshape(B, T, H, 128).transpose(1, 2).clone().requires_grad_()
    vh = kv[..., E:].reshape(B, T, H, 128).transpose(1, 2).clone().requires_grad_()
    s = qh @ kh.transpose(-1, -2) / math.sqrt(128.0)
    ref = (torch.softmax(s, -1) @ vh).transpose(1, 2).reshape(B, T, E)
    ref.backward(dout)
    _close(o, ref.detach())
    _close(lse2, (torch.logsumexp(s, -1) / math.log(2.0)).reshape(B * H, T).detach())
    dq, dk, dv = fo.attention_backward(q, kv, dout, o, lse2, H, round_bf16=False)
    for mine, x in ((dq, qh), (dk, kh), (dv, vh)):       # T = 1: dq and dk are 0, up to rounding of unit-size terms
        _close(mine, x.grad.transpose(1, 2).reshape(B, T, E), floor=1.0)
