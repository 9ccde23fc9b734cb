"""GPU: the native VisualEncoder forward (csrc/visual_encoder.cu around cuDNN's trunk convolutions) against the module
path on the same GPU, same weights: outputs within bf16 rounding, running statistics of all 20 BatchNorm layers and
num_batches_tracked as the module path leaves them, eval mode from the running statistics, and bit-identical repeats."""
import copy

import pytest
import torch

pytestmark = pytest.mark.gpu


def _pair(seed=0):
    import multimodal_av_model_b200 as pkg
    torch.manual_seed(seed)
    nat = pkg.VisualEncoder(relu_type="prelu").cuda()
    for p in nat.parameters():
        p.requires_grad = False
    with torch.no_grad():                      # non-trivial affine BatchNorm and PReLU slopes
        for m in nat.modules():
            if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
                m.weight.uniform_(0.5, 1.5)
                m.bias.uniform_(-0.2, 0.2)
            elif isinstance(m, torch.nn.PReLU):
                m.weight.uniform_(0.05, 0.4)
    ref = copy.deepcopy(nat)
    ref._native_applies = lambda x: False      # the module path, as on the CPU
    return nat, ref


def _bns(m):
    return [x for x in m.modules() if isinstance(x, torch.nn.modules.batchnorm._BatchNorm)]


def _run(m, x):
    with torch.autocast("cuda", dtype=torch.bfloat16):
        return m._forward_impl(x)


# Train-mode BatchNorm normalises with statistics of the batch itself.  In a batch of a few frames (layer4 sees 9 values
# per channel and frame) a one-ulp bf16 difference upstream moves those statistics visibly, and 17 normalisations later
# the outputs differ by a few ulps: batches of <= 24 frames get twice the bound of the config-size batch.
def _tol(x):
    return 2 if x.shape[0] * x.shape[2] <= 24 else 1


def _close(y, z, tol=1):
    y, z = y.float(), z.float()
    d = (y - z).abs()
    assert d.max().item() <= tol * 2 ** -7 * z.abs().max().item() + 1e-2, (d.max().item(), z.abs().max().item())
    assert d.mean().item() <= 1e-2 * z.abs().mean().item(), (d.mean().item(), z.abs().mean().item())


def _stats_close(a, b, tol=1):
    la, lb = _bns(a), _bns(b)
    assert len(la) == len(lb) == 20
    for x, y in zip(la, lb):
        assert int(x.num_batches_tracked) == int(y.num_batches_tracked)
        for u, v in ((x.running_mean, y.running_mean), (x.running_var, y.running_var)):
            torch.testing.assert_close(u, v, rtol=1e-3, atol=tol * 5e-3 * v.abs().max().item())


@pytest.mark.parametrize("shape", [(8, 1, 150, 96, 96), (2, 1, 1, 96, 96), (2, 1, 2, 96, 96), (2, 1, 3, 96, 96),
                                   (1, 1, 12, 96, 96), (2, 1, 5, 88, 92)])
def test_native_visual_forward_matches_module_path_train_and_eval(shape):
    nat, ref = _pair()
    nat.train(); ref.train()
    x = torch.rand(*shape, device="cuda")
    with torch.autocast("cuda", dtype=torch.bfloat16):
        assert nat._native_applies(x)
    assert not nat._native_applies(x)                                  # no autocast: module path
    for _ in range(2):
        y, z = _run(nat, x), _run(ref, x)
        assert y.shape == z.shape == (shape[0], shape[2], 512) and y.dtype == z.dtype == torch.bfloat16
        _close(y, z, _tol(x))
    _stats_close(nat, ref, _tol(x))
    # eval mode: BatchNorm from the running statistics, nothing updated
    nat.eval(); ref.eval()
    before = [b.clone() for b in nat.buffers()]
    with torch.no_grad():
        y, z = _run(nat, x), _run(ref, x)
    _close(y, z, _tol(x))
    assert all(torch.equal(u, v) for u, v in zip(before, nat.buffers()))


def test_native_visual_forward_is_bit_identical_from_equal_states():
    nat, _ = _pair(1)
    twin = copy.deepcopy(nat)
    x = torch.rand(2, 1, 7, 96, 96, device="cuda")
    y1, y2 = _run(nat, x), _run(twin, x)
    assert torch.equal(y1, y2)
    for u, v in zip(nat.buffers(), twin.buffers()):
        assert torch.equal(u, v)


def test_native_visual_forward_runs_inside_the_graphed_segment():
    """The trainer's call goes through forward() -> GraphedSegment: the captured native kernels advance the running
    statistics once per replay (capture warm-ups leave no trace) and match the module path."""
    from multimodal_av_model_b200 import _lib
    nat, ref = _pair(2)
    nat.train(); ref.train()
    x = torch.rand(2, 1, 9, 96, 96, device="cuda")
    c0 = _lib.launch_count
    with torch.autocast("cuda", dtype=torch.bfloat16):
        outs = [nat(x).float() for _ in range(3)]
        refs = [ref._forward_impl(x).float() for _ in range(3)]
    assert _lib.launch_count > c0                                       # this library's kernels ran
    assert nat._graph_seg.captures == 1 and nat._graph_seg.replays == 2
    for y, z in zip(outs, refs):
        _close(y, z, _tol(x))
    _stats_close(nat, ref, _tol(x))
    assert int(nat.frontend3D[1].num_batches_tracked) == 3
