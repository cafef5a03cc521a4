"""The Stage-1 separation loss kernel (csrc/separation.cu, C ABI ogs_separation_loss) against a float64 restatement of
train.py:123-155 (helpers.separation_loss_fp64) at the sizes where its indexing can go wrong: fewer rows than one
128-thread stride, exactly one, one more, several; 1..16 channels; both weight rules (iteration > 35000 keeps only the
top weights); a block of identical all-zero rows (masks without rendered pixels: clamp(min=1) makes their mean 0) and
other exact ties, which the kernel ranks by column."""
import numpy as np
import pytest
import torch

from helpers import grad_violations, min_rank_gap, separation_loss_fp64

pytestmark = pytest.mark.gpu

NS = (2, 3, 31, 127, 128, 129, 300, 1031, 4099)
CS = (1, 3, 6, 16)
ROWS = 128           # rows of the [N, N] reference matrix evaluated (and differentiated) at a time


def _means(N, C, seed):
    """Means on a lattice of step 1/16 (coordinates and every squared distance exact in float32, so the kernel's and the
    reference's inverse distances are the same correctly rounded values up to the final division), spread so that
    squared distances stay below ~160 and distinct inverse distances differ by more than 1e-5 relative; 0..N/8 rows
    are exactly zero and many other rows repeat (C = 1 has only ~200 lattice points)."""
    g = torch.Generator().manual_seed(seed)
    R = max(2, int((40_000 / C) ** 0.5))
    m = torch.randint(0, R, (N, C), generator=g).double() - R // 2
    z = N // 8
    if z:
        k0 = int(torch.randint(0, N - z + 1, (1,), generator=g))
        m[k0:k0 + z] = 0.0
    return m / 16.0


def _reference(m, iteration):
    """(loss, dL/dmean) in float64, a block of rows at a time."""
    leaf = m.clone().requires_grad_(True)
    total = 0.0
    for r0 in range(0, m.shape[0], ROWS):
        part = separation_loss_fp64(leaf, iteration, slice(r0, r0 + ROWS))
        part.backward()
        total += float(part.detach())
    return total, leaf.grad


def _kernel(m, iteration):
    from opengaussian_b200.mask_stats import separation_loss
    x = m.float().cuda().requires_grad_(True)
    loss = separation_loss(x, iteration)
    loss.backward()
    return float(loss), x.grad.double().cpu()


@pytest.mark.parametrize("C", CS)
@pytest.mark.parametrize("N", NS)
def test_separation_kernel_vs_fp64(N, C):
    m = _means(N, C, seed=N * 31 + C)
    gap = min(min_rank_gap(m, slice(r0, r0 + ROWS)) for r0 in range(0, N, ROWS))
    assert gap > 1e-5, f"inputs too close to a rank flip: {gap:.2e}"
    assert N < 8 or int((m.abs().sum(1) == 0).sum()) >= N // 8
    for iteration in (1000, 40_000):
        want_loss, want_grad = _reference(m, iteration)
        got_loss, got_grad = _kernel(m, iteration)
        assert abs(got_loss - want_loss) <= 1e-5 * abs(want_loss), (iteration, got_loss, want_loss)
        frac, worst = grad_violations(got_grad.numpy(), want_grad.numpy(), 1e-3)
        assert frac == 0.0, (iteration, frac, worst)


def test_small_weights_rule_changes_the_loss():
    """The iteration > 35000 rule is live in these inputs (the two weightings give different losses), and the boundary
    weight rank / (N - 1) * 0.9 + 0.1 == 0.9 (N - 1 divisible by 9, N = 127 in the grid above) is computed in float32
    as the reference does."""
    m = _means(127, 6, seed=5)
    a, b = _kernel(m, 1000)[0], _kernel(m, 40_000)[0]
    assert b < 0.9 * a
    r = torch.arange(127).float()
    w = (r / 126) * (1.0 - 0.1) + 0.1
    assert int((w >= 0.9).sum()) == 15                 # ranks 112..126: the boundary rank keeps its weight


def test_seventeen_channels_take_the_torch_path():
    """More channels than the kernel's register tile (16): the reference's own expression on CUDA, same values.  Its
    CUDA argsort may order exact ties either way, so these inputs have none (continuous values; the seed passes the
    rank-gap check)."""
    m = torch.randn(40, 17, generator=torch.Generator().manual_seed(2), dtype=torch.float64) * 0.3
    assert min_rank_gap(m) > 1e-5
    for iteration in (1000, 40_000):
        want_loss, want_grad = _reference(m, iteration)
        got_loss, got_grad = _kernel(m, iteration)
        assert abs(got_loss - want_loss) <= 1e-5 * abs(want_loss), (iteration, got_loss, want_loss)
        frac, worst = grad_violations(got_grad.numpy(), want_grad.numpy(), 1e-3)
        assert frac == 0.0, (iteration, frac, worst)


def test_too_many_masks_is_refused_before_any_launch():
    from opengaussian_b200._lib import OgsError
    from opengaussian_b200.mask_stats import separation_loss
    x = torch.zeros(12289, 3, device="cuda", requires_grad=True)
    torch.cuda.synchronize()
    with pytest.raises(OgsError, match="too large"):
        separation_loss(x, 1000)
    torch.cuda.synchronize()                           # nothing was launched that could have failed
    ok = torch.ones(3, 3, device="cuda")
    assert np.isfinite(float(separation_loss(ok * torch.arange(3, device="cuda")[:, None], 1000)))
