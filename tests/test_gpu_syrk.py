"""The DMMA SYRK (syrk_tma.cu) behind T.gram: G = X'X against a reference product, at every block count the plan
handles and at row counts around the 16-row ring stage and the 32-row split tile.

Diagonal 128-blocks compute only their 8 x 8 tiles on or above the diagonal, dealt 17 per warp; the reduction mirrors
them.  n = 65 .. 2048 covers 1, 2, 3, 4 and 16 blocks per edge, partial last blocks included."""
import numpy as np
import pytest

import tlsq_b200 as T

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps


def _x(M, n, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    # column-major M x n; a non-zero mean makes the Gram's diagonal dominate, like the ALM iterates
    return (torch.randn(n, M, dtype=torch.float64, device="cuda", generator=g) + 0.5).t()


def _check(M, n, seed):
    X = _x(M, n, seed)
    G = T.gram(X)
    ref = X.t() @ X
    bound = M * EPS * (X.abs().t() @ X.abs())             # FP64 error bound of a length-M sum, both sides
    err = (G - ref).abs()
    assert bool((err <= bound).all()), float((err / bound).max())
    assert bool((G == G.t()).all())


@pytest.mark.parametrize("n", [65, 128, 129, 256, 384, 512, 2048])
@pytest.mark.parametrize("M", [4096, 4112, 4126, 4128, 4130, 4144])
def test_gram_matches_reference(M, n):
    _check(M, n, seed=M * 7 + n)


def test_gram_tall():
    """Many tiles per split, a ragged last tile."""
    _check(1_000_018, 256, seed=3)


def test_gram_repeatable():
    """The ring refills a stage once every warp has released it; an early refill would show as run-to-run noise."""
    X = _x(600_000, 256, seed=9)
    G0 = T.gram(X)
    for _ in range(5):
        assert bool((T.gram(X) == G0).all())
