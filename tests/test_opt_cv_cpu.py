"""CPU tests of fit_cv's host side: the default fold drawing and the argument checks made before any device work."""
import numpy as np
import pytest


def test_default_folds_are_balanced_and_reproducible(pkg):
    for N, F in ((100, 5), (101, 5), (7, 2), (1000, 32)):
        f = pkg.draw_folds(N, F, seed=3)
        assert f.shape == (N,) and f.dtype == np.int32
        counts = np.bincount(f, minlength=F)
        assert len(counts) == F and counts.max() - counts.min() <= 1
        assert np.array_equal(f, pkg.draw_folds(N, F, seed=3))
        assert np.array_equal(f, np.random.default_rng(3).permutation(N) % F)
    assert not np.array_equal(pkg.draw_folds(1000, 5, seed=0), pkg.draw_folds(1000, 5, seed=1))


def test_fit_cv_refuses_bnb_and_alt(pkg):
    X, y, P = np.ones((10, 3)), np.ones(10), np.array([[1, 0], [1, 0], [0, 1]])
    for alg in (pkg.BnB, pkg.Alt):
        with pytest.raises(TypeError):
            pkg.fit_cv(alg, X, y, P, [0.1])


@pytest.mark.parametrize("kw,etas", [
    (dict(folds=1), [0.1]),
    (dict(folds=33), [0.1]),
    (dict(folds=2.5), [0.1]),
    (dict(folds=20), [0.1]),                                   # more folds than rows
    (dict(), []),
    (dict(), [0.1] * 65),
    (dict(), [0.1, -1.0]),
    (dict(), [float("nan")]),
    (dict(), [float("inf")]),
    (dict(fold_ids=np.arange(12) % 2), [0.1]),                 # wrong length
    (dict(fold_ids=np.zeros(10, dtype=int)), [0.1]),           # one fold
    (dict(fold_ids=np.arange(10) % 2 * 2), [0.1]),             # fold 1 empty
    (dict(fold_ids=np.arange(10) % 2 - 1), [0.1]),             # negative id
    (dict(fold_ids=np.arange(10) % 2 + 0.5), [0.1]),           # not integers
    (dict(fold_ids=np.arange(10) % 33 + np.r_[np.zeros(9), 32]), [0.1]),
])
def test_fit_cv_checks_arguments_on_the_host(pkg, kw, etas):
    """Bad arguments raise ValueError before a context is made (so also without a GPU)."""
    X, y, P = np.ones((10, 3)), np.ones(10), np.array([[1, 0], [1, 0], [0, 1]])
    with pytest.raises(ValueError):
        pkg.fit_cv(pkg.Opt, X, y, P, etas, **kw)
