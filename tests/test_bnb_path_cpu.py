"""CPU tests of fit_path(BnB)'s host side: the refusals made before any device work, and the library's new export."""
import pytest


def test_fit_path_refuses_alt_and_intercept_enumeration_for_bnb(pkg):
    X, y, P = [[1.0, 2.0, 3.0]] * 4, [1.0] * 4, [[1, 0], [1, 0], [0, 1]]
    with pytest.raises(TypeError):
        pkg.fit_path(pkg.Alt, X, y, P, [0.1])
    with pytest.raises(TypeError):
        pkg.fit_path(pkg.BnB, X, y, P, [0.1], enumerate_intercept=True)


def test_library_exports_bnb_path(pkg):
    assert pkg._abi.lib.pls_version() == 130
    assert hasattr(pkg._abi.lib, "pls_bnb_fit_path")
