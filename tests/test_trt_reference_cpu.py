"""The TRT reference of the GPU tests (trt_reference.c) on the CPU: with magic = (tau - 1/2)^2 its two rates are
equal and it must reproduce the oracle's BGK step; with another magic parameter it must not."""
import numpy as np
import pytest

import helpers as H
import trt_reference as TRT


@pytest.mark.parametrize("name,n", [("ldc", 16), ("pos", 16), ("bif", None), ("cor", None)])
def test_trt_with_equal_rates_is_bgk(name, n):
    bgk, *_ = H.oracle_case(name, n, np.float64)
    trt, *_ = H.oracle_case(name, n, np.float64)
    tau = float(np.float64(H.TAU_POS if name == "pos" else H.TAU_LDC))
    bgk.step(60)
    TRT.step(trt, 60, (tau - 0.5) ** 2)
    err = H.rel_err(trt.fields(), bgk.fields())
    assert err <= 1e-13, err
    assert np.abs(trt.populations() - bgk.populations()).max() <= 1e-14


def test_trt_with_another_magic_differs_from_bgk():
    bgk, *_ = H.oracle_case("pos", 16, np.float64)
    trt, *_ = H.oracle_case("pos", 16, np.float64)
    bgk.step(60)
    TRT.step(trt, 60, 3 / 16)
    assert H.rel_err(trt.fields(), bgk.fields()) > 1e-6
