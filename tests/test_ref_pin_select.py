"""PINS THE ORACLE'S PIXEL SELECTION TO THE REFERENCE: PixelSelector::makeMaps (FullSystem/PixelSelector2.cpp) and the loop of
FullSystem::makeNewTraces, restated in oracle/orc_select.cpp, against the reference's own compiled code.  The reference's results are stored
in tests/golden/ref_select.npz (recorded by tests/golden/make_select_golden.py), so the pin holds on every checkout.

Bar: BIT-EXACT — the whole selection map, numHaveSub and the selector's potential after the call."""
import ctypes
import os

import numpy as np
import pytest

import select_cases as S
from oracle import orc_select

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_select.npz")


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(GOLDEN))


@pytest.fixture(scope="module")
def oracle_results(orc):
    def run(img, c):
        lv = orc.make_images(img, S.K640)
        m, n, pot = orc_select.make_maps(lv, c["density"], c["recursionsLeft"], c["thFactor"], c["potential"], c["B"], c["settings"])
        return m, n, pot, lv, img
    return S.run_cases(run)


def assert_map_equal(got, want, what):
    bad = np.argwhere(got != want)
    assert bad.size == 0, f"{what}: {len(bad)} pixels differ, first (y, x) = {bad[:8].tolist()}: got {got[tuple(bad[:8].T)]}, want {want[tuple(bad[:8].T)]}"


@pytest.mark.parametrize("name", list(S.CASES))
def test_make_maps_bit_exact(oracle_results, gold, name):
    m, n, pot, lv, img = oracle_results[name]
    assert str(gold[f"{name}/image_sha256"]) == S.sha(img), "the case's frame is not the one the reference was run on"
    assert_map_equal(m, gold[f"{name}/map"], name)
    assert n == int(gold[f"{name}/numHaveSub"])
    assert pot == int(gold[f"{name}/potential"])
    assert np.count_nonzero(m) == n


@pytest.mark.parametrize("name", ["quant640", "stripes640", "setfirst_stripes640", "no_direction_stripes"])
def test_cases_have_direction_dependent_cells(oracle_results, name):
    """without pot-cells whose level-0 pick depends on the block direction the n2 chain of select() would go untested"""
    c = S.resolve(name, 3)
    lv = oracle_results[name][3]
    ag0 = lv[0][..., 1] * lv[0][..., 1] + lv[0][..., 2] * lv[0][..., 2]
    assert S.direction_dependent_cells(lv[0], ag0, c["potential"], c["thFactor"]) > 0


def test_cases_cover_the_control_paths(gold):
    pots = {n: (S.resolve(n, 3)["potential"], int(gold[f"{n}/potential"])) for n in S.CASES}
    assert pots["more_points"][1] < pots["more_points"][0]       # quotia > 1.25: re-selected with a smaller potential
    assert pots["fewer_points"][1] > pots["fewer_points"][0]     # quotia < 0.25: re-selected with a larger potential
    for n in ("quant640", "no_recursion_subsample"):               # quotia < 0.95: sub-sampled with randomPattern
        c = S.resolve(n, 3)
        assert int(gold[f"{n}/numHaveSub"]) < c["density"] / 0.95


def test_random_pattern_is_glibc_rand():
    libc = ctypes.CDLL(None)
    libc.srand(3141592)
    want = np.array([libc.rand() & 0xFF for _ in range(20000)], np.uint8)
    assert np.array_equal(orc_select.random_pattern(20000), want)


@pytest.mark.parametrize("name", S.TRACE_CASES)
def test_make_new_traces_bit_exact(orc, gold, name):
    c = S.resolve(name, 3)
    lv = orc.make_images(S.IMAGES[c["img"]](), S.K640)
    P, sub, pot = orc_select.make_new_traces(lv, c["density"], c["recursionsLeft"], c["thFactor"], c["potential"], c["B"], c["settings"])
    assert sub == int(gold[f"{name}/numHaveSub"]) and pot == int(gold[f"{name}/potential"])
    for k in ("u", "v", "type", "color", "weights", "gradH", "energyTH"):
        want = gold[f"{name}/traces/{k}"]
        assert P[k].shape == want.shape, k
        assert np.array_equal(P[k].view(np.uint32) if P[k].dtype == np.float32 else P[k], want.view(np.uint32) if want.dtype == np.float32 else want), k
