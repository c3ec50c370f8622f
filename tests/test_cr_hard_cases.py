"""CPU: the list of hard-to-round inputs (tests/golden/cr_hard_cases.npz, make_cr_hard_cases.py) behind the kernels'
and the oracle's correct rounding of sin / cos (|a| <= 8), acos / asin (|x| <= 1) and pow(p, 2.2f) (0 < p <= 1).

Every entry's result is the correctly rounded value (mpmath, 200 bits); the oracle, which resolves these inputs on its
own in extended precision, returns it; the kernels' table (csrc/cr_hard_cases.inc) holds exactly the list; and the
generator, run again over every float of the domains, finds the same list."""
import importlib.util
import os

import numpy as np
import pytest

from oracle import oracle
from tests import fixtures
from tests.cr_reference import FUNCS, POW_EXP, correctly_rounded

GEN = os.path.join(fixtures.GOLDEN, "make_cr_hard_cases.py")


def generator():
    spec = importlib.util.spec_from_file_location("make_cr_hard_cases", GEN)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def hard_cases():
    z = np.load(os.path.join(fixtures.GOLDEN, "cr_hard_cases.npz"))
    assert list(z["names"]) == FUNCS
    return {name: (z["x"][z["fn"] == i], z["y"][z["fn"] == i]) for i, name in enumerate(FUNCS)}


def oracle_at(name, x):
    xf = x.view(np.float32)
    if name == "pow":
        return oracle.math_probe("pow", xf, np.full_like(xf, POW_EXP)).view(np.uint32)
    return oracle.math_probe(name, xf).view(np.uint32)


@pytest.mark.parametrize("name", FUNCS)
def test_entries_are_correctly_rounded_and_the_oracle_returns_them(name):
    x, y = hard_cases()[name]
    assert x.size > 0 and np.all(np.diff(x.astype(np.int64)) > 0)
    assert np.array_equal(y, correctly_rounded(name, x.view(np.float32)))
    got = oracle_at(name, x)
    assert np.array_equal(got, y), f"oracle wrong on {[hex(v) for v in x[got != y]]}"
    if name == "pow":            # and through the tonemap
        assert np.array_equal(oracle.img_processing(x.view(np.float32), x.size).view(np.uint32), y)


def test_oracle_was_wrong_without_the_guard_on_the_two_acos_inputs():
    """the once-rounded glibc binary64 value misrounds these two (found by the generator); the guard must catch them"""
    x = np.array([0x328885A3, 0x39826222], np.uint32)
    y = np.array([0x3FC90FDB, 0x3FC907B5], np.uint32)
    assert np.array_equal(correctly_rounded("acos", x.view(np.float32)), y)
    once = np.arccos(x.view(np.float32).astype(np.float64)).astype(np.float32).view(np.uint32)
    assert not np.any(once == y)
    assert np.array_equal(oracle_at("acos", x), y)


def test_kernel_table_is_the_list():
    gen = generator()
    z = np.load(os.path.join(fixtures.GOLDEN, "cr_hard_cases.npz"))
    assert int(z["window"]) == gen.WINDOW
    with open(gen.INC) as f:
        assert f.read() == gen.inc_text(z["fn"], z["x"], z["y"])


def test_generator_reproduces_the_committed_list():
    """a fresh binary64 pass over every float of the domains (about 10^10 evaluations, seconds on a few cores)"""
    gen = generator()
    fn, x, y, _ = gen.compute(verbose=False)
    with open(os.path.join(fixtures.GOLDEN, "cr_hard_cases.npz"), "rb") as f:
        assert f.read() == gen.npz_bytes(fn, x, y)
