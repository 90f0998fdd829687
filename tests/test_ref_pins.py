"""The oracle pinned against the REFERENCE's own code.

tests/golden/ref_pins.npz holds seeded inputs and the outputs of LuisaRender's src/util functions for them — the functions
themselves, compiled from /root/reference and executed through the LuisaCompute-AST interpreter of oracle/ref (generator:
tools/gen_ref_pins.py).  Here the oracle's restatements (oracle_unit) must reproduce them:

  * integer results (hashes, LCG / PCG32 states, alias-table picks): bit-exact;
  * float results: |a - b| <= 2e-5 * max(1, |b|) (SURVEY.md §8c: 4 ulp / 1e-5 relative on continuous quantities; the
    reference's two backends themselves differ by more: fma contraction, rsqrt, libm);
    present state: 12 288 cases, 12 073 rows bit-identical, none beyond the tolerance (no outliers are allowed).

When oracle/_ref/librefpins.so is present (this container) the fixture is additionally re-generated live and compared, so a
stale fixture cannot hide a change.
"""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np
import pytest

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))
sys.path.insert(0, str(REPO / "tools"))

import gen_ref_pins as G  # noqa: E402
from oracle import binding as O  # noqa: E402

GOLDEN = REPO / "tests" / "golden" / "ref_pins.npz"
RTOL = 2e-5
MAX_OUTLIER_SHARE = 0.0


@pytest.fixture(scope="module")
def golden():
    assert GOLDEN.exists(), "tests/golden/ref_pins.npz is missing (tools/gen_ref_pins.py)"
    return np.load(GOLDEN)


def _compare(name, kinds, got, want):
    assert got.shape == want.shape
    bad_rows = np.zeros(got.shape[0], dtype=bool)
    for j, k in enumerate(kinds):
        if k == "u":
            bad_rows |= got[:, j] != want[:, j]
        else:
            a = got[:, j].view(np.float32).astype(np.float64)
            b = want[:, j].view(np.float32).astype(np.float64)
            both_nan = np.isnan(a) & np.isnan(b)
            same_inf = np.isinf(a) & np.isinf(b) & (np.sign(a) == np.sign(b))
            with np.errstate(invalid="ignore"):
                close = np.abs(a - b) <= RTOL * np.maximum(1.0, np.abs(b))
            bad_rows |= ~(close | both_nan | same_inf)
    return bad_rows


@pytest.mark.parametrize("name", sorted(G.PINS))
def test_oracle_matches_reference_function(golden, name):
    gens, kinds = G.PINS[name]
    inp = golden[f"{name}/in"]
    want = golden[f"{name}/out"]
    np.testing.assert_array_equal(inp, G.make_inputs(name), err_msg="fixture inputs are not the seeded ones")
    buf, cnt = None, 0
    if name == "sample_alias_table":
        buf = G.alias_buffer(golden["create_alias_table/prob"], golden["create_alias_table/alias"])
        cnt = buf.shape[0]
    got = O.unit(name, inp, len(kinds), buf, cnt)
    bad = _compare(name, kinds, got, want)
    integer_only = set(kinds) == {"u"}
    limit = 0 if integer_only else int(MAX_OUTLIER_SHARE * len(bad))
    if bad.sum() > limit:
        i = int(np.flatnonzero(bad)[0])
        pytest.fail(f"{name}: {int(bad.sum())}/{len(bad)} cases differ from the reference; first: in={inp[i].view(np.float32)} "
                    f"oracle={got[i].view(np.float32)} reference={want[i].view(np.float32)}")


def test_host_alias_table_matches_reference(golden):
    """create_alias_table (src/util/sampling.cpp:38-87) — the host library's table builder against the reference's."""
    import ctypes

    from luisarender_b200 import _ffi as F

    host = F.host_lib()
    values = golden["create_alias_table/values"]
    n = len(values)
    prob = np.zeros(n, dtype=np.float32)
    alias = np.zeros(n, dtype=np.uint32)
    pdf = np.zeros(n, dtype=np.float32)
    host.lrh_create_alias_table.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    assert host.lrh_create_alias_table(values.ctypes.data, n, prob.ctypes.data, alias.ctypes.data, pdf.ctypes.data) == 0
    np.testing.assert_array_equal(alias, golden["create_alias_table/alias"])
    np.testing.assert_array_equal(prob.view(np.uint32), golden["create_alias_table/prob"].view(np.uint32))
    np.testing.assert_array_equal(pdf.view(np.uint32), golden["create_alias_table/pdf"].view(np.uint32))


@pytest.mark.skipif(not G.LIB.exists(), reason="oracle/_ref/librefpins.so not built (needs a LuisaRender source tree: oracle/ref/README.md)")
def test_fixture_is_what_the_reference_computes_now(golden):
    ref = G.RefPins()
    prob, alias, pdf = ref.create_alias_table(golden["create_alias_table/values"])
    np.testing.assert_array_equal(alias, golden["create_alias_table/alias"])
    np.testing.assert_array_equal(prob, golden["create_alias_table/prob"])
    table = G.alias_buffer(prob, alias)
    for name in sorted(G.PINS):
        buf = table if name == "sample_alias_table" else None
        out = ref.eval(name, golden[f"{name}/in"], buf, table.shape[0] if buf is not None else 0)
        np.testing.assert_array_equal(out, golden[f"{name}/out"], err_msg=name)
