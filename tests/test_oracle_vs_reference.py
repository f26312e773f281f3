"""Pins the oracle (oracle/calculators.py) and the plan compiler's column names against the UNMODIFIED reference.

The reference's answers are stored in tests/golden/reference.npz and tests/golden/reference.json (written by
`python -m oracle.make_golden_reference`, which needs the reference tree); the inputs are regenerated here from the
same seeds."""
import ast
import builtins
import json
import os
import warnings

import numpy as np
import pandas as pd
import pytest

from oracle.extract import compare, oracle_rows
from oracle.make_golden_reference import (FRAME_CASES, IMPUTE_CASES, ROLL_CASES, ROLLING_TESTS, TIMEWISE_LENGTHS,
                                          from_columns_input, impute_input, normalise_kind_to_fc, roll_frame,
                                          short_series, timewise_series)
from tests.helpers import synthetic_series
from tsfresh_b200.plan import Plan
from tsfresh_b200.settings import ComprehensiveFCParameters, EfficientFCParameters, MinimalFCParameters

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def npz():
    with np.load(os.path.join(GOLDEN, "reference.npz"), allow_pickle=False) as z:
        return dict(z)


@pytest.fixture(scope="module")
def js():
    with open(os.path.join(GOLDEN, "reference.json")) as f:
        return json.load(f)


def test_settings_match_reference(js):
    for mine, name in ((ComprehensiveFCParameters(), "comprehensive"), (EfficientFCParameters(), "efficient"),
                       (MinimalFCParameters(), "minimal")):
        theirs = {k: ast.literal_eval(v) for k, v in js["settings"][name]}
        assert list(mine.keys()) == list(theirs.keys())
        for k in mine:
            assert mine[k] == theirs[k], k


@pytest.mark.parametrize("kind,length,count", FRAME_CASES)
def test_oracle_matches_reference(npz, kind, length, count):
    series = list(synthetic_series(11, count, length, kind))
    settings = ComprehensiveFCParameters()
    key = "frame_%s_%d_%d" % (kind, length, count)
    plan = Plan(settings)
    assert ["value__" + s for s in plan.suffixes] == list(npz[key + "_columns"])
    mine = oracle_rows([s.astype(np.float64) for s in series], settings)
    bad = compare(mine, npz[key], plan.suffixes, rtol=1e-12)
    assert not bad, bad[:20]


def test_oracle_matches_reference_short_series(npz):
    series = short_series()
    settings = ComprehensiveFCParameters()
    plan = Plan(settings)
    mine = oracle_rows([s.astype(np.float64) for s in series], settings)
    bad = compare(mine, npz["frame_short"], plan.suffixes, rtol=1e-12)
    assert not bad, bad[:20]


def test_oracle_impute_matches_reference(npz):
    """oracle/impute.py against tsfresh.utilities.dataframe_functions (:49-212) on random matrices."""
    from oracle import impute as oi
    for seed, rows, cols in IMPUTE_CASES:
        m = impute_input(seed, rows, cols)
        st = oi.range_values(m)
        want = npz["impute%d_range" % seed]
        assert np.array_equal(st[0], want[0])
        assert np.array_equal(st[1], want[1])
        assert np.array_equal(st[2], want[2])
        assert np.array_equal(oi.impute(m), npz["impute%d" % seed])
        assert np.array_equal(oi.impute_zero(m), npz["impute%d_zero" % seed])


def test_roll_time_series_views_reproduce_reference_frame(npz):
    """tsfresh_b200.roll_time_series(...).to_frame() == the reference's materialised rolled frame (ids, row order,
    values) for both directions, shuffled input and a missing sort column."""
    from tsfresh_b200 import roll_time_series
    df = roll_frame()
    for shuffle in (False, True):
        d = df.sample(frac=1.0, random_state=1).reset_index(drop=True) if shuffle else df
        for k, (rd, mx, mn) in enumerate(ROLL_CASES):
            key = "roll%d_%d" % (int(shuffle), k)
            got = roll_time_series(d, column_id="id", column_sort="time", rolling_direction=rd, max_timeshift=mx,
                                   min_timeshift=mn).to_frame()
            assert [tuple(i) for i in npz[key + "_id"].tolist()] == list(got["id"]), (shuffle, rd, mx, mn)
            assert np.array_equal(npz[key + "_time"], got["time"])
            for c in "ab":
                assert np.array_equal(npz[key + "_" + c], got[c])
    d = df.drop(columns=["time"])
    got = roll_time_series(d, column_id="id", rolling_direction=2, max_timeshift=5).to_frame()
    assert [tuple(i) for i in npz["roll_nosort_id"].tolist()] == list(got["id"])
    assert np.array_equal(npz["roll_nosort_sort"], got["sort"].to_numpy())


def _frame(cols):
    return pd.DataFrame({c["name"]: pd.Series(c["values"], dtype=c["dtype"]) for c in cols})


def _assert_frame_matches(got, want_cols, column_id, where):
    for c in want_cols:
        if c["name"] == column_id != "id":
            continue            # the reference keeps the parent id column; here it is the first element of the "id" pairs
        assert c["name"] in got.columns, (where, c["name"])
        g = list(got[c["name"]])
        if c["tuples"]:
            assert g == [tuple(v) for v in c["values"]], (where, c["name"])
        elif pd.api.types.is_numeric_dtype(c["dtype"]):
            assert np.array_equal(np.asarray(g, np.float64), np.asarray(c["values"], np.float64), equal_nan=True), \
                (where, c["name"])
        else:
            assert g == c["values"], (where, c["name"])


def test_reference_rolling_test_cases_pass_on_the_view_implementation(js):
    """Every roll_time_series call of the reference's own RollingTestCase (tests/units/utilities/
    test_dataframe_functions.py:18-944) replayed on tsfresh_b200.roll_time_series(...).to_frame(): positive / negative /
    larger-shift / stacked (kind column) / dict / order / warning / validation cases give the frames, exception types
    and warnings the reference gave."""
    from tsfresh_b200 import roll_time_series as mine
    cases = js["rolling_test_case"]
    assert [c["test"] for c in cases] == ROLLING_TESTS
    for case in cases:
        assert case["calls"], case["test"]
        for n, call in enumerate(case["calls"]):
            where = (case["test"], n)
            data = ({k: _frame(v) for k, v in call["input"].items()} if call["input_is_dict"] else _frame(call["input"]))
            if "raises" in call:
                with pytest.raises(getattr(builtins, call["raises"])):
                    mine(data, show_warnings=True, **call["kwargs"])
                continue
            with warnings.catch_warnings(record=True) as caught:
                warnings.simplefilter("always")
                r = mine(data, show_warnings=True, **call["kwargs"])
            messages = {str(w.message) for w in caught}
            for m in call["warnings"]:
                assert m in messages, (where, m)
            if call["input_is_dict"]:
                assert isinstance(r, dict) and sorted(r) == sorted(call["output"]), where
                for k, want in call["output"].items():
                    _assert_frame_matches(r[k].to_frame(), want, call["kwargs"]["column_id"], where + (k,))
            else:
                _assert_frame_matches(r.to_frame(), call["output"], call["kwargs"]["column_id"], where)


def test_from_columns_matches_reference(js):
    """settings.from_columns (settings.py:23-83): same kind_to_fc_parameters and same errors as the reference."""
    from tsfresh_b200.settings import from_columns
    ref = js["from_columns"]
    mine = from_columns(from_columns_input() + ["skipme"], columns_to_ignore=["skipme"])
    assert normalise_kind_to_fc(mine) == ast.literal_eval(ref["parsed"]) and list(mine) == ref["kinds"]
    expected = [(["nounderscore"], ValueError), ([3], TypeError), (["value__not_a_calculator"], ValueError)]
    assert [[bad, err.__name__] for bad, err in expected] == ref["errors"]
    for bad, err in expected:
        with pytest.raises(err):
            from_columns(bad)


def test_linear_trend_timewise_matches_reference(npz):
    """feature_calculators.py:2274-2306 with its own known answers (test_feature_calculations.py:1796-1935) and on
    irregularly sampled random series"""
    from oracle import calculators as C
    param = [{"attr": a} for a in ("pvalue", "rvalue", "intercept", "slope", "stderr")]
    x = pd.Series([0, 1, 3, 6], index=pd.DatetimeIndex(["2018-01-01 04:00:00", "2018-01-01 05:00:00", "2018-01-01 07:00:00",
                                                         "2018-01-01 10:00:00"]))
    got = C.linear_trend_timewise(x.to_numpy(), x.index.as_unit("ns").asi8, param)
    assert got[3] == pytest.approx(1.0, abs=1e-3) and got[2] == pytest.approx(0.0, abs=1e-3)
    rng = np.random.default_rng(12)
    for n in TIMEWISE_LENGTHS:
        s = timewise_series(rng, n)
        got = C.linear_trend_timewise(s.to_numpy(), s.index.asi8, param)
        np.testing.assert_allclose(got, npz["timewise%d" % n], rtol=1e-12, equal_nan=True)
