"""Nullable scans on the CPU side: the oracle's pushed-down filters over columns with validity bitmaps (the reference's own
Restrictions when oracle/_ref is built, Restrictions.cpp:67-162,392-405) against a numpy evaluation, and the port against the
reference-compiled build — this is what pins the NULL semantics the GPU program pipeline is then compared with."""
import datetime
import os

import numpy as np
import pytest

from oracle import oracle as O

import _reference_answers as R
from _nullable import cases, nullable_lineitem


def _np_eval(li, valid, filters, sum_column, date):
    cat = lambda k: np.concatenate([c[k] for c in li.chunks])
    lo64 = lambda a: a[:, :8].copy().view(np.int64).reshape(-1)
    vals = {}
    for k in valid:
        a = cat(k)
        vals[k] = lo64(a) if a.ndim == 2 else a.astype(np.int64)
    keep = np.ones(li.num_rows, bool)
    for c, op, v in filters:
        if op == "notnull":
            keep &= valid[c]
            continue
        if isinstance(v, str):
            v = date(v) if "-" in v else int(round(float(v) * 100))
        elif li.spec(c).phys == "decimal128":
            v *= 100
        keep &= {"<": vals[c] < v, "<=": vals[c] <= v, ">": vals[c] > v, ">=": vals[c] >= v, "=": vals[c] == v, "!=": vals[c] != v}[op]
    total = int(vals[sum_column][keep & valid[sum_column]].sum()) if sum_column else 0
    return int(keep.sum()), total


@pytest.mark.parametrize("kind", ["port", "reference"])
def test_pushed_down_filters_over_nullable_columns(kind):
    """Each flavour against numpy and against the reference-compiled build's stored answers.  Where oracle/_ref is not built,
    the "reference" case checks those stored answers against numpy."""
    li, valid = nullable_lineitem()
    date = lambda s: (datetime.date.fromisoformat(s) - datetime.date(1970, 1, 1)).days
    stored = R.stored()["nullable_scans"]
    if kind == "reference" and not os.path.exists(O.REF_LIB):
        got = stored
    else:
        got = R.nullable_scan_answers(O.Oracle(kind, workers=3), li, date)
        assert got == stored
    assert len(got) == len(cases(date)) + 1
    for (filters, _, sum_column), answer in zip(cases(date), got):
        assert tuple(answer) == _np_eval(li, valid, filters, sum_column, date), filters
    # a comparison WITHOUT its NOTNULL partner reads the cell under a NULL like any other (the reference relies on the optimizer to add it)
    assert got[-1][0] == li.num_rows
