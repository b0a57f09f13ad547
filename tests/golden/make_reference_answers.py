#!/usr/bin/env python
"""Store what the reference-compiled oracle answers on the seeded tables of test_oracle_kat.test_port_equals_reference_objects
and test_oracle_nullable.test_pushed_down_filters_over_nullable_columns in reference_oracle_answers.json.

Run where build() could compile oracle/_ref (it needs the reference checkout); the JSON is committed so the tests run anywhere.
"""
import datetime
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path[:0] = [os.path.dirname(TESTS), TESTS]

import _reference_answers as R  # noqa: E402
from _nullable import nullable_lineitem  # noqa: E402
from oracle import oracle as O  # noqa: E402

o = O.Oracle("reference", workers=4)
date = lambda s: (datetime.date.fromisoformat(s) - datetime.date(1970, 1, 1)).days
out = {"oracle": o.kind, "tpch": R.tpch_answers(o, R.tpch_tables()), "nullable_scans": R.nullable_scan_answers(o, nullable_lineitem()[0], date)}
assert out["oracle"] == "reference", out["oracle"]
with open(R.PATH, "w") as f:
    json.dump(out, f, separators=(",", ":"))
    f.write("\n")
print({k: (len(v) if isinstance(v, (list, dict)) else v) for k, v in out.items()})
