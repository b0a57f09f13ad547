"""What the reference-compiled oracle (oracle/_ref: the reference's own runtime objects) answers on seeded tables.
golden/make_reference_answers.py stores these answers in golden/reference_oracle_answers.json, so the tests hold the port to
them also where oracle/_ref cannot be built."""
import json
import os

from lingodb_b200 import datagen

from _nullable import cases

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_oracle_answers.json")


def stored():
    with open(PATH) as f:
        return json.load(f)


def tpch_tables():
    return datagen.tpch(0.03, seed=9, chunk_rows=5000)


def tpch_answers(o, tables):
    """Q6 / Q1 / Q3 / Q5 on `tables` and Q9 on a second seeded set, as the JSON-able rows the oracle returns."""
    h = {k: o.table(v) for k, v in tables.items()}
    out = {"q6": o.q6(h["lineitem"])[0], "q1": o.q1(h["lineitem"])[0], "q3": o.q3(h["customer"], h["orders"], h["lineitem"])[0],
           "q5": o.q5(h["customer"], h["orders"], h["lineitem"], h["supplier"], h["nation"], h["region"])[0]}
    t9 = datagen.tpch(0.02, seed=4, chunk_rows=3000, with_parts=True)
    h = {k: o.table(v) for k, v in t9.items()}
    out["q9"] = o.q9(h["part"], h["supplier"], h["lineitem"], h["partsupp"], h["orders"], h["nation"])[0]
    return out


def nullable_scan_answers(o, li, date):
    """[count, sum] of every nullable case's pushed-down filters, then of one comparison without its NOTNULL partner."""
    h = o.table(li)
    out = [list(o.scan_count_sum(h, filters, sum_column)) for filters, _, sum_column in cases(date)]
    out.append(list(o.scan_count_sum(h, [("l_suppkey", ">=", 0)], None)))
    o.free(h)
    return out
