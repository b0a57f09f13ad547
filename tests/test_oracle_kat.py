"""Pins the CPU oracle against the reference's OWN known-answer vectors (tests/golden/reference_kats.json,
extracted from /root/reference by tests/golden/make_golden.py) and cross-checks its two flavours."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from lingodb_b200 import datagen
from oracle import oracle as O

import _reference_answers as R

GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_kats.json")))
M64 = 2**64


def flavours():
    kinds = ["port"]
    if os.path.exists(O.REF_LIB):
        kinds.append("reference")
    return kinds


@pytest.fixture(scope="module", params=flavours())
def orc(request):
    return O.Oracle(request.param, workers=3)


def test_hash_kats_from_hash_mlir(orc):
    L, h = orc.lib, GOLD["hash"]
    assert L.oracle_hash_i64(10) == h["i32_10"] == h["i64_10"]
    assert L.oracle_hash_bool(1) == h["bool_true"]
    assert L.oracle_hash_i128(10001, 0) == h["decimal15_2_100.01"]  # decimal<15,2> 100.01 is hashed as i128: high, then low
    days = L.oracle_parse_date(b"2020-06-11")
    assert days == 18424
    assert L.oracle_hash_date_days(days) == h["date_2020-06-11"]  # dates are hashed as i64 nanoseconds
    secs = days * 86400 + 12 * 3600 + 30 * 60
    assert L.oracle_hash_i64(secs) == h["timestamp_s_2020-06-11_12:30:00"]
    assert L.oracle_hash_string(b"hello world!", 12) == h["string_hello_world!"]
    assert L.oracle_hash_i64(1) == h["int8_1"] % M64  # TestStorage.cpp:289,411


def test_hash_tuple_combine_order(orc):
    """7-tuple of hash.mlir: pins combine(new, total) = new ^ bswap(total) and the i128 high-then-low order."""
    L = orc.lib
    days = L.oracle_parse_date(b"2020-06-11")
    pieces = [L.oracle_hash_i64(10), L.oracle_hash_i64(10), L.oracle_hash_i64(-1), L.oracle_hash_i64(0), L.oracle_hash_i64(10001),
              L.oracle_hash_i64(days * 86400000000000), L.oracle_hash_i64(days * 86400 + 45000), L.oracle_hash_string(b"hello world!", 12)]
    total = pieces[0]
    for p in pieces[1:]:
        total = L.oracle_hash_combine(p, total)
    assert total == GOLD["hash"]["tuple7"]


def test_xxh64_known_answers(orc):
    # published XXH64 vectors (seed 0): llvm::xxHash64 is used for strings longer than 12 bytes (Hash.cpp:13-16)
    L = orc.lib
    assert L.oracle_xxh64(b"", 0) == 0xEF46DB3751D8E999
    assert L.oracle_xxh64(b"a", 1) == 0xD24EC4F1A98C6E5B
    assert L.oracle_xxh64(b"abc", 3) == 0x44BC2CF5AD770999
    s = b"Nobody inspects the spammish repetition"
    assert L.oracle_xxh64(s, len(s)) == 0xFBCEA83C8A378BF1
    assert L.oracle_hash_string(s, len(s)) == 0xFBCEA83C8A378BF1  # len > 12 → xxHash64 of the bytes


def _dec(s, scale):
    neg = s.startswith("-")
    ip, _, fp = s.lstrip("-").partition(".")
    v = int(ip + fp.ljust(scale, "0")[:scale])
    return -v if neg else v


def test_q1_avg_formula_against_tpch_sf1_answers(orc):
    """avg(decimal(12,2)) = (sum * 10^19) sdiv count, decimal(31,21) — reproduces tpchSf1.test:25-28 digit for digit."""
    L = orc.lib
    for row in GOLD["tpch_sf1"]["q1"]:
        cnt = int(row["count_order"])
        lo, hi = C.c_int64(), C.c_int64()
        for sum_col, avg_col in (("sum_qty", "avg_qty"), ("sum_base_price", "avg_price")):
            L.oracle_avg_dec12_2(_dec(row[sum_col], 2), cnt, C.byref(lo), C.byref(hi))
            assert O.i128((lo.value, hi.value)) == _dec(row[avg_col], 21), (row, avg_col)
        # sum(l_discount) is not printed: the avg must be consistent with SOME integer sum (unique within +-1)
        want = _dec(row["avg_disc"], 21)
        s = (want * cnt) // 10**19
        found = False
        for cand in (s, s + 1):
            L.oracle_avg_dec12_2(cand, cnt, C.byref(lo), C.byref(hi))
            found |= O.i128((lo.value, hi.value)) == want
        assert found


def test_decimal_multiplication_semantics(orc):
    # scales add, no rescale: 1478493 rows' sum_charge has 6 fraction digits, sum_disc_price 4 (tpchSf1.test:25)
    row = GOLD["tpch_sf1"]["q1"][0]
    assert len(row["sum_charge"].split(".")[1]) == 6 and len(row["sum_disc_price"].split(".")[1]) == 4
    L = orc.lib
    lo, hi = C.c_int64(), C.c_int64()
    L.oracle_mul_i128(-5, -1, 7, 0, C.byref(lo), C.byref(hi))
    assert O.i128((lo.value, hi.value)) == -35
    L.oracle_mul_i128(2**62, 0, 8, 0, C.byref(lo), C.byref(hi))
    assert O.i128((lo.value, hi.value)) == 2**65
    L.oracle_parse_decimal(b"0.05", 2, C.byref(lo), C.byref(hi))
    assert lo.value == 5
    L.oracle_parse_decimal(b"-12.3", 2, C.byref(lo), C.byref(hi))
    assert O.i128((lo.value, hi.value)) == -1230


# ---------------------------------------------------------------- independent evaluation of the SQL in numpy
def _cols(t, names):
    out = {}
    for n in names:
        spec = t.spec(n)
        parts = [c[n] for c in t.chunks]
        if spec.phys == "decimal128":
            out[n] = np.concatenate([p[:, :8].copy().view(np.int64).reshape(-1) for p in parts]) if parts else np.zeros(0, np.int64)
        else:
            out[n] = np.concatenate(parts) if parts else np.zeros(0, np.int32)
    return out


@pytest.fixture(scope="module")
def tables():
    return R.tpch_tables()


def test_q6_and_q1_match_numpy(orc, tables):
    li = tables["lineitem"]
    c = _cols(li, ["l_shipdate", "l_discount", "l_quantity", "l_extendedprice", "l_tax", "l_returnflag", "l_linestatus"])
    h = orc.table(li)
    d0, d1 = orc.lib.oracle_parse_date(b"1994-01-01"), orc.lib.oracle_parse_date(b"1995-01-01")
    m = (c["l_shipdate"] >= d0) & (c["l_shipdate"] < d1) & (c["l_discount"] >= 5) & (c["l_discount"] <= 7) & (c["l_quantity"] < 2400)
    want = sum(int(a) * int(b) for a, b in zip(c["l_extendedprice"][m], c["l_discount"][m]))
    assert orc.q6(h)[0] == {"revenue": want}
    cut = orc.lib.oracle_parse_date(b"1998-09-02")
    rows, _ = orc.q1(h)
    m = c["l_shipdate"] <= cut
    keys = sorted(set(zip(c["l_returnflag"][m].tolist(), c["l_linestatus"][m].tolist())))
    assert [(r["l_returnflag"], r["l_linestatus"]) for r in rows] == keys
    for r in rows:
        g = m & (c["l_returnflag"] == r["l_returnflag"]) & (c["l_linestatus"] == r["l_linestatus"])
        ext, disc, tax, qty = (c[k][g].astype(object) for k in ("l_extendedprice", "l_discount", "l_tax", "l_quantity"))
        assert r["count_order"] == int(g.sum())
        assert r["sum_qty"] == int(qty.sum()) and r["sum_base_price"] == int(ext.sum())
        assert r["sum_disc_price"] == int((ext * (100 - disc)).sum())
        assert r["sum_charge"] == int((ext * (100 - disc) * (100 + tax)).sum())
        assert r["avg_qty"] == int(qty.sum()) * 10**19 // r["count_order"]
        assert r["avg_disc"] == int(disc.sum()) * 10**19 // r["count_order"]


def test_q3_and_q5_match_python(orc, tables):
    li = _cols(tables["lineitem"], ["l_orderkey", "l_suppkey", "l_extendedprice", "l_discount", "l_shipdate"])
    od = _cols(tables["orders"], ["o_orderkey", "o_custkey", "o_orderdate", "o_shippriority"])
    cu = _cols(tables["customer"], ["c_custkey", "c_nationkey"])
    su = _cols(tables["supplier"], ["s_suppkey", "s_nationkey"])
    seg = []
    for ch in tables["customer"].chunks:
        offs, data = ch["c_mktsegment"]
        b = bytes(data)
        seg += [b[offs[i]:offs[i + 1]].decode() for i in range(len(offs) - 1)]
    h = {k: orc.table(v) for k, v in tables.items()}
    # Q3
    d = orc.lib.oracle_parse_date(b"1995-03-15")
    building = {int(k) for k, s in zip(cu["c_custkey"], seg) if s == "BUILDING"}
    orders = {int(k): (int(dt), int(sp)) for k, ck, dt, sp in zip(od["o_orderkey"], od["o_custkey"], od["o_orderdate"], od["o_shippriority"]) if dt < d and int(ck) in building}
    rev = {}
    for k, e, dc, sd in zip(li["l_orderkey"], li["l_extendedprice"], li["l_discount"], li["l_shipdate"]):
        if sd > d and int(k) in orders:
            rev[int(k)] = rev.get(int(k), 0) + int(e) * (100 - int(dc))
    want = sorted(({"l_orderkey": k, "revenue": v, "o_orderdate": orders[k][0], "o_shippriority": orders[k][1]} for k, v in rev.items()),
                  key=lambda r: (-r["revenue"], r["o_orderdate"], r["l_orderkey"]))[:10]
    assert orc.q3(h["customer"], h["orders"], h["lineitem"])[0] == want
    # Q5
    asia = {i for i, (_, r) in enumerate(datagen.NATIONS) if datagen.REGIONS[r] == "ASIA"}
    cust = {int(k): int(n) for k, n in zip(cu["c_custkey"], cu["c_nationkey"]) if int(n) in asia}
    supp = {int(k): int(n) for k, n in zip(su["s_suppkey"], su["s_nationkey"]) if int(n) in asia}
    d0, d1 = orc.lib.oracle_parse_date(b"1994-01-01"), orc.lib.oracle_parse_date(b"1995-01-01")
    onat = {int(k): cust[int(ck)] for k, ck, dt in zip(od["o_orderkey"], od["o_custkey"], od["o_orderdate"]) if d0 <= dt < d1 and int(ck) in cust}
    rev = {}
    for k, sk, e, dc in zip(li["l_orderkey"], li["l_suppkey"], li["l_extendedprice"], li["l_discount"]):
        n = onat.get(int(k))
        if n is not None and supp.get(int(sk)) == n:
            rev[n] = rev.get(n, 0) + int(e) * (100 - int(dc))
    want = sorted(({"n_name": datagen.NATIONS[n][0], "revenue": v} for n, v in rev.items()), key=lambda r: (-r["revenue"], r["n_name"]))
    assert orc.q5(h["customer"], h["orders"], h["lineitem"], h["supplier"], h["nation"], h["region"])[0] == want


def test_port_equals_reference_objects(tables):
    """The port answers as the reference's own runtime objects do: against their stored answers always, and against the
    reference-compiled build itself where oracle/_ref is built."""
    want = R.stored()["tpch"]
    assert len(want["q9"]) > 150
    for kind in (["port", "reference"] if os.path.exists(O.REF_LIB) else ["port"]):
        got = R.tpch_answers(O.Oracle(kind, workers=4), tables)
        for q in ("q6", "q1", "q3", "q5", "q9"):
            assert got[q] == want[q], (kind, q)


def test_oracle_edge_cases(orc):
    s = datagen.scale(0.001, seed=1)
    empty = datagen.lineitem(s, n_rows=0)
    h = orc.table(empty)
    assert orc.q1(h)[0] == []
    assert orc.q6(h)[0] == {"revenue": 0}
    ragged = datagen.lineitem(s, chunk_rows=777)  # ragged batches, last one short
    whole = datagen.lineitem(s, chunk_rows=1 << 20)
    assert orc.q1(orc.table(ragged))[0] == orc.q1(orc.table(whole))[0]
    with pytest.raises(RuntimeError):
        orc.q6(orc.table(whole), date_ge="garbage")


# ---------------------------------------------------------------- Q9 (scalar runtime + pipeline)
def test_extract_year_and_const_like(orc):
    import datetime
    L, d = orc.lib, GOLD["dates"]
    days = L.oracle_parse_date(d["date"].encode())
    assert L.oracle_extract_year(days * 86400 * 10**9) == d["extract_year"]  # test/lit/DB/dates.mlir:23-26
    for days in (-366, -365, -1, 0, 58, 59, 60, 364, 365, 789, 8035, 10440, 10591, 10592, 11016, 11017, 19000, 47482, -25567):
        want = (datetime.date(1970, 1, 1) + datetime.timedelta(days=days)).year
        assert L.oracle_extract_year(days * 86400 * 10**9) == want, days
        assert L.oracle_extract_year(days * 86400 * 10**9 + 86399 * 10**9) == want, days  # floor<days> of a timestamp inside the day
    for s, needle, want in ((b"forest green navy", b"green", 1), (b"greengreen", b"green", 1), (b"gree n", b"green", 0), (b"", b"green", 0),
                            (b"a long string of more than twelve bytes ending in gree", b"green", 0), (b"xgreen", b"green", 1), (b"abc", b"", 1)):
        assert L.oracle_const_like_contains(s, len(s), needle) == want, s


def test_q9_matches_python(orc):
    import datetime
    t = datagen.tpch(0.02, seed=13, chunk_rows=4000, with_parts=True)
    li = _cols(t["lineitem"], ["l_orderkey", "l_partkey", "l_suppkey", "l_quantity", "l_extendedprice", "l_discount"])
    od = _cols(t["orders"], ["o_orderkey", "o_orderdate"])
    su = _cols(t["supplier"], ["s_suppkey", "s_nationkey"])
    ps = _cols(t["partsupp"], ["ps_partkey", "ps_suppkey", "ps_supplycost"])
    pk = _cols(t["part"], ["p_partkey"])["p_partkey"]
    names = []
    for ch in t["part"].chunks:
        offs, data = ch["p_name"]
        b = bytes(data)
        names += [b[offs[i]:offs[i + 1]].decode() for i in range(len(offs) - 1)]
    h = {k: orc.table(v) for k, v in t.items()}
    for needle in ("green", "y"):
        parts = {int(k) for k, n in zip(pk, names) if needle in n}
        cost = {}
        for a, b, c in zip(ps["ps_partkey"], ps["ps_suppkey"], ps["ps_supplycost"]):
            if int(a) in parts:
                cost.setdefault((int(a), int(b)), []).append(int(c))
        nat = {int(k): int(n) for k, n in zip(su["s_suppkey"], su["s_nationkey"])}
        year = {int(k): (datetime.date(1970, 1, 1) + datetime.timedelta(days=int(d))).year for k, d in zip(od["o_orderkey"], od["o_orderdate"])}
        acc = {}
        for ok, p, s, q, e, dc in zip(li["l_orderkey"], li["l_partkey"], li["l_suppkey"], li["l_quantity"], li["l_extendedprice"], li["l_discount"]):
            for c in cost.get((int(p), int(s)), ()):
                key = (datagen.NATIONS[nat[int(s)]][0], year[int(ok)])
                acc[key] = acc.get(key, 0) + int(e) * (100 - int(dc)) - c * int(q)
        want = [{"nation": n, "o_year": y, "sum_profit": v} for (n, y), v in sorted(acc.items(), key=lambda kv: (kv[0][0], -kv[0][1]))]
        got, _ = orc.q9(h["part"], h["supplier"], h["lineitem"], h["partsupp"], h["orders"], h["nation"], needle)
        assert got == want, needle
    # the result's key set is the one the reference's own Q9 answer has (tpchSf1.test:20632-20807): 25 nations x 1992..1998
    got, _ = orc.q9(h["part"], h["supplier"], h["lineitem"], h["partsupp"], h["orders"], h["nation"])
    assert [[r["nation"], r["o_year"]] for r in got] == GOLD["tpch_sf1"]["q9_keys"]
