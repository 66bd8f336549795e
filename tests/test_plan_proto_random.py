"""Randomised round trip of the protobuf plan decoder: seeded random well-typed stage plans (nested expressions of every kind
over a seven-column schema, under Filter / Projection / Aggregate / HashJoin with residual filter / Sort / Limit) were encoded
as datafusion.PhysicalPlanNode by the fixture generator (google.protobuf over the reference's .proto files;
tests/golden/make_proto_wire.py stored the bytes in tests/golden/proto_random_plans.json.gz) and are decoded by
csrc/common/plan_proto.hpp; typed(decoded) must equal typed(source), the source plan being rebuilt here from its seed."""
import base64
import gzip
import json
import os
import random

from ballista_b200 import engine
from ballista_b200 import plan as P

HERE = os.path.dirname(os.path.abspath(__file__))

SCH = [P.field("k", "i64"), P.field("g", "utf8", True), P.field("x", P.dec(15, 2), True), P.field("y", "f64", True),
       P.field("d", "date32"), P.field("b", "bool", True), P.field("n", "i32", True)]
COL = {"i64": 0, "utf8": 1, "dec": 2, "f64": 3, "date32": 4, "bool": 5, "i32": 6}
c = P.col


class Gen:
    def __init__(self, seed, shift=0):
        self.r = random.Random(seed)
        self.shift = shift          # column offset (right side of a join filter)

    def col(self, t):
        return c(COL[t] + self.shift)

    def lit(self, t):
        r = self.r
        if r.random() < 0.08:
            return P.lit_null({"dec": P.dec(15, 2)}.get(t, t))
        return {"i64": lambda: P.lit_i64(r.randrange(-10**12, 10**12)), "i32": lambda: P.lit_i32(r.randrange(-2**31, 2**31)),
                "f64": lambda: P.lit_f64(r.choice([0.0, -1.5, 3.25e10, 1e-7, 12345.678])), "dec": lambda: P.lit_dec(r.randrange(-10**14, 10**14), 15, 2),
                "utf8": lambda: P.lit_utf8(r.choice(["", "a", "BUILDING", "q\"uo\\te", "naïve ✓", "tab\tnl\n"])),
                "date32": lambda: P.lit_date(f"{r.randrange(1992, 1999)}-{r.randrange(1, 13):02d}-{r.randrange(1, 29):02d}"),
                "bool": lambda: P.lit_bool(r.random() < 0.5)}[t]()

    def expr(self, t, depth):
        r = self.r
        if depth <= 0 or r.random() < 0.25:
            return self.col(t) if r.random() < 0.6 else self.lit(t)
        d = depth - 1
        if t == "bool":
            k = r.randrange(8)
            if k == 0:
                return P.binop(r.choice(["and", "or"]), self.expr("bool", d), self.expr("bool", d))
            if k == 1:
                return P.not_(self.expr("bool", d))
            if k == 2:
                ot = r.choice(["i64", "f64", "dec", "utf8", "date32", "i32"])
                return (P.is_null if r.random() < 0.5 else P.is_not_null)(self.expr(ot, d))
            if k == 3:
                return P.in_list(self.expr("i64", d), [P.lit_i64(r.randrange(100)) for _ in range(r.randrange(1, 5))], negated=r.random() < 0.3)
            if k == 4:
                return P.like(self.col("utf8"), r.choice(["%a%", "B_ILD%", "%", "x\\%y"]), negated=r.random() < 0.3)
            ot = r.choice(["i64", "f64", "dec", "utf8", "date32"])
            return P.binop(r.choice(["=", "!=", "<", "<=", ">", ">="]), self.expr(ot, d), self.expr(ot, d))
        if t in ("i64", "f64", "dec"):
            k = r.randrange(6)
            if k == 0:
                return P.neg(self.expr(t, d))
            if k == 1:
                return P.case([[self.expr("bool", d), self.expr(t, d)] for _ in range(r.randrange(1, 3))], self.expr(t, d) if r.random() < 0.7 else None)
            if k == 2 and t == "i64":
                return P.cast(self.expr("i32", d), "i64")
            if k == 2 and t == "f64":
                return P.cast(self.expr(r.choice(["i64", "dec"]), d), "f64")
            ops = ["+", "-", "*"] + (["%", "/"] if t != "dec" else [])
            return P.binop(r.choice(ops), self.expr(t, d), self.expr(t, d))
        if t == "utf8":
            if r.random() < 0.5:
                return P.fn("substr", self.expr("utf8", d), P.lit_i64(r.randrange(1, 4)), P.lit_i64(r.randrange(1, 5)))
            return P.case([[self.expr("bool", d), self.expr("utf8", d)]], self.lit("utf8"))
        if t == "i32":
            return P.fn("date_part_year", self.expr("date32", d)) if r.random() < 0.5 else self.col("i32")
        return self.col(t)   # date32


def _plan(seed):
    g = Gen(seed)
    r = g.r
    scan = P.scan("t", SCH)
    node = P.filter_(g.expr("bool", 3), scan) if r.random() < 0.7 else scan
    shape = r.randrange(4)
    if shape == 0:
        exprs = [(g.expr(r.choice(list(COL)), 3), f"e{i}") for i in range(r.randrange(1, 6))]
        node = P.project(exprs, node)
        keys = [P.sort_key(c(i), r.random() < 0.5, r.random() < 0.5) for i in range(min(2, len(exprs)))]
        node = P.sort(keys, node, fetch=r.choice([None, 7]))
        return P.shuffle_writer(node, 1)
    if shape == 1:
        gb = [(g.expr(r.choice(["i64", "utf8", "date32"]), 1), f"k{i}") for i in range(r.randrange(0, 3))]
        aggs = [P.agg(fn, g.expr(t, 2), f"a{i}") for i, (fn, t) in enumerate(r.sample([("sum", "dec"), ("avg", "dec"), ("min", "date32"), ("max", "utf8"),
                                                                                          ("sum", "i64"), ("avg", "f64"), ("count", "i32")], r.randrange(1, 5)))]
        if r.random() < 0.5:
            aggs.append(P.agg("count", None, "cnt"))
        node = P.aggregate("Partial", gb, aggs, node)
        nk = len(gb)
        return P.shuffle_writer(node, 2, [c(i) for i in range(nk)] or None, 8 if nk else 0) if nk else P.shuffle_writer(node, 2)
    if shape == 2:
        other = P.scan("u", SCH)
        both = Gen(seed * 7 + 1)
        lf, rf = Gen(seed * 7 + 2), Gen(seed * 7 + 3, shift=len(SCH))
        filt = P.binop(r.choice(["<", ">=", "!="]), lf.expr(r.choice(["i64", "dec"]), 1), rf.expr("i64", 1)) if r.random() < 0.7 else None
        if filt is not None and r.random() < 0.5:
            filt = P.and_(filt, P.is_not_null(rf.col("utf8")), both.expr("bool", 1))
        jt = r.choice(["Inner", "Left", "Right", "Full", "LeftSemi", "LeftAnti", "RightSemi", "RightAnti"])
        j = P.hash_join(node, other, [[c(0), c(0)]] + ([[c(4), c(4)]] if r.random() < 0.3 else []), jt, "Partitioned", filter=filt,
                        projection=[0, 3, 8, 9] if jt in ("Inner", "Left", "Right", "Full") and r.random() < 0.5 else None)
        return P.shuffle_writer(P.limit(j, 100, global_=r.random() < 0.5), 3, [c(0)], 4)
    node = P.sort_preserving_merge([P.sort_key(g.expr("dec", 2), False)], P.coalesce_batches(node), fetch=r.choice([None, 3]))
    return P.shuffle_writer(node, 4, [g.expr("i64", 2), c(1)], 16, sort_shuffle=False)


def _strip(t):
    if isinstance(t, dict):
        return {k: _strip(v) for k, v in t.items() if not (k == "name" and "col" in t)}
    if isinstance(t, list):
        return [_strip(v) for v in t]
    return t


def test_random_plans_round_trip():
    with gzip.open(os.path.join(HERE, "golden", "proto_random_plans.json.gz"), "rt") as fh:
        fix = json.load(fh)
    assert fix["seeds"] == 600
    ok = rejected = 0
    for seed in range(600):
        ir = json.dumps(_plan(seed), separators=(",", ":"))
        try:
            want = json.loads(engine.plan_typed_json(ir))
        except engine.B200Error:
            rejected += 1          # an ill-typed combination (e.g. decimal precision overflow): not a plan
            assert str(seed) not in fix["plans"], f"seed {seed}"
            continue
        proto = base64.b64decode(fix["plans"][str(seed)])
        got = json.loads(engine.plan_typed_json(engine.plan_proto_to_json(proto)))
        assert _strip(got) == _strip(want), f"seed {seed}"
        ok += 1
    assert ok >= 300, (ok, rejected)
