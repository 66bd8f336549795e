"""The protobuf plan decoder (csrc/common/plan_proto.hpp, C-ABI b200_plan_proto_to_json / b200_stage_prepare_proto): a Ballista
task's plan bytes -> the stage-plan IR.  Host-only code: runs without a GPU.

Fixtures: tests/golden/proto_plans.json -- every stage of the 22 TPC-H queries plus shapes they do not contain, serialised as
datafusion.PhysicalPlanNode by google.protobuf with message classes built from the REFERENCE's .proto files
(tests/golden/make_proto_plans.py; ballista/core/proto/*.proto).  Check: the typed plan (b200_plan_typed_json: resolved
column indices, expression / aggregate types, every node's output schema) of the decoded IR equals the typed plan of the IR the
bytes were generated from; the fixture bytes must also be, field for field, what google.protobuf read in them with the
reference's message definitions (tests/golden/proto_plans_wire.json.gz)."""
import base64
import gzip
import json
import os

import pytest

from ballista_b200 import engine

HERE = os.path.dirname(os.path.abspath(__file__))
with open(os.path.join(HERE, "golden", "proto_plans.json")) as fh:
    FIX = json.load(fh)
CASES = FIX["cases"]


def _strip_cosmetic(t):
    """Column display names inside expressions are cosmetic (PhysicalColumn.name); everything else must match."""
    if isinstance(t, dict):
        return {k: _strip_cosmetic(v) for k, v in t.items() if not (k == "name" and "col" in t)}
    if isinstance(t, list):
        return [_strip_cosmetic(v) for v in t]
    return t


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_decoded_plan_equals_source_plan(case):
    proto = base64.b64decode(case["proto_b64"])
    got_ir = engine.plan_proto_to_json(proto)
    got = json.loads(engine.plan_typed_json(got_ir))
    want = json.loads(engine.plan_typed_json(case["ir"]))
    assert _strip_cosmetic(got) == _strip_cosmetic(want)


def test_all_tpch_stages_are_covered():
    names = {c["name"].split("/")[0] for c in CASES}
    assert {f"q{i}" for i in range(1, 23)} <= names
    assert len(CASES) >= 150


def test_job_id_override_and_scan_files():
    case = [c for c in CASES if c["name"] == "q5/stage5"][0]
    ir = json.loads(engine.plan_proto_to_json(base64.b64decode(case["proto_b64"]), job_id="job-42"))
    assert ir["op"] == "SortShuffleWriterExec" and ir["job_id"] == "job-42" and ir["stage_id"] == 5
    scan = ir["input"]
    assert scan["op"] == "DataSourceExec" and scan["table"] == "lineitem"
    assert scan["file_groups"] == [["/data/tpch/lineitem/part-0.parquet"]]


def test_malformed_and_unsupported_inputs():
    with pytest.raises(engine.B200Error) as e:
        engine.plan_proto_to_json(b"\x0a\xff\xff\xff\xff\x0f")      # length runs past the end
    assert e.value.code == -1
    with pytest.raises(engine.B200Error) as e:
        engine.plan_proto_to_json(b"")                                # no PhysicalPlanType
    assert e.value.code == -1
    # a node the device engine does not implement is named, not guessed at: CrossJoinExecNode = field 16
    with pytest.raises(engine.B200Error) as e:
        engine.plan_proto_to_json(bytes([0x82, 0x01, 0x00]))                 # key = 16 << 3 | 2 as a varint, empty body
    assert e.value.code == -2 and "16" in str(e.value)
    # unknown fields are skipped (forward compatibility): an unknown varint field 99 appended to the root message
    case = [c for c in CASES if c["name"] == "q1/stage1"][0]
    proto = base64.b64decode(case["proto_b64"])
    assert engine.plan_proto_to_json(proto + bytes([0x98, 0x06, 0x2a])) == engine.plan_proto_to_json(proto)


def _read_varint(buf, i):
    v = shift = 0
    while True:
        b = buf[i]
        i += 1
        v |= (b & 0x7f) << shift
        shift += 7
        if not b & 0x80:
            return v, i


def wire_fields(buf):
    """[(field number, wire type, value)] of one protobuf message, schema-less: varints and fixed-width values as unsigned
    ints, length-delimited values as bytes."""
    out, i = [], 0
    while i < len(buf):
        key, i = _read_varint(buf, i)
        num, wt = key >> 3, key & 7
        if wt == 0:
            v, i = _read_varint(buf, i)
        elif wt in (1, 5):
            n = 8 if wt == 1 else 4
            v, i = int.from_bytes(buf[i:i + n], "little"), i + n
        elif wt == 2:
            n, i = _read_varint(buf, i)
            v, i = bytes(buf[i:i + n]), i + n
        else:
            raise ValueError(f"wire type {wt}")
        out.append((num, wt, v))
    assert i == len(buf)
    return out


def _matches_tree(buf, tree):
    fields = wire_fields(buf)
    assert [(n, wt) for n, wt, _ in fields] == [(t[0], t[2]) for t in tree]
    for (_, wt, v), (_, _, _, want) in zip(fields, tree):
        if isinstance(want, list):
            _matches_tree(v, want)
        elif wt == 2:
            assert base64.b64encode(v).decode() == want
        else:
            assert v == want


def test_fixture_is_what_the_reference_protos_describe():
    """Every fixture is, field for field, the datafusion.PhysicalPlanNode google.protobuf parsed from it with the reference's
    message definitions (tests/golden/proto_plans_wire.json.gz, made by tests/golden/make_proto_wire.py, which also checked that
    each parse had no unknown field and re-serialised byte-identically)."""
    with gzip.open(os.path.join(HERE, "golden", "proto_plans_wire.json.gz"), "rt") as fh:
        wire = json.load(fh)["cases"]
    assert sorted(wire) == sorted(c["name"] for c in CASES)
    for c in CASES:
        tree = wire[c["name"]]
        _matches_tree(base64.b64decode(c["proto_b64"]), tree)
        assert [f[1] for f in tree] == ["extension"]                  # every stage is rooted at a Ballista shuffle writer
        ext = tree[0][3]
        node = [f[3] for f in ext if f[1] == "node"]
        assert len(node) == 1 and [f[1] for f in node[0]] in (["shuffle_writer"], ["sort_shuffle_writer"])
        assert sum(f[1] == "inputs" for f in ext) == 1


class _DecodedPlans:
    """The oracle engine fed with IR decoded from the protobuf fixtures instead of the IR text the driver passes."""

    def __init__(self, eng, query):
        self._e, self._q = eng, query

    def __getattr__(self, name):
        return getattr(self._e, name)

    def create_query_stage_exec(self, job_id, stage_id, plan_json):
        proto = base64.b64decode([c for c in CASES if c["name"] == f"{self._q}/stage{stage_id}"][0]["proto_b64"])
        return self._e.create_query_stage_exec(job_id, stage_id, engine.plan_proto_to_json(proto, job_id=job_id))


@pytest.mark.parametrize("q", [f"q{i}" for i in range(1, 23)])
def test_decoded_plans_execute_like_their_source(oracle, oracle_lib, q):
    """End to end on the CPU oracle (same plan front end as the device engine): a query whose every stage is decoded from plan
    bytes returns the table the IR text returns -- join filters through column_indices, Final aggregates typed from
    input_schema, scans named after their files."""
    from ballista_b200 import driver, tpch
    from test_tpch_queries import load_tables
    from util import assert_tables_equal
    load_tables(oracle, oracle_lib, 20, tpch.union_tables([q]), 2)
    stages = tpch.QUERIES[q][1](4)
    want = driver.run_stages(oracle, stages, f"{q}-ir")
    got = driver.run_stages(_DecodedPlans(oracle, q), stages, f"{q}-pb")
    assert (want is None) == (got is None)
    if want is not None:
        assert_tables_equal(got, want, sort=False)


def test_task_definitions_decode():
    """TaskDefinition / MultiTaskDefinition bytes (what LaunchTask / LaunchMultiTask / PollWork deliver): identities, props."""
    t = FIX["tasks"]
    assert engine.task_definition_decode(base64.b64decode(t["single_b64"]), multi=False) == t["single"]
    assert engine.task_definition_decode(base64.b64decode(t["multi_b64"]), multi=True) == t["multi"]
    with pytest.raises(engine.B200Error):
        engine.task_definition_decode(b"\x08\x01", multi=False)     # a task without plan bytes


def test_decoder_survives_damaged_bytes():
    """Plan bytes arrive over the network: truncations, bit flips and absurd nesting must produce an error or a plan, never a
    crash or a hang (bounds-checked wire reader, recursion limit)."""
    import random
    rnd = random.Random(20260923)
    protos = [base64.b64decode(c["proto_b64"]) for c in CASES if c["name"] in ("q5/stage8", "q21/stage9", "extra/expressions", "extra/agg_partial_final")]
    assert len(protos) == 4
    outcomes = {"ok": 0, "error": 0}
    for raw in protos:
        for _ in range(300):
            b = bytearray(raw)
            kind = rnd.randrange(3)
            if kind == 0:
                b = b[:rnd.randrange(len(b))]
            elif kind == 1:
                for _k in range(rnd.randrange(1, 4)):
                    b[rnd.randrange(len(b))] ^= 1 << rnd.randrange(8)
            else:
                at = rnd.randrange(len(b))
                b[at:at] = bytes(rnd.randrange(256) for _k in range(rnd.randrange(1, 9)))
            try:
                json.loads(engine.plan_proto_to_json(bytes(b)))
                outcomes["ok"] += 1
            except engine.B200Error:
                outcomes["error"] += 1
    assert outcomes["error"] > 100
    # a filter nested 100 000 deep: FilterExecNode (field 12) { input = 1 } wrapped around itself
    inner = b""
    for _ in range(2000):
        inner = bytes([0x62]) + _varint(len(inner) + 1 + len(_varint(len(inner)))) + bytes([0x0a]) + _varint(len(inner)) + inner
    with pytest.raises(engine.B200Error):
        engine.plan_proto_to_json(inner)


def _varint(v):
    out = bytearray()
    while True:
        c = v & 0x7f
        v >>= 7
        out.append(c | (0x80 if v else 0))
        if not v:
            return bytes(out)


def test_shuffle_reader_locations_pass_through():
    """A resolved ShuffleReaderExec names where every map output lives (PartitionLocation): the decoder hands that to the host."""
    case = [c for c in CASES if c["name"] == "q5/stage6"][0]
    ir = json.loads(engine.plan_proto_to_json(base64.b64decode(case["proto_b64"])))

    def readers(n):
        out = [n] if n.get("op") == "ShuffleReaderExec" else []
        for k in ("input", "left", "right"):
            if k in n:
                out += readers(n[k])
        return out
    rs = readers(ir)
    assert rs, "q5 stage 6 reads shuffles"
    for r in rs:
        assert len(r["locations"]) == 2 and all(len(p) == 2 for p in r["locations"])
        l0, l1 = r["locations"][1]
        assert l0 == {"map_partition_id": 0, "job_id": "job", "stage_id": r["stage_id"], "partition_id": 1, "executor_id": "exec-0",
                      "host": "10.0.0.1", "port": 50050, "num_rows": 1001, "num_bytes": 16000, "is_sort_shuffle": False}
        assert l1["file_id"] == 7 and l1["is_sort_shuffle"] is True and l1["executor_id"] == "exec-1"


@pytest.mark.parametrize("case", FIX["statuses"], ids=[c["name"] for c in FIX["statuses"]])
def test_task_status_bytes(case):
    """b200_task_status_encode writes, byte for byte, the TaskStatus google.protobuf serialises from the reference's message
    definitions for the same outcome (successful / fetch failed / killed / execution error, with operator metrics)."""
    r = case["result"]
    tr = engine.TaskResult(task_id=r["task_id"], stage_id=r["stage_id"], stage_attempt_num=r["stage_attempt_num"], partition_id=r["partition_id"],
                           launch_time=r["launch_time"], start_exec_time=r["start_exec_time"], end_exec_time=r["end_exec_time"], status=r["status"],
                           fetch_map_stage_id=r.get("fetch_map_stage_id", 0), fetch_map_partition_id=r.get("fetch_map_partition_id", 0),
                           fetch_executor_id=r["fetch_executor_id"].encode() if "fetch_executor_id" in r else None,
                           error_message=r["error_message"].encode() if "error_message" in r else None)
    parts = [engine.ShuffleWritePartition(partition_id=p["partition_id"], num_batches=p["num_batches"], num_rows=p["num_rows"], num_bytes=p["num_bytes"],
                                          file_id=p["file_id"], is_sort_shuffle=p["is_sort_shuffle"]) for p in case["partitions"]]
    mets = [engine.OperatorMetrics(name=m["name"].encode(), output_rows=m["output_rows"], input_rows=m["input_rows"], elapsed_compute_ns=m["elapsed_compute_ns"],
                                   bytes_read=m["bytes_read"], bytes_written=m["bytes_written"], kernel_launches=m["kernel_launches"]) for m in case["metrics"]]
    got = engine.task_status_encode(case["job_id"], case["executor_id"], tr, parts, mets)
    assert got == base64.b64decode(case["expected_b64"])
