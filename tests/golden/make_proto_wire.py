"""Record what the reference's protobuf schema says about the plan fixtures, so the tests need no copy of the reference.

    python tests/golden/make_proto_wire.py REFERENCE_CHECKOUT     (reads ballista/core/proto/*.proto there; commit the output)

Writes two gzip-compressed JSON files next to this script:
  proto_plans_wire.json.gz    every fixture of proto_plans.json parsed with message classes built from the reference's .proto
                              files: a field tree [number, name, wire type, value], a sub-message's value being its own tree
                              (PhysicalExtensionNode.node holds a BallistaPhysicalPlanNode and is expanded as one).  The
                              generator checks that each fixture parses with no unknown field and re-serialises byte-identically.
  proto_random_plans.json.gz  the seeded random stage plans of tests/test_plan_proto_random.py, encoded as
                              datafusion.PhysicalPlanNode by make_proto_plans.encode (google.protobuf over the same schema).
Needs a built libb200exec.so (the engine types each plan before it is encoded).
"""
import base64
import gzip
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, HERE)

import make_proto_plans as M  # noqa: E402
import protoc_lite  # noqa: E402
from test_plan_proto import wire_fields  # noqa: E402

RANDOM_SEEDS = 600


def tree(buf, desc, classes):
    """The wire fields of `buf` named by message descriptor `desc`; every field must be one the schema declares."""
    out = []
    for num, wt, v in wire_fields(buf):
        fd = desc.fields_by_number[num]
        if wt == 2 and fd.message_type is not None:
            v = tree(v, fd.message_type, classes)
        elif desc.full_name == "datafusion.PhysicalExtensionNode" and fd.name == "node":
            v = tree(v, classes["ballista.protobuf.BallistaPhysicalPlanNode"].DESCRIPTOR, classes)
        elif wt == 2:
            v = base64.b64encode(v).decode()
        out.append([num, fd.name, wt, v])
    return out


def _write(name, obj):
    with open(os.path.join(HERE, name), "wb") as fh:
        fh.write(gzip.compress(json.dumps(obj, separators=(",", ":")).encode(), 9, mtime=0))


def main(reference):
    classes, _ = protoc_lite.load_ballista(os.path.join(reference, "ballista", "core", "proto"))
    M.CLS = classes
    P = classes["datafusion.PhysicalPlanNode"]
    with open(os.path.join(HERE, "proto_plans.json")) as fh:
        cases = json.load(fh)["cases"]
    wire = {}
    for c in cases:
        raw = base64.b64decode(c["proto_b64"])
        m = P()
        m.ParseFromString(raw)
        assert m.SerializeToString() == raw, c["name"]
        wire[c["name"]] = tree(raw, P.DESCRIPTOR, classes)
    _write("proto_plans_wire.json.gz", {"generated_by": "tests/golden/make_proto_wire.py", "cases": wire})

    from ballista_b200 import engine
    from test_plan_proto_random import _plan
    plans = {}
    for seed in range(RANDOM_SEEDS):
        ir = json.dumps(_plan(seed), separators=(",", ":"))
        try:
            engine.plan_typed_json(ir)
        except engine.B200Error:
            continue            # ill-typed combination: the test counts it as rejected
        plans[str(seed)] = base64.b64encode(M.encode(ir)).decode()
    _write("proto_random_plans.json.gz", {"generated_by": "tests/golden/make_proto_wire.py", "seeds": RANDOM_SEEDS, "plans": plans})
    print(len(wire), "fixtures,", len(plans), "of", RANDOM_SEEDS, "random plans")


if __name__ == "__main__":
    main(sys.argv[1])
