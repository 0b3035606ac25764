"""blaze_b200/proto.py declares the hot-path subset of the reference's auron.proto programmatically;
every message/field/number/type is checked against the reference's field table, stored in
tests/golden/auron_proto_fields.json (regenerated from the .proto text by tests/golden/make_proto_fields.py)."""
import json
import os

from blaze_b200 import proto as P

REF = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "auron_proto_fields.json")


def _load_reference():
    ref = json.load(open(REF))
    return ref["messages"], ref["enums"]


def test_field_numbers_match_reference_proto():
    msgs, enums = _load_reference()
    from google.protobuf import descriptor_pb2 as dpb
    F = dpb.FieldDescriptorProto
    scalar = {F.TYPE_STRING: "string", F.TYPE_BYTES: "bytes", F.TYPE_BOOL: "bool", F.TYPE_UINT32: "uint32",
              F.TYPE_UINT64: "uint64", F.TYPE_INT64: "int64", F.TYPE_INT32: "int32"}
    checked = 0
    for m in P.FILE_DESCRIPTOR.message_type:
        assert m.name in msgs, f"message {m.name} not in the reference proto"
        for f in m.field:
            assert f.name in msgs[m.name], f"{m.name}.{f.name} not in the reference proto"
            num, typ, rep = msgs[m.name][f.name]
            assert num == f.number, f"{m.name}.{f.name}: field number {f.number} != reference {num}"
            assert rep == (f.label == F.LABEL_REPEATED), f"{m.name}.{f.name}: repeated mismatch"
            ours = f.type_name.split(".")[-1] if f.type in (F.TYPE_MESSAGE, F.TYPE_ENUM) else scalar[f.type]
            assert ours == typ.split(".")[-1], f"{m.name}.{f.name}: type {ours} != reference {typ}"
            checked += 1
    for e in P.FILE_DESCRIPTOR.enum_type:
        for v in e.value:
            assert enums[e.name][v.name] == v.number
    assert checked > 80


def test_roundtrip_through_protobuf_runtime():
    from blaze_b200 import exprs as E, plans as PL, types as T
    s = T.Schema([T.Field("#1", T.int64, False), T.Field("#2", T.decimal128(7, 2), True)])
    plan = PL.AggExec(PL.HashAgg, [E.GroupingExpr("#1", E.Column("#1"))],
                      [E.AggExpr("#3", E.PARTIAL, PL.create_agg(E.AGG_SUM, [E.ScalarFunction("UnscaledValue", [E.Column("#2")], T.int64)], s, T.int64))],
                      True, PL.FilterExec([E.IsNotNull(E.Column("#2"))], PL.MemoryExec(s)))
    node = P.PhysicalPlanNode()
    node.ParseFromString(plan.plan_bytes())
    assert node.WhichOneof("PhysicalPlanType") == "agg" and node.agg.supports_partial_skipping
    assert node.agg.input.filter.input.ffi_reader.schema.columns[1].arrow_type.DECIMAL.whole == 7
    td = P.task_definition(node, 3, 4, 5)
    t = P.TaskDefinition(); t.ParseFromString(td)
    assert (t.task_id.stage_id, t.task_id.partition_id, t.task_id.task_id) == (3, 4, 5)
