"""Plan-serde surface: the subset of the reference's `auron.proto` needed by the hot path,
declared programmatically (no protoc in this image) with the SAME package, message names and
field numbers, so bytes produced here are byte-compatible with what the Spark side emits and
what `auron-serde` decodes (native-engine/auron-serde/proto/auron.proto:27-55, 58-125, 143-148,
169-198, 271-311, 363-366, 470-473, 489-510, 675-696, 729-740, 751-760, 786-789, 824-826, 860-896).

`tests/test_proto_compat.py` checks every field number declared here against the reference's
field table, stored in `tests/golden/auron_proto_fields.json`.
"""
from __future__ import annotations

from typing import Optional

from google.protobuf import descriptor_pb2 as dpb
from google.protobuf import descriptor_pool, message_factory

from . import exprs as E
from . import types as T
from .types import DataType, Schema

_F = dpb.FieldDescriptorProto
_PKG = "plan.protobuf"


def _msg(fd, name, fields, oneofs=()):
    m = fd.message_type.add()
    m.name = name
    for o in oneofs:
        m.oneof_decl.add().name = o
    for spec in fields:
        fname, num, ftype = spec[0], spec[1], spec[2]
        f = m.field.add()
        f.name, f.number = fname, num
        kw = spec[3] if len(spec) > 3 else {}
        f.label = _F.LABEL_REPEATED if kw.get("repeated") else _F.LABEL_OPTIONAL
        if isinstance(ftype, str):
            if ftype.startswith("enum:"):
                f.type = _F.TYPE_ENUM
                f.type_name = f".{_PKG}.{ftype[5:]}"
            else:
                f.type = _F.TYPE_MESSAGE
                f.type_name = f".{_PKG}.{ftype}"
        else:
            f.type = ftype
        if "oneof" in kw:
            f.oneof_index = kw["oneof"]
    return m


def _enum(fd, name, values):
    e = fd.enum_type.add()
    e.name = name
    for n, v in values:
        ev = e.value.add()
        ev.name, ev.number = n, v


def _build_pool():
    fd = dpb.FileDescriptorProto()
    fd.name = "auron_hotpath_subset.proto"
    fd.package = _PKG
    fd.syntax = "proto3"
    R = {"repeated": True}

    _msg(fd, "EmptyMessage", [])
    _enum(fd, "TimeUnit", [("Second", 0), ("Millisecond", 1), ("Microsecond", 2), ("Nanosecond", 3)])
    _msg(fd, "Timestamp", [("time_unit", 1, "enum:TimeUnit"), ("timezone", 2, _F.TYPE_STRING)])
    _msg(fd, "Decimal", [("whole", 1, _F.TYPE_UINT64), ("fractional", 2, _F.TYPE_INT64)])
    O = {"oneof": 0}
    _msg(fd, "ArrowType", [
        ("NONE", 1, "EmptyMessage", O), ("BOOL", 2, "EmptyMessage", O), ("INT8", 4, "EmptyMessage", O),
        ("INT16", 6, "EmptyMessage", O), ("INT32", 8, "EmptyMessage", O), ("INT64", 10, "EmptyMessage", O),
        ("FLOAT32", 12, "EmptyMessage", O), ("FLOAT64", 13, "EmptyMessage", O), ("UTF8", 14, "EmptyMessage", O),
        ("BINARY", 15, "EmptyMessage", O), ("DATE32", 17, "EmptyMessage", O),
        ("TIMESTAMP", 20, "Timestamp", O), ("DECIMAL", 24, "Decimal", O),
    ], oneofs=["arrow_type_enum"])
    _msg(fd, "Field", [("name", 1, _F.TYPE_STRING), ("arrow_type", 2, "ArrowType"), ("nullable", 3, _F.TYPE_BOOL),
                       ("children", 4, "Field", R)])
    _msg(fd, "Schema", [("columns", 1, "Field", R)])
    _msg(fd, "ScalarValue", [("ipc_bytes", 1, _F.TYPE_BYTES)])

    _enum(fd, "AggFunction", [("MIN", 0), ("MAX", 1), ("SUM", 2), ("AVG", 3), ("COUNT", 4), ("COLLECT_LIST", 5),
                              ("COLLECT_SET", 6), ("FIRST", 7), ("FIRST_IGNORES_NULL", 8), ("BLOOM_FILTER", 9),
                              ("BRICKHOUSE_COLLECT", 1000), ("BRICKHOUSE_COMBINE_UNIQUE", 1001), ("UDAF", 1002)])
    _enum(fd, "AggExecMode", [("HASH_AGG", 0), ("SORT_AGG", 1)])
    _enum(fd, "AggMode", [("PARTIAL", 0), ("PARTIAL_MERGE", 1), ("FINAL", 2)])
    _enum(fd, "ScalarFunction", [("Abs", 0), ("SparkExtFunctions", 10000)])

    _msg(fd, "PhysicalColumn", [("name", 1, _F.TYPE_STRING), ("index", 2, _F.TYPE_UINT32)])
    _msg(fd, "BoundReference", [("index", 1, _F.TYPE_UINT64), ("data_type", 2, "ArrowType"), ("nullable", 3, _F.TYPE_BOOL)])
    _msg(fd, "PhysicalBinaryExprNode", [("l", 1, "PhysicalExprNode"), ("r", 2, "PhysicalExprNode"), ("op", 3, _F.TYPE_STRING)])
    _msg(fd, "PhysicalAggExprNode", [("agg_function", 1, "enum:AggFunction"), ("children", 3, "PhysicalExprNode", R),
                                      ("return_type", 4, "ArrowType")])
    _msg(fd, "PhysicalIsNull", [("expr", 1, "PhysicalExprNode")])
    _msg(fd, "PhysicalIsNotNull", [("expr", 1, "PhysicalExprNode")])
    _msg(fd, "PhysicalNot", [("expr", 1, "PhysicalExprNode")])
    _msg(fd, "PhysicalWhenThen", [("when_expr", 1, "PhysicalExprNode"), ("then_expr", 2, "PhysicalExprNode")])
    _msg(fd, "PhysicalCaseNode", [("expr", 1, "PhysicalExprNode"), ("when_then_expr", 2, "PhysicalWhenThen", R),
                                   ("else_expr", 3, "PhysicalExprNode")])
    _msg(fd, "PhysicalCastNode", [("expr", 1, "PhysicalExprNode"), ("arrow_type", 2, "ArrowType")])
    _msg(fd, "PhysicalTryCastNode", [("expr", 1, "PhysicalExprNode"), ("arrow_type", 2, "ArrowType")])
    _msg(fd, "PhysicalNegativeNode", [("expr", 1, "PhysicalExprNode")])
    _msg(fd, "PhysicalInListNode", [("expr", 1, "PhysicalExprNode"), ("list", 2, "PhysicalExprNode", R), ("negated", 3, _F.TYPE_BOOL)])
    _msg(fd, "PhysicalScalarFunctionNode", [("name", 1, _F.TYPE_STRING), ("fun", 2, "enum:ScalarFunction"),
                                             ("args", 3, "PhysicalExprNode", R), ("return_type", 4, "ArrowType")])
    _msg(fd, "PhysicalSCAndExprNode", [("left", 1, "PhysicalExprNode"), ("right", 2, "PhysicalExprNode")])
    _msg(fd, "PhysicalSCOrExprNode", [("left", 1, "PhysicalExprNode"), ("right", 2, "PhysicalExprNode")])
    _msg(fd, "PhysicalSortExprNode", [("expr", 1, "PhysicalExprNode"), ("asc", 2, _F.TYPE_BOOL), ("nulls_first", 3, _F.TYPE_BOOL)])
    _msg(fd, "PhysicalExprNode", [
        ("column", 1, "PhysicalColumn", O), ("literal", 2, "ScalarValue", O), ("bound_reference", 3, "BoundReference", O),
        ("binary_expr", 4, "PhysicalBinaryExprNode", O), ("agg_expr", 5, "PhysicalAggExprNode", O),
        ("is_null_expr", 6, "PhysicalIsNull", O), ("is_not_null_expr", 7, "PhysicalIsNotNull", O),
        ("not_expr", 8, "PhysicalNot", O), ("case_", 9, "PhysicalCaseNode", O), ("cast", 10, "PhysicalCastNode", O),
        ("sort", 11, "PhysicalSortExprNode", O),
        ("negative", 12, "PhysicalNegativeNode", O), ("in_list", 13, "PhysicalInListNode", O),
        ("scalar_function", 14, "PhysicalScalarFunctionNode", O), ("try_cast", 15, "PhysicalTryCastNode", O),
        ("sc_and_expr", 3000, "PhysicalSCAndExprNode", O), ("sc_or_expr", 3001, "PhysicalSCOrExprNode", O),
    ], oneofs=["ExprType"])

    _msg(fd, "FilterExecNode", [("input", 1, "PhysicalPlanNode"), ("expr", 2, "PhysicalExprNode", R)])
    _msg(fd, "ProjectionExecNode", [("input", 1, "PhysicalPlanNode"), ("expr", 2, "PhysicalExprNode", R),
                                     ("expr_name", 3, _F.TYPE_STRING, R), ("data_type", 4, "ArrowType", R)])
    _msg(fd, "EmptyPartitionsExecNode", [("schema", 1, "Schema"), ("num_partitions", 2, _F.TYPE_UINT32)])
    _msg(fd, "FFIReaderExecNode", [("num_partitions", 1, _F.TYPE_UINT32), ("schema", 2, "Schema"),
                                    ("export_iter_provider_resource_id", 3, _F.TYPE_STRING)])
    _msg(fd, "AggExecNode", [
        ("input", 1, "PhysicalPlanNode"), ("exec_mode", 2, "enum:AggExecMode"), ("grouping_expr", 3, "PhysicalExprNode", R),
        ("agg_expr", 4, "PhysicalExprNode", R), ("mode", 5, "enum:AggMode", R), ("grouping_expr_name", 6, _F.TYPE_STRING, R),
        ("agg_expr_name", 7, _F.TYPE_STRING, R), ("initial_input_buffer_offset", 8, _F.TYPE_UINT64),
        ("supports_partial_skipping", 9, _F.TYPE_BOOL)])
    _enum(fd, "JoinType", [("INNER", 0), ("LEFT", 1), ("RIGHT", 2), ("FULL", 3), ("SEMI", 4), ("ANTI", 5), ("EXISTENCE", 6)])
    _enum(fd, "JoinSide", [("LEFT_SIDE", 0), ("RIGHT_SIDE", 1)])
    _msg(fd, "JoinOn", [("left", 1, "PhysicalExprNode"), ("right", 2, "PhysicalExprNode")])
    _msg(fd, "HashJoinExecNode", [("schema", 1, "Schema"), ("left", 2, "PhysicalPlanNode"), ("right", 3, "PhysicalPlanNode"), ("on", 4, "JoinOn", R),
                                  ("join_type", 5, "enum:JoinType"), ("build_side", 6, "enum:JoinSide")])
    _msg(fd, "BroadcastJoinBuildHashMapExecNode", [("input", 1, "PhysicalPlanNode"), ("keys", 2, "PhysicalExprNode", R)])
    _msg(fd, "BroadcastJoinExecNode", [("schema", 1, "Schema"), ("left", 2, "PhysicalPlanNode"), ("right", 3, "PhysicalPlanNode"), ("on", 4, "JoinOn", R),
                                       ("join_type", 5, "enum:JoinType"), ("broadcast_side", 6, "enum:JoinSide"), ("cached_build_hash_map_id", 7, _F.TYPE_STRING)])
    _msg(fd, "FileRange", [("start", 1, _F.TYPE_INT64), ("end", 2, _F.TYPE_INT64)])
    _msg(fd, "PartitionedFile", [("path", 1, _F.TYPE_STRING), ("size", 2, _F.TYPE_UINT64), ("last_modified_ns", 3, _F.TYPE_UINT64),
                                 ("partition_values", 4, "ScalarValue", R), ("range", 5, "FileRange")])
    _msg(fd, "FileGroup", [("files", 1, "PartitionedFile", R)])
    _msg(fd, "ScanLimit", [("limit", 1, _F.TYPE_UINT32)])
    _msg(fd, "FileScanExecConf", [("num_partitions", 1, _F.TYPE_INT64), ("partition_index", 2, _F.TYPE_INT64), ("file_group", 3, "FileGroup"), ("schema", 4, "Schema"),
                                  ("projection", 6, _F.TYPE_UINT32, R), ("limit", 7, "ScanLimit"), ("partition_schema", 9, "Schema")])
    _msg(fd, "ParquetScanExecNode", [("base_conf", 1, "FileScanExecConf"), ("pruning_predicates", 2, "PhysicalExprNode", R), ("fsResourceId", 3, _F.TYPE_STRING)])
    _msg(fd, "FetchLimit", [("limit", 1, _F.TYPE_UINT64)])
    _msg(fd, "SortExecNode", [("input", 1, "PhysicalPlanNode"), ("expr", 2, "PhysicalExprNode", R), ("fetch_limit", 3, "FetchLimit")])
    _msg(fd, "PhysicalSingleRepartition", [("partition_count", 1, _F.TYPE_UINT64)])
    _msg(fd, "PhysicalHashRepartition", [("hash_expr", 1, "PhysicalExprNode", R), ("partition_count", 2, _F.TYPE_UINT64)])
    _msg(fd, "PhysicalRoundRobinRepartition", [("partition_count", 1, _F.TYPE_UINT64)])
    _msg(fd, "PhysicalRepartition", [
        ("single_repartition", 1, "PhysicalSingleRepartition", O), ("hash_repartition", 2, "PhysicalHashRepartition", O),
        ("round_robin_repartition", 3, "PhysicalRoundRobinRepartition", O),
    ], oneofs=["RepartitionType"])
    _msg(fd, "ShuffleWriterExecNode", [("input", 1, "PhysicalPlanNode"), ("output_partitioning", 2, "PhysicalRepartition"),
                                       ("output_data_file", 3, _F.TYPE_STRING), ("output_index_file", 4, _F.TYPE_STRING)])
    _msg(fd, "PhysicalPlanNode", [
        ("shuffle_writer", 2, "ShuffleWriterExecNode", O), ("parquet_scan", 5, "ParquetScanExecNode", O), ("projection", 6, "ProjectionExecNode", O), ("sort", 7, "SortExecNode", O),
        ("hash_join", 11, "HashJoinExecNode", O), ("broadcast_join_build_hash_map", 12, "BroadcastJoinBuildHashMapExecNode", O),
        ("broadcast_join", 13, "BroadcastJoinExecNode", O), ("filter", 8, "FilterExecNode", O),
        ("empty_partitions", 15, "EmptyPartitionsExecNode", O), ("agg", 16, "AggExecNode", O),
        ("ffi_reader", 18, "FFIReaderExecNode", O),
    ], oneofs=["PhysicalPlanType"])
    _msg(fd, "PartitionId", [("stage_id", 2, _F.TYPE_UINT32), ("partition_id", 4, _F.TYPE_UINT32), ("task_id", 5, _F.TYPE_UINT64)])
    _msg(fd, "TaskDefinition", [("task_id", 1, "PartitionId"), ("plan", 2, "PhysicalPlanNode")])

    pool = descriptor_pool.DescriptorPool()
    pool.Add(fd)
    return pool, fd


_POOL, FILE_DESCRIPTOR = _build_pool()


def cls(name: str):
    return message_factory.GetMessageClass(_POOL.FindMessageTypeByName(f"{_PKG}.{name}"))


PhysicalPlanNode = cls("PhysicalPlanNode")
PhysicalExprNode = cls("PhysicalExprNode")
ArrowType = cls("ArrowType")
TaskDefinition = cls("TaskDefinition")
SchemaMsg = cls("Schema")

_EMPTY_TYPES = {T.BOOL: "BOOL", T.INT8: "INT8", T.INT16: "INT16", T.INT32: "INT32", T.INT64: "INT64",
                T.FLOAT32: "FLOAT32", T.FLOAT64: "FLOAT64", T.DATE32: "DATE32", T.BINARY: "BINARY", T.NULLTYPE: "NONE"}


def arrow_type_msg(dt: DataType):
    """convertDataType (NativeConverters.scala:117-144): Decimal{whole=precision, fractional=scale},
    TimestampType -> TIMESTAMP{Microsecond, tz ""}."""
    m = ArrowType()
    if dt.id == T.DECIMAL128:
        m.DECIMAL.whole = dt.precision
        m.DECIMAL.fractional = dt.scale
    elif dt.id == T.TIMESTAMP_US:
        m.TIMESTAMP.time_unit = 2
        m.TIMESTAMP.timezone = ""
    else:
        getattr(m, _EMPTY_TYPES[dt.id]).SetInParent()
    return m


def schema_msg(schema: Schema):
    m = SchemaMsg()
    for f in schema:
        c = m.columns.add()
        c.name = f.name
        c.arrow_type.CopyFrom(arrow_type_msg(f.dtype))
        c.nullable = f.nullable
    return m


def literal_ipc_bytes(value, dt: DataType) -> bytes:
    """ScalarValue.ipc_bytes = a complete Arrow IPC *stream* holding one 1-row batch whose single
    field is named "" (NativeConverters.scala:382-403; decoded at auron-serde/src/lib.rs:447-457)."""
    import decimal
    import pyarrow as pa
    at = T.to_arrow_type(dt)
    if value is not None and dt.id == T.DECIMAL128:
        value = decimal.Decimal(int(value)).scaleb(-dt.scale, decimal.Context(prec=60))
    if dt.id == T.DATE32 and value is not None:
        arr = pa.array([int(value)], pa.int32()).cast(at)
    elif dt.id == T.TIMESTAMP_US and value is not None:
        arr = pa.array([int(value)], pa.int64()).cast(at)
    else:
        arr = pa.array([value], type=at)
    rb = pa.RecordBatch.from_arrays([arr], schema=pa.schema([pa.field("", at, True)]))
    sink = pa.BufferOutputStream()
    with pa.ipc.new_stream(sink, rb.schema) as w:
        w.write_batch(rb)
    return sink.getvalue().to_pybytes()


def expr_msg(e: E.Expr):
    m = PhysicalExprNode()
    if isinstance(e, E.Column):
        m.column.name = e.name
    elif isinstance(e, E.BoundReference):
        m.bound_reference.index = e.index
        if e.dtype is not None:
            m.bound_reference.data_type.CopyFrom(arrow_type_msg(e.dtype))
        m.bound_reference.nullable = e.is_nullable
    elif isinstance(e, E.Literal):
        m.literal.ipc_bytes = literal_ipc_bytes(e.value, e.dtype)
    elif isinstance(e, E.BinaryExpr):
        m.binary_expr.l.CopyFrom(expr_msg(e.left))
        m.binary_expr.r.CopyFrom(expr_msg(e.right))
        m.binary_expr.op = e.op
    elif isinstance(e, E.IsNull):
        m.is_null_expr.expr.CopyFrom(expr_msg(e.expr))
    elif isinstance(e, E.IsNotNull):
        m.is_not_null_expr.expr.CopyFrom(expr_msg(e.expr))
    elif isinstance(e, E.Not):
        m.not_expr.expr.CopyFrom(expr_msg(e.expr))
    elif isinstance(e, E.Negative):
        m.negative.expr.CopyFrom(expr_msg(e.expr))
    elif isinstance(e, E.Cast):
        m.cast.expr.CopyFrom(expr_msg(e.expr))
        m.cast.arrow_type.CopyFrom(arrow_type_msg(e.dtype))
    elif isinstance(e, E.TryCast):
        m.try_cast.expr.CopyFrom(expr_msg(e.expr))
        m.try_cast.arrow_type.CopyFrom(arrow_type_msg(e.dtype))
    elif isinstance(e, E.Case):
        c = getattr(m, "case_")
        if e.expr is not None:
            c.expr.CopyFrom(expr_msg(e.expr))
        for w, t in e.when_then:
            wt = c.when_then_expr.add()
            wt.when_expr.CopyFrom(expr_msg(w))
            wt.then_expr.CopyFrom(expr_msg(t))
        if e.else_expr is not None:
            c.else_expr.CopyFrom(expr_msg(e.else_expr))
        if e.expr is None and e.else_expr is None and not e.when_then:
            c.SetInParent()
    elif isinstance(e, E.InList):
        m.in_list.expr.CopyFrom(expr_msg(e.expr))
        for x in e.list:
            m.in_list.list.add().CopyFrom(expr_msg(x))
        m.in_list.negated = e.negated
    elif isinstance(e, E.SCAnd):
        m.sc_and_expr.left.CopyFrom(expr_msg(e.left))
        m.sc_and_expr.right.CopyFrom(expr_msg(e.right))
    elif isinstance(e, E.SCOr):
        m.sc_or_expr.left.CopyFrom(expr_msg(e.left))
        m.sc_or_expr.right.CopyFrom(expr_msg(e.right))
    elif isinstance(e, E.ScalarFunction):
        sf = m.scalar_function
        sf.name = e.name
        sf.fun = 10000                                   # ScalarFunction.SparkExtFunctions
        for a in e.args:
            sf.args.add().CopyFrom(expr_msg(a))
        sf.return_type.CopyFrom(arrow_type_msg(e.return_type))
    else:
        raise TypeError(f"cannot serialise expression {e!r}")
    return m


def agg_expr_msg(a: E.AggFunctionExpr):
    m = PhysicalExprNode()
    m.agg_expr.agg_function = a.function
    for c in a.children:
        m.agg_expr.children.add().CopyFrom(expr_msg(c))
    m.agg_expr.return_type.CopyFrom(arrow_type_msg(a.return_type))
    return m


# ---- plan node builders ---------------------------------------------------------------------------

def ffi_reader_node(schema: Schema, resource_id: str = "", num_partitions: int = 1):
    n = PhysicalPlanNode()
    n.ffi_reader.num_partitions = num_partitions
    n.ffi_reader.schema.CopyFrom(schema_msg(schema))
    n.ffi_reader.export_iter_provider_resource_id = resource_id
    return n


def empty_partitions_node(schema: Schema, num_partitions: int = 1):
    n = PhysicalPlanNode()
    n.empty_partitions.schema.CopyFrom(schema_msg(schema))
    n.empty_partitions.num_partitions = num_partitions
    return n


def filter_node(input_node, predicates):
    n = PhysicalPlanNode()
    n.filter.input.CopyFrom(input_node)
    for p in predicates:
        n.filter.expr.add().CopyFrom(expr_msg(p))
    return n


def projection_node(input_node, exprs, names, data_types):
    n = PhysicalPlanNode()
    n.projection.input.CopyFrom(input_node)
    for e, name, dt in zip(exprs, names, data_types):
        n.projection.expr.add().CopyFrom(expr_msg(e))
        n.projection.expr_name.append(name)
        n.projection.data_type.add().CopyFrom(arrow_type_msg(dt))
    return n


def agg_node(input_node, exec_mode, groupings, aggs, supports_partial_skipping=False,
             initial_input_buffer_offset=0):
    n = PhysicalPlanNode()
    a = n.agg
    a.input.CopyFrom(input_node)
    a.exec_mode = exec_mode
    for g in groupings:
        a.grouping_expr.add().CopyFrom(expr_msg(g.expr))
        a.grouping_expr_name.append(g.field_name)
    for ag in aggs:
        a.agg_expr.add().CopyFrom(agg_expr_msg(ag.agg))
        a.agg_expr_name.append(ag.field_name)
        a.mode.append(ag.mode)
    a.initial_input_buffer_offset = initial_input_buffer_offset
    a.supports_partial_skipping = supports_partial_skipping
    return n


def parquet_scan_node(file_schema: Schema, files, projection=None, pruning_predicates=(), limit=None, fs_resource_id=""):
    """files: [(path, size, (range_start, range_end) | None)] (FileScanExecConf, auron.proto:404-413)"""
    n = PhysicalPlanNode()
    c = n.parquet_scan.base_conf
    c.num_partitions, c.partition_index = 1, 0
    for path, size, rng in files:
        f = c.file_group.files.add()
        f.path, f.size = path, size
        if rng is not None:
            f.range.start, f.range.end = rng
    c.schema.CopyFrom(schema_msg(file_schema))
    for i in (projection if projection is not None else range(len(file_schema))):
        c.projection.append(i)
    if limit is not None:
        c.limit.limit = limit
    for p in pruning_predicates:
        n.parquet_scan.pruning_predicates.add().CopyFrom(expr_msg(p))
    n.parquet_scan.fsResourceId = fs_resource_id
    return n


def sort_node(input_node, sort_exprs, fetch=None):
    """sort_exprs: [(expr, asc, nulls_first)] (PhysicalSortExprNode, auron.proto:178-182); fetch: optional FetchLimit"""
    n = PhysicalPlanNode()
    n.sort.input.CopyFrom(input_node)
    for e, asc, nulls_first in sort_exprs:
        x = n.sort.expr.add()
        x.sort.expr.CopyFrom(expr_msg(e))
        x.sort.asc, x.sort.nulls_first = asc, nulls_first
    if fetch is not None:
        n.sort.fetch_limit.limit = fetch
    return n


def join_build_node(input_node, keys):
    n = PhysicalPlanNode()
    n.broadcast_join_build_hash_map.input.CopyFrom(input_node)
    for k in keys:
        n.broadcast_join_build_hash_map.keys.add().CopyFrom(expr_msg(k))
    return n


def join_node(schema: Schema, left_node, right_node, on, join_type: int, map_side: int, broadcast: bool, cached_id: str = ""):
    """HashJoinExecNode (broadcast=False, `build_side`) / BroadcastJoinExecNode (broadcast=True, `broadcast_side`); on = [(left expr, right expr)]"""
    n = PhysicalPlanNode()
    j = n.broadcast_join if broadcast else n.hash_join
    j.schema.CopyFrom(schema_msg(schema))
    j.left.CopyFrom(left_node)
    j.right.CopyFrom(right_node)
    for l, r in on:
        o = j.on.add()
        o.left.CopyFrom(expr_msg(l))
        o.right.CopyFrom(expr_msg(r))
    j.join_type = join_type
    if broadcast:
        j.broadcast_side = map_side
        j.cached_build_hash_map_id = cached_id
    else:
        j.build_side = map_side
    return n


def shuffle_writer_node(input_node, partitioning, data_file: str, index_file: str):
    """partitioning: ("single",) | ("hash", [exprs], n) | ("round_robin", n)  (PhysicalRepartition, auron.proto:629-649)"""
    n = PhysicalPlanNode()
    w = n.shuffle_writer
    w.input.CopyFrom(input_node)
    kind = partitioning[0]
    if kind == "single":
        w.output_partitioning.single_repartition.partition_count = 1
    elif kind == "hash":
        for e in partitioning[1]:
            w.output_partitioning.hash_repartition.hash_expr.add().CopyFrom(expr_msg(e))
        w.output_partitioning.hash_repartition.partition_count = partitioning[2]
    elif kind == "round_robin":
        w.output_partitioning.round_robin_repartition.partition_count = partitioning[1]
    else:
        raise ValueError(kind)
    w.output_data_file, w.output_index_file = data_file, index_file
    return n


def task_definition(plan_node, stage_id=0, partition_id=0, task_id=0) -> bytes:
    t = TaskDefinition()
    t.task_id.stage_id, t.task_id.partition_id, t.task_id.task_id = stage_id, partition_id, task_id
    t.plan.CopyFrom(plan_node)
    return t.SerializeToString()
