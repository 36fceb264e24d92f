"""The gRPC schema table of client_b200/grpc/_proto.py against the reference's own .proto files.

The fixture tests/golden/proto_schema.json is the parse of the reference's
src/rust/triton-client/proto/{grpc_service,model_config}.proto (the only copy of the
wire schema in the reference) made by oracle/gen_proto_fixture.py.  Every message, field (name,
number, type, repeated / map / oneof membership), enum value and rpc of package `inference` must be
present in the descriptors the drop-in builds at import time, and nothing else may be there --
the goldens of tests/test_wire_parity.py are serialised through these descriptors, so this is what
keeps them from agreeing with themselves."""

import hashlib
import json
import os

import pytest
from google.protobuf import descriptor as D

from client_b200.grpc import _proto

HERE = os.path.dirname(os.path.abspath(__file__))
FIXTURE = os.path.join(HERE, "golden", "proto_schema.json")

SCALAR = {
    "double": D.FieldDescriptor.TYPE_DOUBLE, "float": D.FieldDescriptor.TYPE_FLOAT, "int32": D.FieldDescriptor.TYPE_INT32,
    "int64": D.FieldDescriptor.TYPE_INT64, "uint32": D.FieldDescriptor.TYPE_UINT32, "uint64": D.FieldDescriptor.TYPE_UINT64,
    "bool": D.FieldDescriptor.TYPE_BOOL, "string": D.FieldDescriptor.TYPE_STRING, "bytes": D.FieldDescriptor.TYPE_BYTES,
}


@pytest.fixture(scope="module")
def schema():
    with open(FIXTURE) as fh:
        return json.load(fh)["packages"]["inference"]


@pytest.fixture(scope="module")
def file_desc():
    return _proto.build_modules()[0].DESCRIPTOR


def _all_messages(file_desc):
    out = {}

    def walk(desc, prefix):
        if desc.GetOptions().map_entry:
            return
        name = prefix + desc.name
        out[name] = desc
        for nested in desc.nested_types:
            walk(nested, name + ".")

    for m in file_desc.message_types_by_name.values():
        walk(m, "")
    return out


def _all_enums(file_desc):
    out = {e.name: e for e in file_desc.enum_types_by_name.values()}
    for name, m in _all_messages(file_desc).items():
        for e in m.enum_types:
            out[name + "." + e.name] = e
    return out


def _is_repeated(fd):
    return fd.is_repeated if hasattr(fd, "is_repeated") else fd.label == D.FieldDescriptor.LABEL_REPEATED


def _check_type(fd, type_name, kind, where):
    if kind == "scalar":
        assert fd.type == SCALAR[type_name], where
    elif kind == "enum":
        assert fd.type == D.FieldDescriptor.TYPE_ENUM and fd.enum_type.full_name == "inference." + type_name, where
    else:
        assert fd.type == D.FieldDescriptor.TYPE_MESSAGE and fd.message_type.full_name == "inference." + type_name, where


def test_fixture_is_the_parse_of_the_reference_protos():
    """The committed fixture hashes to the digest of what the generator printed for the reference's
    .proto files (tests/golden/reference_digests.json)."""
    with open(FIXTURE) as fh:
        committed = json.load(fh)["packages"]
    with open(os.path.join(HERE, "golden", "reference_digests.json")) as fh:
        want = json.load(fh)["proto_schema_parse"]["digest"]
    assert hashlib.sha256(json.dumps(committed, sort_keys=True, separators=(",", ":")).encode()).hexdigest() == want


def test_every_message_and_field_matches_the_reference(schema, file_desc):
    ours = _all_messages(file_desc)
    assert sorted(ours) == sorted(schema["messages"]), "message set differs from grpc_service.proto + model_config.proto"
    checked = 0
    for mname, msg in schema["messages"].items():
        desc = ours[mname]
        want = {f["name"]: f for f in msg["fields"]}
        assert sorted(f.name for f in desc.fields) == sorted(want), mname
        for fd in desc.fields:
            f = want[fd.name]
            where = "%s.%s" % (mname, fd.name)
            assert fd.number == f["number"], where
            if f["type"] == "map":
                assert _is_repeated(fd) and fd.message_type.GetOptions().map_entry, where
                key, value = fd.message_type.fields_by_name["key"], fd.message_type.fields_by_name["value"]
                assert key.type == SCALAR[f["key"]], where
                _check_type(value, f["value"], f["kind"], where)
            else:
                assert _is_repeated(fd) == (f["label"] == "repeated"), where
                _check_type(fd, f["type"], f["kind"], where)
            group = fd.containing_oneof.name if fd.containing_oneof is not None else None
            assert group == f.get("oneof"), where
            checked += 1
    assert checked == sum(len(m["fields"]) for m in schema["messages"].values()) and checked > 300  # 105 messages


def test_every_enum_value_matches_the_reference(schema, file_desc):
    ours = _all_enums(file_desc)
    assert sorted(ours) == sorted(schema["enums"])
    for ename, values in schema["enums"].items():
        assert [[v.name, v.number] for v in ours[ename].values] == values, ename


def test_service_rpcs_match_the_reference(schema, file_desc):
    want = schema["services"]["GRPCInferenceService"]
    svc = file_desc.services_by_name["GRPCInferenceService"]
    assert sorted(m.name for m in svc.methods) == sorted(want)
    for m in svc.methods:
        req, resp, cs, ss = want[m.name]
        assert (m.input_type.full_name, m.output_type.full_name) == ("inference." + req, "inference." + resp), m.name
        assert (bool(m.client_streaming), bool(m.server_streaming)) == (cs, ss), m.name
    assert svc.full_name == _proto.SERVICE_NAME


def test_model_config_sections_round_trip():
    """ADVICE r1: get_model_config(...).config.dynamic_batching / instance_group / sequence_batching
    exist and survive serialisation and as_json."""
    from google.protobuf import json_format

    service_pb2, _, model_config_pb2 = _proto.build_modules()
    c = model_config_pb2.ModelConfig(name="m", max_batch_size=8)
    c.dynamic_batching.preferred_batch_size.extend([4, 8])
    c.dynamic_batching.priority_queue_policy[3].max_queue_size = 7
    g = c.instance_group.add()
    g.kind, g.count = model_config_pb2.ModelInstanceGroup.KIND_GPU, 2
    c.parameters["k"].string_value = "v"
    c.version_policy.specific.versions.extend([1, 3])
    c.optimization.cuda.graphs = True
    back = service_pb2.ModelConfigResponse.FromString(service_pb2.ModelConfigResponse(config=c).SerializeToString())
    assert back.config == c and back.config.WhichOneof("scheduling_choice") == "dynamic_batching"
    js = json_format.MessageToDict(back, preserving_proto_field_name=True)
    assert js["config"]["instance_group"][0] == {"kind": "KIND_GPU", "count": 2}
    assert js["config"]["dynamic_batching"]["priority_queue_policy"]["3"] == {"max_queue_size": 7}
    c2 = model_config_pb2.ModelConfig()
    c2.sequence_batching.oldest.max_candidate_sequences = 4
    assert c2.WhichOneof("scheduling_choice") == "sequence_batching"
    assert c2.sequence_batching.WhichOneof("strategy_choice") == "oldest"
