"""The orbslam2.KeyFrameData schema (reference: proto/Keyframe.proto:1-70) restated as a dynamically built descriptor for
the python protobuf runtime (no protoc needed).  test_serialize.py checks the restatement against a digest of the
reference's .proto text as parse_proto_text reads it, and uses the runtime's own serializer / parser as the wire-format oracle."""
import re

from google.protobuf import descriptor_pb2, descriptor_pool, message_factory

F = descriptor_pb2.FieldDescriptorProto
TYPES = {"float": F.TYPE_FLOAT, "double": F.TYPE_DOUBLE, "int32": F.TYPE_INT32, "int64": F.TYPE_INT64, "uint32": F.TYPE_UINT32, "uint64": F.TYPE_UINT64,
         "bytes": F.TYPE_BYTES}

# message -> [(name, number, type, repeated)]; type is a scalar name, a message name, or ("map", key, value)
SCHEMA = {
    "KeyPoint": [("x", 1, "float", False), ("y", 2, "float", False), ("octave", 3, "int32", False), ("angle", 4, "float", False)],
    "Descriptor": [("data", 1, "bytes", False)],
    "BowVector": [("words", 1, ("map", "uint32", "double"), False)],
    "FeatureVector.FeatureNode": [("node_id", 1, "uint32", False), ("feature_ids", 2, "uint32", True)],
    "FeatureVector": [("nodes", 1, "FeatureVector.FeatureNode", True)],
    "Pose": [("rotation", 1, "float", True), ("translation", 2, "float", True)],
    "ConnectedKeyFrame": [("id", 1, "uint64", False), ("weight", 2, "int32", False)],
    "KeyFrameData": [("id", 1, "uint64", False), ("max_u", 2, "float", False), ("max_v", 3, "float", False), ("min_u", 4, "float", False),
                     ("min_v", 5, "float", False), ("keypoints", 6, "KeyPoint", True), ("right_u", 7, "float", True), ("depths", 8, "float", True),
                     ("descriptors", 9, "Descriptor", True), ("bow_vector", 10, "BowVector", False), ("feature_vector", 11, "FeatureVector", False),
                     ("pose", 12, "Pose", False), ("connected_kfs", 13, "ConnectedKeyFrame", True), ("children_ids", 14, "uint64", True),
                     ("loop_edges", 15, "uint64", True), ("map_points", 16, "int64", True)],
    "KeyFrameList": [("next_id", 1, "uint64", False), ("scale_factors", 2, "float", True), ("keyframes", 3, "KeyFrameData", True)],
}

_classes = None


def _add_fields(msg, fields):
    for name, number, typ, repeated in fields:
        f = msg.field.add(name=name, number=number, label=F.LABEL_REPEATED if repeated else F.LABEL_OPTIONAL)
        if isinstance(typ, tuple):  # map<k, v> == repeated nested entry message with map_entry = true
            entry = msg.nested_type.add(name=name.capitalize() + "Entry")
            entry.options.map_entry = True
            entry.field.add(name="key", number=1, label=F.LABEL_OPTIONAL, type=TYPES[typ[1]])
            entry.field.add(name="value", number=2, label=F.LABEL_OPTIONAL, type=TYPES[typ[2]])
            f.label, f.type, f.type_name = F.LABEL_REPEATED, F.TYPE_MESSAGE, ".orbslam2_restated." + msg.name + "." + entry.name
        elif typ in TYPES:
            f.type = TYPES[typ]
        else:
            f.type, f.type_name = F.TYPE_MESSAGE, ".orbslam2_restated." + typ


def messages():
    """-> dict name -> message class (package orbslam2_restated so it cannot clash with a real generated module)"""
    global _classes
    if _classes is None:
        fdp = descriptor_pb2.FileDescriptorProto(name="orbx_keyframe_restated.proto", package="orbslam2_restated", syntax="proto3")
        top = {}
        for full, fields in SCHEMA.items():
            if "." in full:
                continue
            top[full] = fdp.message_type.add(name=full)
        for full, fields in SCHEMA.items():
            if "." in full:
                outer, inner = full.split(".")
                nested = top[outer].nested_type.add(name=inner)
                _add_fields(nested, fields)
        for full, fields in SCHEMA.items():
            if "." not in full:
                _add_fields(top[full], fields)
        pool = descriptor_pool.DescriptorPool()
        pool.Add(fdp)
        _classes = {n: message_factory.GetMessageClass(pool.FindMessageTypeByName("orbslam2_restated." + n)) for n in SCHEMA}
    return _classes


def parse_proto_text(text: str):
    """Minimal .proto reader for the reference's file: -> the same structure as SCHEMA"""
    text = re.sub(r"//[^\n]*", "", text)
    out, stack = {}, []
    for tok in re.finditer(r"message\s+(\w+)\s*\{|\}|((repeated)\s+)?(map\s*<\s*(\w+)\s*,\s*(\w+)\s*>|[\w.]+)\s+(\w+)\s*=\s*(\d+)\s*;", text):
        if tok.group(1):
            stack.append(tok.group(1))
            out[".".join(stack)] = []
        elif tok.group(0) == "}":
            if stack:
                stack.pop()
        else:
            typ = ("map", tok.group(5), tok.group(6)) if tok.group(5) else tok.group(4)
            if not isinstance(typ, tuple) and typ not in TYPES:
                cands = [k for k in out if k == typ or k.endswith("." + typ)]  # nested messages are referenced by their short name
                typ = cands[0] if cands else typ
            out[".".join(stack)].append((tok.group(7), int(tok.group(8)), typ, bool(tok.group(3))))
    return out
