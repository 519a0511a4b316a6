"""The hand-built protobuf descriptors (nucliadb_b200/nidx_protos.py: there is no protoc here) against the reference's own .proto files
(nidx/nidx_protos/*.proto), as parsed into tests/golden/reference_facts.json by tests/golden/make_reference_facts.py: every field
declared by hand must exist in the reference message with the same number, type and cardinality -- the wire compatibility of the
outer boundary (NidxSearcher.Search / NidxApi.NewShard / IndexMessage)."""
import json
import os

from google.protobuf import descriptor_pb2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_facts.json")))["nidx_protos"]
_F = descriptor_pb2.FieldDescriptorProto
_SCALAR = {_F.TYPE_STRING: "string", _F.TYPE_BYTES: "bytes", _F.TYPE_INT32: "int32", _F.TYPE_INT64: "int64", _F.TYPE_UINT32: "uint32",
           _F.TYPE_UINT64: "uint64", _F.TYPE_FLOAT: "float", _F.TYPE_BOOL: "bool", _F.TYPE_DOUBLE: "double"}


def test_hand_built_descriptors_match_the_reference_protos():
    from nucliadb_b200 import nidx_protos as P

    ref_msgs, ref_enums = REF["messages"], REF["enums"]
    checked = 0

    def short(type_name, scope):
        return type_name.lstrip(".")

    def check_message(md, full):
        nonlocal checked
        assert full in ref_msgs, f"message {full} is not in the reference"
        ref = ref_msgs[full]
        for fd in md.field:
            assert fd.name in ref, f"{full}.{fd.name} is not in the reference"
            num, typ, rep = ref[fd.name]
            assert fd.number == num, (full, fd.name, fd.number, num)
            is_map = fd.type == _F.TYPE_MESSAGE and any(n.name == fd.type_name.split(".")[-1] and n.options.map_entry for n in md.nested_type)
            if is_map:
                entry = next(n for n in md.nested_type if n.name == fd.type_name.split(".")[-1])
                kt, vt = entry.field[0], entry.field[1]
                want_k = _SCALAR[kt.type]
                want_v = _SCALAR.get(vt.type) or vt.type_name.split(".")[-1]
                assert typ.startswith("map<") and typ[4:-1].split(",")[0] == want_k and typ[4:-1].split(",")[1].split(".")[-1] == want_v, (full, fd.name, typ)
            else:
                assert (fd.label == _F.LABEL_REPEATED) == rep, (full, fd.name, "repeated")
                if fd.type in _SCALAR:
                    if fd.type == _F.TYPE_INT32 and typ not in _SCALAR.values():
                        # an enum (of this package, unqualified, or of another file), carried as its int32 wire type
                        assert typ.startswith("utils.") or any(e == typ or e.endswith("." + typ) for e in ref_enums), (full, fd.name, typ)
                    else:
                        assert typ == _SCALAR[fd.type], (full, fd.name, typ, _SCALAR[fd.type])
                elif fd.type == _F.TYPE_ENUM and not fd.type_name:
                    pass
                elif fd.type in (_F.TYPE_MESSAGE, _F.TYPE_ENUM):
                    assert typ.split(".")[-1] == fd.type_name.split(".")[-1], (full, fd.name, typ, fd.type_name)
            checked += 1
        for nested in md.nested_type:
            if not nested.options.map_entry:
                check_message(nested, full + "." + nested.name)

    seen_files = 0
    for fname in ("nidx_protos/noderesources.proto", "nidx_protos/nodereader.proto", "nidx_protos/nodewriter.proto", "nidx_protos/noderesources_shards.proto"):
        fdp = descriptor_pb2.FileDescriptorProto()
        P.POOL.FindFileByName(fname).CopyToProto(fdp)
        seen_files += 1
        for md in fdp.message_type:
            check_message(md, fdp.package + "." + md.name)
        for ed in fdp.enum_type:
            full = fdp.package + "." + ed.name
            assert full in ref_enums, full
            for v in ed.value:
                assert ref_enums[full].get(v.name) == v.number, (full, v.name)
    assert seen_files == 4 and checked > 80
    # the two rpc paths
    assert REF["services"]["nidx.NidxSearcher"]["Search"] == ["nodereader.SearchRequest", "nodereader.SearchResponse"]
    assert REF["services"]["nidx.NidxApi"]["NewShard"] == ["nodewriter.NewShardRequest", "noderesources.ShardCreated"]
    assert P.SEARCH_METHOD == "/nidx.NidxSearcher/Search" and P.NEW_SHARD_METHOD == "/nidx.NidxApi/NewShard"
