"""Facts the tests compare this project against, read from a checkout of the original nucliadb sources: the HNSW and RaBitQ
constants and the search-cost model of nidx_vector, the segment file names, the messages, enums and rpcs of nidx_protos/*.proto
and the method signatures of nidx_binding.pyi.  Output: tests/golden/reference_facts.json (committed), read by
tests/test_constants_vs_reference.py, tests/test_protos_vs_reference.py and tests/test_host_logic.py.

    python tests/golden/make_reference_facts.py <nucliadb checkout>
"""
import ast
import json
import os
import re
import sys

HERE = os.path.dirname(os.path.abspath(__file__))


def rust_const(src, name):
    m = re.search(rf"const\s+{name}\s*:\s*\w+\s*=\s*([0-9.]+)\s*;", src)
    assert m, name
    return float(m.group(1)) if "." in m.group(1) else int(m.group(1))


def rust_str_const(src, name):
    m = re.search(rf'const\s+{name}\s*:\s*&str\s*=\s*"([^"]+)"', src)
    assert m, name
    return m.group(1)


def vector_facts(ref):
    src = lambda p: open(os.path.join(ref, "nidx", "nidx_vector", "src", p)).read()
    params, rabitq, segment = src("hnsw/params.rs"), src("vector_types/rabitq.rs"), src("segment.rs")
    prune = re.search(r"fn prune_m\(m: usize\) -> usize \{\s*m \* (\d+) / (\d+)", params)
    body = segment[segment.index("fn use_hnsw("):]
    body = body[: body.index("\n}\n")]
    full = re.findall(r"full_cost = (\d+);", body)
    search = re.findall(r"search_mult = ([^;]+);", body)
    rerank = re.findall(r"rerank_mult = ([^;]+);", body)
    rq_search = re.fullmatch(r"rabitq::RERANKING_FACTOR \* (\d+) / (\d+)", search[0])
    rq_rerank = re.fullmatch(r"rabitq::RERANKING_FACTOR / (\d+)", rerank[0])
    log = re.search(r"\(\(total_nodes as f32\)\.ln\(\) - ([0-9.]+)\)\.powi\((\d+)\)", body)
    assert prune and len(full) == len(search) == len(rerank) == 2 and rq_search and rq_rerank and log
    files = {"hnsw/disk/v2.rs": ("GRAPH_FILENAME", "EDGES_FILENAME"), "data_store/v2/vector_store.rs": ("FILENAME",),
             "data_store/v2/quant_vector_store.rs": ("FILENAME",), "data_store/v2/paragraph_store.rs": ("FILENAME_DATA", "FILENAME_POS")}
    return {
        "hnsw_params": {**{c: rust_const(params, c) for c in ("M", "M_MAX", "M_MAX_0", "EF_CONSTRUCTION", "EF_SEARCH")},
                        "prune_m_ratio": [int(prune.group(1)), int(prune.group(2))]},
        "rabitq": {c: rust_const(rabitq, c) for c in ("EPSILON", "RERANKING_FACTOR", "RERANKING_LIMIT")},
        "use_hnsw": {"with_rabitq": {"full_cost": int(full[0]), "search_mult_of_reranking_factor": [int(rq_search.group(1)), int(rq_search.group(2))],
                                     "rerank_divisor_of_reranking_factor": int(rq_rerank.group(1))},
                     "without_rabitq": {"full_cost": int(full[1]), "search_mult": int(search[1]), "rerank_mult": int(rerank[1])},
                     "log_offset": float(log.group(1)), "log_power": int(log.group(2))},
        "segment_file_names": {f"{path}:{c}": rust_str_const(src(path), c) for path, consts in files.items() for c in consts},
    }


def parse_proto(path):
    """-> ({full message name: {field: (number, type, repeated)}}, {full enum name: {value name: number}},
    {full service name: {rpc: (request type, response type)}}); handles nesting, oneof, map<>."""
    text = re.sub(r"//[^\n]*", "", open(path).read())
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    pkg = re.search(r"\bpackage\s+([\w.]+)\s*;", text).group(1)
    services = {}
    for name, body in re.findall(r"\bservice\s+(\w+)\s*\{((?:[^{}]|\{[^{}]*\})*)\}", text):
        rpcs = re.findall(r"rpc\s+(\w+)\s*\(\s*(?:stream\s+)?([\w.]+)\s*\)\s*returns\s*\(\s*(?:stream\s+)?([\w.]+)\s*\)", body)
        services[f"{pkg}.{name}"] = {r: (req, resp) for r, req, resp in rpcs}
    tokens = re.findall(r"[{};=<>,]|[\w.]+|\"[^\"]*\"|\[[^\]]*\]", text)
    msgs, enums = {}, {}
    stack = []          # [(kind, name)]
    i = 0
    while i < len(tokens):
        t = tokens[i]
        if t in ("message", "enum", "oneof", "service") and tokens[i + 2] == "{":
            name = tokens[i + 1]
            if t == "oneof":
                stack.append(("oneof", None))
            else:
                scope = ".".join([pkg] + [n for k, n in stack if k == "message"] + [name])
                stack.append((t, name))
                if t == "message":
                    msgs[scope] = {}
                elif t == "enum":
                    enums[scope] = {}
            i += 3
            continue
        if t == ";":
            i += 1
            continue
        if t == "{":                 # any other block (rpc bodies, option blocks)
            stack.append(("block", None))
            i += 1
            continue
        if t == "}":
            stack.pop()
            i += 1
            continue
        kinds = [k for k, _ in stack]
        if kinds and kinds[-1] == "enum" and i + 2 < len(tokens) and tokens[i + 1] == "=":
            scope = ".".join([pkg] + [n for k, n in stack if k in ("message", "enum")])
            enums[scope][t] = int(tokens[i + 2])
            i += 3
            continue
        if kinds and kinds[-1] in ("message", "oneof") and t not in ("option", "reserved", "extensions"):
            scope = ".".join([pkg] + [n for k, n in stack if k == "message"])
            rep = False
            j = i
            if tokens[j] in ("repeated", "optional"):
                rep = tokens[j] == "repeated"
                j += 1
            if tokens[j] == "map" and tokens[j + 1] == "<":
                ktype, vtype, name, num = tokens[j + 2], tokens[j + 4], tokens[j + 6], int(tokens[j + 8])
                msgs[scope][name] = (num, f"map<{ktype},{vtype}>", True)
                i = j + 9
            elif j + 3 < len(tokens) and tokens[j + 2] == "=":
                msgs[scope][tokens[j + 1]] = (int(tokens[j + 3]), tokens[j], rep)
                i = j + 4
            else:
                i += 1
                continue
            while i < len(tokens) and tokens[i] != ";" and tokens[i] not in ("}", "{"):
                i += 1
            continue
        i += 1
    return msgs, enums, services


def proto_facts(ref):
    d = os.path.join(ref, "nidx", "nidx_protos")
    msgs, enums, services = {}, {}, {}
    for f in sorted(os.listdir(d)):
        if f.endswith(".proto"):
            m, e, s = parse_proto(os.path.join(d, f))
            msgs.update(m)
            enums.update(e)
            services.update(s)
    return {"messages": msgs, "enums": enums, "services": services}


def binding_facts(ref):
    pyi = os.path.join(ref, "nidx", "nidx_binding", "nidx_binding.pyi")
    cls = next(n for n in ast.parse(open(pyi).read()).body if isinstance(n, ast.ClassDef) and n.name == "NidxBinding")
    return {"NidxBinding": {"methods": {n.name: [a.arg for a in n.args.args] for n in cls.body if isinstance(n, ast.FunctionDef)},
                            "attributes": [n.target.id for n in cls.body if isinstance(n, ast.AnnAssign)]}}


def main():
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    ref = sys.argv[1]
    facts = {"generator": "tests/golden/make_reference_facts.py", "nidx_vector": vector_facts(ref), "nidx_protos": proto_facts(ref),
             "nidx_binding": binding_facts(ref)}
    with open(os.path.join(HERE, "reference_facts.json"), "w") as f:
        json.dump(facts, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
