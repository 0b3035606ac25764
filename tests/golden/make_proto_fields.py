"""Generate tests/golden/auron_proto_fields.json, the message / field / enum table of the reference's
`native-engine/auron-serde/proto/auron.proto` that tests/test_proto_compat.py checks blaze_b200/proto.py against:
`python tests/golden/make_proto_fields.py <path to auron.proto>`."""
import json
import os
import re
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "auron_proto_fields.json")
SOURCE = "kwai/blaze (Apache Auron) @ d1eaef148a58, native-engine/auron-serde/proto/auron.proto"


def parse(path):
    """{"messages": {message: {field: [number, type, repeated]}}, "enums": {enum: {value: number}}}"""
    text = re.sub(r"//.*", "", open(path).read())
    msgs = {}
    for m in re.finditer(r"message\s+(\w+)\s*\{", text):
        name, i, depth = m.group(1), m.end(), 1
        j = i
        while depth:
            depth += {"{": 1, "}": -1}.get(text[j], 0)
            j += 1
        body = text[i:j - 1]
        fields = {}
        for f in re.finditer(r"(repeated\s+)?([\w.]+)\s+(\w+)\s*=\s*(\d+)\s*;", body):
            fields[f.group(3)] = [int(f.group(4)), f.group(2), bool(f.group(1))]
        msgs[name] = fields
    enums = {}
    for m in re.finditer(r"enum\s+(\w+)\s*\{([^}]*)\}", text):
        enums[m.group(1)] = {a: int(b) for a, b in re.findall(r"(\w+)\s*=\s*(\d+)\s*;", m.group(2))}
    return {"source": SOURCE, "messages": msgs, "enums": enums}


if __name__ == "__main__":
    with open(OUT, "w") as f:
        json.dump(parse(sys.argv[1]), f, indent=1, sort_keys=True)
        f.write("\n")
