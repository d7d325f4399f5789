#!/usr/bin/env python
"""Extract the field names (in declaration order) of the reference's BaLog structs from
<rootba checkout>/src/rootba/bal/ba_log.hpp into tests/golden/ba_log_fields.json.

    python tests/golden/make_ba_log_fields.py <rootba checkout>

The JSON is committed, so the tests do not need the reference.
The per-iteration structs become top-level columns of ba_log.json, the others live under "_static"
(src/rootba/bal/ba_log.cpp:62-150)."""
import json
import os
import re
import sys

SRC = os.path.join(sys.argv[1], "src", "rootba", "bal", "ba_log.hpp")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ba_log_fields.json")

txt = open(SRC).read()
txt = re.sub(r"//[^\n]*", "", txt)  # commented-out members must not count
structs = {}
for m in re.finditer(r"BEGIN_VISITABLES\((\w+)\);(.*?)END_VISITABLES;", txt, flags=re.S):
    name, body = m.group(1), m.group(2)
    fields = []
    for f in re.finditer(r"VISITABLE(?:_INIT|_META)?\(\s*([^,()]+(?:<[^>]*>)?)\s*,\s*(\w+)", body):
        fields.append({"type": f.group(1).strip(), "name": f.group(2)})
    structs[name] = fields
json.dump({"source": "src/rootba/bal/ba_log.hpp", "structs": structs}, open(OUT, "w"), indent=1)
print({k: len(v) for k, v in structs.items()})
