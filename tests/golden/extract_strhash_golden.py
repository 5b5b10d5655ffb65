"""Transcribe the StrHashMap known answers of the reference's own Go test into a JSON fixture (data only).

Run in the build container (needs /root/reference):   python tests/golden/extract_strhash_golden.py
Writes tests/golden/strhash_kat.json, which is committed; the GPU box and the CPU test-suite read only the JSON.

Source (path relative to /root/reference):
  pkg/common/hashmap/strhashmap_test.go:60-136   TestIterator: StrHashMap ids with / without hasNull, and with every even row NULL
"""
import json
import os
import re

from extract_goldens import OUT, REF, _func_body


def strhash_kats():
    """TestIterator: six key columns with value i in row i (char: strconv.Itoa(i)), Rows rows; StrHashMap with and without hasNull, the third
    case with every even row NULL in every column.  Expected ids of Insert (Find returns the same)."""
    path = "pkg/common/hashmap/strhashmap_test.go"
    src = open(os.path.join(REF, path)).read()
    rows = int(re.search(r"^\s*Rows\s*=\s*(\d+)", src, re.M).group(1))
    body = _func_body(src, "TestIterator")
    widths = {"int8": 1, "int16": 2, "int32": 4, "int64": 8, "decimal64": 8, "char": 0, "varchar": 0}
    cases = []
    for blk in body.split("mp.Free()")[:-1]:
        has_null = re.search(r"NewStrHashMap\((true|false)", blk).group(1) == "true"
        types_ = re.findall(r"types\.New\(types\.T_(\w+),", blk)
        with_null = "newVectorsWithNull(" in blk
        want = [int(x) for x in re.search(r"require\.Equal\(t, \[\]uint64\{([^}]*)\}, vs\[:Rows\]\)", blk).group(1).split(",")]
        cases.append({"has_null": has_null, "columns": [{"type": t, "width": widths[t]} for t in types_],
                      "values": list(range(rows)), "null_rows": [j for j in range(rows) if j % 2 == 0] if with_null else [],
                      "want_ids": want})
    assert len(cases) == 3, cases
    return {"_source": path + ":60-136", "_values": "row i holds i in every fixed column and strconv.Itoa(i) in the char column; "
            "null_rows are NULL in every column", "rows": rows, "cases": cases}


def main():
    data = strhash_kats()
    with open(os.path.join(OUT, "strhash_kat.json"), "w") as f:
        json.dump(data, f, indent=1)
    print("strhash_kat", len(data["cases"]))


if __name__ == "__main__":
    main()
