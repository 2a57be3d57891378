"""Extracts the golden NTT vectors of the reference's own test-suite
(ring/ntt_test.go:10-89 of tuneinsight/lattigo v6.2.0: six vectors, N in {16..512}, two
59-bit limbs each) into tests/golden/ntt_vectors.json.

    python tests/golden/extract_ntt_vectors.py <lattigo checkout>/ring/ntt_test.go

The tests read only the JSON file. Only numeric literals are extracted -- no reference code is copied.
"""
import json
import os
import re
import sys

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ntt_vectors.json")


def main():
    if len(sys.argv) != 2:
        sys.exit("usage: python tests/golden/extract_ntt_vectors.py <lattigo v6.2.0 checkout>/ring/ntt_test.go")
    src = open(sys.argv[1]).read()
    body = src[src.index("var testVector"):]
    body = body[: body.index("\n}\n") + 3]
    # each vector: N, Qis, poly (2 rows), polyNTT (2 rows)
    vectors = []
    # split on the top-level entries: "\t{\n\t\tN,\n"
    for m in re.finditer(r"\n\t\{\n\t\t(\d+),\n\t\t\[\]uint64\{([^}]*)\},\n\t\tPoly\{\[\]\[\]uint64\{(.*?)\n\t\t\}\},\n\t\tPoly\{\[\]\[\]uint64\{(.*?)\n\t\t\}\},\n\t\},", body, re.S):
        N = int(m.group(1))
        qis = [int(x) for x in re.findall(r"\d+", m.group(2))]
        rows = lambda t: [[int(x) for x in re.findall(r"\d+", r)] for r in re.findall(r"\{([^{}]*)\}", t)]
        poly, poly_ntt = rows(m.group(3)), rows(m.group(4))
        assert len(poly) == len(qis) == len(poly_ntt) and all(len(r) == N for r in poly + poly_ntt), (N, [len(r) for r in poly + poly_ntt])
        vectors.append({"N": N, "Qis": qis, "poly": poly, "polyNTT": poly_ntt})
    assert len(vectors) == 6, len(vectors)
    json.dump({"source": "tuneinsight/lattigo v6.2.0 ring/ntt_test.go:10-89", "vectors": vectors}, open(OUT, "w"))
    print("wrote", OUT, [v["N"] for v in vectors])


if __name__ == "__main__":
    main()
