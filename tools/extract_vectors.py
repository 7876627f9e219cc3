#!/usr/bin/env python3
"""Extracts the reference's own known-answer vectors into tests/golden/reference_vectors.json.

Usage: tools/extract_vectors.py <libgoldilocks source tree> (reads its test/*.inc.cxx).  The JSON it writes is
committed; the tests read only the JSON.

Sources (SURVEY.md section 8(c)):
  test/vectors.inc.cxx:3-29       RFC 7748 X448 iterated ladder after 1 / 1000 / 10^6 iterations
  test/vectors.inc.cxx:34-43      Elligator pathological input
  test/vectors.inc.cxx:46-751     RFC 8032 Ed448 x 11 (sk, pk, message, prehash flag, context, signature)
  test/elligator_vectors.inc.cxx  16 decaf encodings of i*B, 16 Elligator input -> encoding pairs
"""
import json, os, re, sys

if len(sys.argv) != 2:
    sys.exit(__doc__)
REF = sys.argv[1]
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden", "reference_vectors.json")


def strip_comments(t):
    t = re.sub(r"/\*.*?\*/", "", t, flags=re.S)
    return re.sub(r"//[^\n]*", "", t)


def array_body(text, name):
    """text of the brace-balanced initialiser that follows `name ... = {`"""
    m = re.search(re.escape(name) + r"[^;{]*?=\s*\{", text, flags=re.S)
    assert m, name
    i = m.end() - 1
    depth = 0
    for j in range(i, len(text)):
        if text[j] == "{":
            depth += 1
        elif text[j] == "}":
            depth -= 1
            if depth == 0:
                return text[i + 1:j]
    raise ValueError(name)


def hexbytes(s):
    return bytes(int(x, 16) for x in re.findall(r"0x([0-9a-fA-F]{1,2})", s))


def rows(body):
    out, depth, start = [], 0, None
    for j, ch in enumerate(body):
        if ch == "{":
            if depth == 0:
                start = j
            depth += 1
        elif ch == "}":
            depth -= 1
            if depth == 0:
                out.append(hexbytes(body[start:j]))
    return out


def blocks(text, name):
    """entries of a `Block name[] = { Block(arr[i],len), Block(NULL,0) ... }` table -> [(arr, i, len) | None]"""
    body = array_body(text, "::" + name + "[]")
    out = []
    for m in re.finditer(r"Block\(\s*(NULL|(\w+)\[(\d+)\])\s*,\s*(\d+)\s*\)", body):
        out.append(None if m.group(1) == "NULL" else (m.group(2), int(m.group(3)), int(m.group(4))))
    return out


def main():
    v = strip_comments(open(os.path.join(REF, "test", "vectors.inc.cxx")).read())
    e = strip_comments(open(os.path.join(REF, "test", "elligator_vectors.inc.cxx")).read())
    arrays = {n: rows(array_body(v, n + "[]")) for n in
              ("ed448_eddsa_sk", "ed448_eddsa_pk", "ed448_eddsa_message", "ed448_eddsa_context", "ed448_eddsa_sig")}
    pre = re.findall(r"true|false", array_body(v, "::eddsa_prehashed[]"))
    tabs = {n: blocks(v, n) for n in ("eddsa_sk", "eddsa_pk", "eddsa_message", "eddsa_context", "eddsa_sig")}
    n = len(tabs["eddsa_pk"])
    assert n == 11 and len(pre) == 11

    def get(tab, t, arrname):
        ent = tabs[tab][t]
        if ent is None:
            return b""
        arr, i, ln = ent
        assert arr == arrname
        data = arrays[arr][i]
        assert len(data) >= ln or ln == 0, (tab, t, len(data), ln)
        return data[:ln]

    eddsa = []
    for t in range(n):
        eddsa.append(dict(sk=get("eddsa_sk", t, "ed448_eddsa_sk").hex(), pk=get("eddsa_pk", t, "ed448_eddsa_pk").hex(),
                          msg=get("eddsa_message", t, "ed448_eddsa_message").hex(), prehashed=pre[t] == "true",
                          context=get("eddsa_context", t, "ed448_eddsa_context").hex(), sig=get("eddsa_sig", t, "ed448_eddsa_sig").hex()))
    out = dict(
        source="otrv4/libgoldilocks test/vectors.inc.cxx + test/elligator_vectors.inc.cxx (RFC 7748, RFC 8032, SAGE-computed decaf/Elligator)",
        x448_iter={"1": hexbytes(array_body(v, "rfc7748_1[56]")).hex(), "1000": hexbytes(array_body(v, "rfc7748_1000[56]")).hex(),
                   "1000000": hexbytes(array_body(v, "rfc7748_1000000[56]")).hex()},
        elli_patho=hexbytes(array_body(v, "elli_patho_448[56]")).hex(),
        eddsa=eddsa,
        base_multiples=[r.hex() for r in rows(array_body(e, "base_multiples<Ed448Goldilocks>::values"))],
        elligator_inputs=[r.hex() for r in rows(array_body(e, "elligator_examples<Ed448Goldilocks>::inputs"))],
        elligator_outputs=[r.hex() for r in rows(array_body(e, "elligator_examples<Ed448Goldilocks>::outputs"))],
    )
    assert len(out["base_multiples"]) == 16 and len(out["elligator_inputs"]) == 16 and len(out["elligator_outputs"]) == 16
    assert all(len(x) == 112 for x in out["base_multiples"] + out["elligator_inputs"] + out["elligator_outputs"])
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", os.path.normpath(OUT), "eddsa cases:", len(eddsa), "msg lens:", [len(c["msg"]) // 2 for c in eddsa])


if __name__ == "__main__":
    main()
