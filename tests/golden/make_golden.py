#!/usr/bin/env python3
"""Extract the reference's own search vectors into a JSON fixture.

Reads tests/aho_corasick_crate_test.rs of a daachorse 4.0.0 checkout (the 136 ``SearchTest``
vectors at :63-382, the collections at :50-59 and the 12 test configurations at :537-645) and
writes tests/golden/search_tests.json.  Only *data* (names, patterns, haystacks, expected
``(value, start, end)`` triples) is extracted; no reference source code is copied.  The tests
read the JSON file only, so they need no copy of the crate:

    python tests/golden/make_golden.py <daachorse checkout>
"""
import json
import os
import re
import sys

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "search_tests.json")

GROUPS = ["BASICS", "STANDARD", "LEFTMOST", "LEFTMOST_FIRST", "LEFTMOST_LONGEST",
          "NON_OVERLAPPING", "OVERLAPPING"]


def rust_str(lit):
    """Decode a Rust string literal body (the fixtures only use plain text)."""
    assert "\\" not in lit, lit
    return lit


def split_top(s):
    """Split on top-level commas."""
    parts, depth, cur, in_str = [], 0, "", False
    for ch in s:
        if in_str:
            cur += ch
            if ch == '"':
                in_str = False
            continue
        if ch == '"':
            in_str = True
            cur += ch
        elif ch in "([":
            depth += 1
            cur += ch
        elif ch in ")]":
            depth -= 1
            cur += ch
        elif ch == "," and depth == 0:
            parts.append(cur.strip())
            cur = ""
        else:
            cur += ch
    if cur.strip():
        parts.append(cur.strip())
    return parts


def parse_group(src, name):
    m = re.search(r"const %s: &'static \[SearchTest\] = &\[" % name, src)
    assert m, name
    i = m.end()
    tests = []
    while True:
        j = src.find("t!(", i)
        end_group = src.find("];", i)
        if j < 0 or (end_group >= 0 and end_group < j):
            break
        # balanced scan from the '(' of t!(
        k = j + 2
        depth, in_str = 0, False
        while True:
            ch = src[k]
            if in_str:
                if ch == '"':
                    in_str = False
            elif ch == '"':
                in_str = True
            elif ch == "(":
                depth += 1
            elif ch == ")":
                depth -= 1
                if depth == 0:
                    break
            k += 1
        body = src[j + 3:k]
        tname, pats, hay, matches = split_top(body)
        pats = [rust_str(x) for x in re.findall(r'"((?:[^"\\]|\\.)*)"', pats)]
        hay = rust_str(re.fullmatch(r'"((?:[^"\\]|\\.)*)"', hay).group(1))
        triples = [[int(a), int(b), int(c)]
                   for a, b, c in re.findall(r"\((\d+),\s*(\d+),\s*(\d+)\)", matches)]
        tests.append({"name": tname, "patterns": pats, "haystack": hay, "matches": triples})
        i = k + 1
    return tests


def main():
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    src = open(os.path.join(sys.argv[1], "tests", "aho_corasick_crate_test.rs"), encoding="utf-8").read()
    groups = {g: parse_group(src, g) for g in GROUPS}
    total = sum(len(v) for v in groups.values())
    assert total == 136, total
    doc = {
        "source": "daac-tools/daachorse 4.0.0 tests/aho_corasick_crate_test.rs:63-382",
        "triple_order": ["value", "start", "end"],
        "groups": groups,
        # collections, tests/aho_corasick_crate_test.rs:50-59
        "collections": {
            "AC_STANDARD_NON_OVERLAPPING": ["BASICS", "NON_OVERLAPPING", "STANDARD"],
            "AC_STANDARD_OVERLAPPING": ["BASICS", "OVERLAPPING"],
            "AC_LEFTMOST_LONGEST": ["BASICS", "NON_OVERLAPPING", "LEFTMOST", "LEFTMOST_LONGEST"],
            "AC_LEFTMOST_FIRST": ["BASICS", "NON_OVERLAPPING", "LEFTMOST", "LEFTMOST_FIRST"],
        },
        # the 12 configurations, tests/aho_corasick_crate_test.rs:537-645:
        # (variant, iterator, collection, match kind)
        "configs": [
            ["bytewise", "find_iter", "AC_STANDARD_NON_OVERLAPPING", "Standard"],
            ["bytewise", "find_stepper", "AC_STANDARD_NON_OVERLAPPING", "Standard"],
            ["bytewise", "find_overlapping_iter", "AC_STANDARD_OVERLAPPING", "Standard"],
            ["bytewise", "find_overlapping_stepper", "AC_STANDARD_OVERLAPPING", "Standard"],
            ["bytewise", "leftmost_find_iter", "AC_LEFTMOST_LONGEST", "LeftmostLongest"],
            ["bytewise", "leftmost_find_iter", "AC_LEFTMOST_FIRST", "LeftmostFirst"],
            ["charwise", "find_iter", "AC_STANDARD_NON_OVERLAPPING", "Standard"],
            ["charwise", "find_stepper", "AC_STANDARD_NON_OVERLAPPING", "Standard"],
            ["charwise", "find_overlapping_iter", "AC_STANDARD_OVERLAPPING", "Standard"],
            ["charwise", "find_overlapping_stepper", "AC_STANDARD_OVERLAPPING", "Standard"],
            ["charwise", "leftmost_find_iter", "AC_LEFTMOST_LONGEST", "LeftmostLongest"],
            ["charwise", "leftmost_find_iter", "AC_LEFTMOST_FIRST", "LeftmostFirst"],
        ],
    }
    with open(OUT, "w", encoding="utf-8") as f:
        json.dump(doc, f, indent=1, ensure_ascii=False)
        f.write("\n")
    print("wrote %s: %d vectors in %d groups" % (OUT, total, len(groups)), file=sys.stderr)


if __name__ == "__main__":
    main()
