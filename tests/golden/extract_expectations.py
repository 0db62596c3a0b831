#!/usr/bin/env python
"""Transcribes the reference's committed test expectations (the golden vectors of this path) into
tests/golden/reference_expectations.json.

Run against a checkout of the reference:

    python tests/golden/extract_expectations.py <dune-hdd checkout>

The tests only read the JSON.  Every vector keeps the file and line it came from.  Keys: "<file stem>" ->
"<partitioning or '-'>" -> "<mu,mu_bar,mu_hat or '-'>" -> "<type>" -> {values, line}.
Only the four expectation files that are reproducible offline are transcribed (SURVEY.md 8c): the SPE10 ones need
perm_case1.dat, which the reference does not ship.
"""
import json
import os
import re
import sys

FILES = ["linearelliptic-swipdg-expectations_esv2007_2daluconform.cxx",
         "linearelliptic-swipdg-expectations_esv2007_2dsgrid.cxx",
         "linearelliptic-block-swipdg-expectations_esv2007_2daluconform.cxx",
         "linearelliptic-block-swipdg-expectations_os2014_2daluconform.cxx"]


def parse(path):
    out = {}
    part, mus, types = "-", "-", []
    for no, raw in enumerate(open(path), 1):
        line = raw.split("//")[0]
        m = re.search(r'partitioning\(\) == "(\[[^"]*\])"', line)
        if m:
            part, mus = m.group(1), "-"
        m = re.search(r"mu == ([0-9.]+) && mu_bar == ([0-9.]+) && mu_hat == ([0-9.]+)", line)
        if m:
            mus = ",".join(m.groups())
        m = re.findall(r'type(?:\.substr\(0, \d+\))? == "([^"]+)"', line)
        if m:
            types = m
        m = re.search(r"return \{([^}]*)\};", line)
        if m and types:
            vals = [float(v) for v in m.group(1).split(",") if v.strip()]
            for t in types:
                out.setdefault(part, {}).setdefault(mus, {})[t] = {"values": vals, "line": no}
            types = []
    return out


def main():
    if len(sys.argv) != 2:
        sys.exit("usage: %s <dune-hdd checkout>" % sys.argv[0])
    ref = sys.argv[1]
    data = {"_source": "tobiasleibner/dune-hdd test/*.cxx, transcribed by tests/golden/extract_expectations.py"}
    for f in FILES:
        data[f[:-4]] = parse(os.path.join(ref, "test", f))
    dst = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_expectations.json")
    with open(dst, "w") as fh:
        json.dump(data, fh, indent=1, sort_keys=True)
    print("wrote", dst)


if __name__ == "__main__":
    main()
