"""Checks that every reference citation of the form `<path>.py:<line>[-<line>]` in the repo's sources and docs names a
reference file (SpeechT5 tree first, sibling trees second) and a line range inside it. The line counts of the cited
reference files are stored in tests/golden/ref_pins.json (`reference_line_counts`, written from the reference by
tests/golden/make_golden_ref_pins.py, which must be re-run when a citation names a file not listed there). Prints the
broken ones and exits 1 if any.
usage: python tools/check_citations.py [-v]"""
import glob
import json
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PINS = os.path.join(ROOT, "tests", "golden", "ref_pins.json")
ALIAS = {"legacy_ddp.py": "fairseq/distributed/legacy_distributed_data_parallel.py"}  # SURVEY.md:15 shorthand
PAT = re.compile(r"([A-Za-z0-9_./-]+\.py):(\d+)(?:-(\d+))?")
UNCHECKED = ("SURVEY.md", "PAPERS.md", "SNIPPETS.md", "BASELINE.md", "VERDICT.md", "ADVICE.md")


def citations(root=ROOT):
    """(reference path, first line, last line, citing file, its line number, citation text) of every citation in the
    sources and docs that does not name a file of this repository."""
    files = [p for pat in ("*.md", "include/*.h", "oracle/*.py", "speecht5_b200/**/*.py", "speecht5_b200/csrc/*",
                           "tests/**/*.py", "bench.py", "__graft_entry__.py")
             for p in glob.glob(os.path.join(root, pat), recursive=True)]
    out = []
    for f in sorted(set(files)):
        if os.path.basename(f) in UNCHECKED:
            continue
        for ln, line in enumerate(open(f, errors="ignore"), 1):
            for m in PAT.finditer(line):
                path, a, b = m.group(1), int(m.group(2)), int(m.group(3) or m.group(2))
                if "..." in path:
                    continue
                path = path.lstrip("./")
                if path.split("/", 2)[:2] == ["root", "reference"]:  # an absolute path into the reference checkout
                    path = path.split("/", 2)[2]
                path = ALIAS.get(path, path)
                if os.path.exists(os.path.join(root, path)):  # a citation of this repo's own file
                    continue
                out.append((path, a, b, f, ln, m.group(0)))
    return out


def index(paths):
    by_tail = {}
    for rel in paths:
        parts = rel.split("/")
        for i in range(len(parts)):
            by_tail.setdefault("/".join(parts[i:]), []).append(rel)
    return by_tail


def main():
    verbose = "-v" in sys.argv
    with open(PINS, encoding="utf-8") as fh:
        lens = json.load(fh)["reference_line_counts"]
    by_tail = index(lens)
    bad, n = [], 0
    for path, a, b, f, ln, cite in citations():
        cands = by_tail.get(path)
        if not cands:
            bad.append((f, ln, cite, "no such reference file"))
            continue
        n += 1
        cands = sorted(cands, key=lambda p: (0 if p.startswith("SpeechT5/") else 1, len(p)))
        if not any(a <= b <= lens[c] for c in cands):
            bad.append((f, ln, cite, f"line range outside the file ({lens[cands[0]]} lines)"))
        elif verbose:
            print("ok", cite)
    for f, ln, cite, why in bad:
        print(f"{f[len(ROOT) + 1:]}:{ln}: {cite}: {why}")
    print(f"{n} citations checked, {len(bad)} broken")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
