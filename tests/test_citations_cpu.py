"""Every `file.rs:line` / `file.py:line` citation of the reference in the headers, docs and oracle must point at an existing
line of the reference. The line counts of the reference's files are stored in tests/golden/reference_line_counts.json
(tests/ref_shim/make_ref_fixtures.py)."""
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LINE_COUNTS = os.path.join(ROOT, "tests", "golden", "reference_line_counts.json")
FILES = ["include/sdb200.h", "DESIGN.md", "INTEGRATION.md", "oracle/sd_oracle.py", "stable_diffusion_burn_b200/topology.py",
         "stable_diffusion_burn_b200/tokenizer.py", "stable_diffusion_burn_b200/dumpdir.py", "stable_diffusion_burn_b200/pipeline.py",
         "stable_diffusion_burn_b200/csrc/dumpdir.cu", "stable_diffusion_burn_b200/csrc/model_build.cu", "rust/sdb200_ffi.rs",
         "stable_diffusion_burn_b200/mpk.py", "tools/sample.py", "tests/ref_shim/run_reference.py", "tests/test_ref_pin_cpu.py"]
CITE = re.compile(r"((?:[A-Za-z_]+/)+[A-Za-z_]+\.(?:rs|py)):(\d+)(?:-(\d+))?")


def test_cited_lines_exist():
    with open(LINE_COUNTS) as f:
        lengths = json.load(f)  # path relative to the reference checkout -> number of lines
    bad, checked = [], 0
    for rel in FILES:
        text = open(os.path.join(ROOT, rel), encoding="utf-8").read()
        for m in CITE.finditer(text):
            path, lo, hi = m.group(1), int(m.group(2)), int(m.group(3) or m.group(2))
            if path.startswith(("tests/", "oracle/", "stable_diffusion_burn_b200/", "tools/", "profiles/", "csrc/")):
                continue  # a citation of this repo
            hits = [f for f in lengths if ("/" + f).endswith("/" + path)]
            if len(hits) != 1:
                bad.append(f"{rel}: {m.group(0)} -> {len(hits)} candidate files")
                continue
            n = lengths[hits[0]]
            checked += 1
            if not (1 <= lo <= hi <= n):
                bad.append(f"{rel}: {m.group(0)} beyond the {n} lines of {hits[0]}")
    assert checked > 100, checked
    assert not bad, "\n".join(bad[:40])
