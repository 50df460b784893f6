"""Generate tests/golden/ref_harness_golden.pt and tests/golden/reference_sources.json from the UNMODIFIED reference:
the first-iteration traces oracle/ref_gpu.py records when it drives the reference on CPU (tests/test_ref_gpu_cpu.py's
tiny spec, greedy and stochastic) and the sha256 of every reference file tools/vendor_ref.py vendors.  Needs the
reference's sources:

    python tests/golden/make_ref_harness_golden.py
"""
import hashlib
import json
import os
import sys
import tempfile

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.dirname(HERE))

import vendor_ref  # noqa: E402
from test_ref_gpu_cpu import run_harness  # noqa: E402

assert os.path.isdir(vendor_ref.SRC) and vendor_ref.vendor(), f"no reference sources at {vendor_ref.SRC}"
with open(os.path.join(vendor_ref.DST, "MANIFEST.json")) as f:
    files = json.load(f)["files"]
sources = {}
for rel in sorted(files):
    with open(os.path.join(vendor_ref.SRC, rel), "rb") as fh:
        sources[rel] = hashlib.sha256(fh.read()).hexdigest()
with open(os.path.join(HERE, "reference_sources.json"), "w") as f:
    json.dump(sources, f, indent=1)
    f.write("\n")

traces = {}
with tempfile.TemporaryDirectory() as tmp:
    for greedy in (False, True):
        _, traces[greedy] = run_harness(greedy, os.path.join(tmp, f"trace_{greedy}.pt"))
torch.save(traces, os.path.join(HERE, "ref_harness_golden.pt"))
print({g: [t["accept_len"] for t in tr] for g, tr in traces.items()}, len(sources), "reference files")
