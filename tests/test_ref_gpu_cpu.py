"""Plumbing self-test of oracle/ref_gpu.py (the harness that times the UNMODIFIED reference on the GPU for bench.py's
`reference_gpu` block) with --device cpu on tiny models, in a subprocess: the reference's top-level module names
(Engine / Tree / utils) collide with this repository's drop-in shims, so it can never share a process with the tests.
The harness tests are skipped when oracle/_ref has not been vendored (tools/vendor_ref.py needs the reference's
sources); what the harness produced from the reference is stored in tests/golden/ref_harness_golden.pt, and the CPU
oracle is checked against it everywhere."""
import hashlib
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")
REF_DIR = os.path.join(ROOT, "oracle", "_ref")

SCRIPT = r"""
import json, sys, torch
sys.path.insert(0, r"%(root)s/oracle")
import ref_gpu
sys.path.append(r"%(root)s")
from sequoia_b200.model import LlamaConfigLite
spec = dict(draft="d", target="t", growmap="L40_growmaps/4x4-tree.pt", greedy=%(greedy)s, T=0.6, top_p=1.0, M=128, prefix=32,
            max_len=48, _cfgs={"d": LlamaConfigLite(64, 128, 1, 4, 4), "t": LlamaConfigLite(64, 128, 2, 4, 2)})
out = ref_gpu.run(spec, 4, 3, 2, r"%(trace)s", device="cpu")
tr = torch.load(r"%(trace)s")
out["trace_len"] = len(tr)
out["trace_tokens"] = int(tr[0]["tree_tokens"].numel())
print("RESULT " + json.dumps(out))
"""


def run_harness(greedy, trace_path):
    """oracle/ref_gpu.py on the vendored reference, SCRIPT's spec: -> (its JSON result, its first-iteration trace)."""
    code = SCRIPT % {"root": ROOT, "greedy": greedy, "trace": trace_path}
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1]
    return json.loads(line[len("RESULT "):]), torch.load(trace_path)


def assert_trace_equal(got, want):
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert torch.equal(g["tree_tokens"], w["tree_tokens"]), g["prompt"]
        assert (g["accept_len"], g["terminal"]) == (w["accept_len"], w["terminal"]), g["prompt"]
        assert torch.equal(g["valid_tokens"], w["valid_tokens"]), g["prompt"]
        assert torch.equal(g["target_logits_head"], w["target_logits_head"]), g["prompt"]


@pytest.mark.skipif(not os.path.isfile(os.path.join(REF_DIR, "utils.py")), reason="oracle/_ref not vendored")
@pytest.mark.parametrize("greedy", [False, True])
def test_reference_harness_runs_the_vendored_reference(greedy, tmp_path):
    out, trace = run_harness(greedy, str(tmp_path / "trace.pt"))
    assert out["impl"] == "reference_gpu" and out["value"] > 0 and out["steps"] == 4
    assert out["trace_len"] == 2 and out["trace_tokens"] == 16            # 4x4 tree: 17 nodes - root
    assert all(a >= 32 for a in out["first_iter_accept_lens"])
    assert_trace_equal(trace, torch.load(os.path.join(G, "ref_harness_golden.pt"))[greedy])


@pytest.mark.parametrize("greedy", [False, True])
def test_oracle_matches_reference_harness_golden(greedy):
    """The CPU oracle on the harness's tiny spec (same random-init weights, prompts and per-prompt seeds) reproduces,
    bit for bit, the first decode iteration the unmodified reference produced through oracle/ref_gpu.py."""
    from oracle import sequoia_oracle as O
    from sequoia_b200.model import LlamaConfigLite, _RandomInit, full_state_dict
    gm = torch.load(os.path.join(ROOT, "L40_growmaps", "4x4-tree.pt"))
    S, M, prefix = gm["size"], 128, 32

    def engine(c, seed, kind):
        oc = O.LlamaCfg(c.hidden_size, c.intermediate_size, c.num_hidden_layers, c.num_attention_heads,
                        c.num_key_value_heads, c.vocab_size, c.rms_norm_eps, c.rope_theta, c.max_position_embeddings)
        return O.EngineOracle(O.LlamaOracle(oc, full_state_dict(c, _RandomInit(c, seed, torch.device("cpu"))), M, kind))

    g = torch.Generator().manual_seed(17)
    prompts = [torch.randint(3, 32000, (prefix,), generator=g) for _ in range(2)]       # ref_gpu.run's prompt stream
    trace = []
    for pi, prompt in enumerate(prompts):
        draft = engine(LlamaConfigLite(64, 128, 1, 4, 4), 1, "FI")
        target = engine(LlamaConfigLite(64, 128, 2, 4, 2), 2, "TG")
        torch.manual_seed(1000 + pi)
        tree = (O.GreedyTreeOracle(draft, target, prompt, gm, max_length=M) if greedy else
                O.SpecTreeOracle(draft, target, prompt, gm, temperature=0.6, top_p=1.0, max_length=M))
        tree.construct_grow_map()
        tokens = tree.tokens[prefix:prefix + S - 1].clone()
        valid, a, _, term = tree.verify()
        trace.append({"prompt": pi, "tree_tokens": tokens, "accept_len": int(a), "terminal": bool(term),
                      "valid_tokens": valid[:a].clone(), "target_logits_head": tree.target_logits[:, :64].float()})
    assert_trace_equal(trace, torch.load(os.path.join(G, "ref_harness_golden.pt"))[greedy])


def test_vendor_manifest_matches_files():
    """The vendored copy is byte-identical to what the recipe recorded and to the reference's own files, whose sha256
    sums are stored in tests/golden/reference_sources.json (nobody edited the reference)."""
    mf = os.path.join(REF_DIR, "MANIFEST.json")
    if not os.path.isfile(mf):
        pytest.skip("oracle/_ref not vendored")
    with open(mf) as f:
        m = json.load(f)
    with open(os.path.join(G, "reference_sources.json")) as f:
        want = json.load(f)
    assert set(m["files"]) == set(want)
    for rel, sha in m["files"].items():
        with open(os.path.join(REF_DIR, rel), "rb") as fh:
            assert hashlib.sha256(fh.read()).hexdigest() == sha, rel
        assert sha == want[rel], f"{rel} differs from the reference's file"
