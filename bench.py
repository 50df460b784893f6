#!/usr/bin/env python
"""Benchmark of the Sequoia hot path on B200 (BASELINE.json metric: decoded tokens/s + mean accepted length/step).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config c2]

One "step" = one construct_grow_map() + verify() iteration of tests/testbed.py's simulation_fast loop (:80-87).
Workload (config c2, BASELINE.json configs[1]): random-init Llama-68m draft -> random-init Llama-2-7B target, growmap
A100_growmaps/68m_7b/growmaps/A100-CNN-68m-7b-stochastic.pt (128-node tree), T=0.6, P=1.0, M=384, synthetic prompts
torch.randint(3, 32000, (128,)) (seed 17), decode until 256 tokens.  With N > 1 ranks the target is tensor-sharded
over the N GPUs (NCCL allreduce, 2 per layer) while the draft stays on rank 0: total work is fixed => "strong".

Prints ONE JSON line on rank 0 (see README / DESIGN.md for every field).  `value` is timed with CUDA events around
the decode loops with everything already resident in HBM; `e2e` goes through the public API from pinned HOST buffers
(prompt H2D, Tree construction incl. its CPU-drawn random numbers, prefill, decode, D2H of the result).
`--impl reference` times the reference's own algorithm (the torch-CPU oracle port, oracle/) on the host cores.
`reference_gpu` (N=1) = the UNMODIFIED reference (oracle/_ref, vendored by tools/vendor_ref.py) timed on this same GPU in
a separate process through its own tests/testbed.py setup -- the bar BASELINE.json's north_star names -- plus a
full-size parity check of the first decode iteration of the first prompts (same weights, prompts, per-prompt seeds).
`tp_parity` (N>1) = the tensor-parallel target checked against an unsharded copy before the timed region.
`--config c5` = the reference's tree-shape sweep (tests/run.sh:1-30: SpecInfer policy over 30 KxL trees, M=512).
`--dump-outputs DIR` writes what the last timed step computed as DIR/<name>.npy (see dump_outputs), so that two builds
run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

CONFIGS = {
    # name: (draft, target, growmap, greedy, T, top_p, M, prefix, max_len)
    "c1": ("llama-68m", "llama-160m", "L40_growmaps/2-chain.pt", True, 0.6, 1.0, 288, 128, 256),
    "c2": ("llama-68m", "llama-2-7b", "A100_growmaps/68m_7b/growmaps/A100-CNN-68m-7b-stochastic.pt", False, 0.6, 1.0, 384,
           128, 256),
    # c2 with the growmap tree_search.py derives from this GPU's measured draft/verify times (B200_growmaps/)
    "c2b": ("llama-68m", "llama-2-7b", "B200_growmaps/68m_7b-demo_acceptance.pt", False, 0.6, 1.0, 384, 128, 256),
    "c3": ("llama-68m", "llama-2-13b", "L40_growmaps/8x8-tree.pt", False, 0.6, 1.0, 384, 128, 256),
    "c4": ("llama-2-7b", "llama-2-70b", "L40_growmaps/L40-CNN-7b-70b-stochastic.pt", False, 0.6, 1.0, 1024, 128, 256),
}
# tests/run.sh:1-30 of the reference: K chains of length L ("KxL-tree.pt"), driven through SpecInferTree, M=512
SWEEP = [f"{k}x{n // k}" for n in (8, 16, 32, 64, 128) for k in (1, 2, 4, 8, 16, 32, 64, 128) if k <= n]
CONFIGS["c5"] = ("llama-68m", "llama-2-7b", "L40_growmaps/{shape}-tree.pt", False, 0.6, 1.0, 512, 128, 256)
METRIC = "decoded tokens/sec (mean accepted len/step in config.accepted_tokens_per_step), Sequoia tree speculative decoding, 68m->7B Llama (config c2 unless --config says otherwise)"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_tf_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f).get("bf16_tflops_sustained", 1420.0))
    return 1420.0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------------
def synthetic_prompts(n, length, seed=17):
    from data_converter import synthetic_prompts as sp
    return sp(n, length, 32000, seed)


def _buffers(M, dev):
    return dict(attn_mask=torch.full((M, M), torch.finfo(torch.float16).min, dtype=torch.float16, device=dev),
                sequence=torch.arange(M, device=dev).unsqueeze(-1), new_tokens_buffer=torch.zeros(M, device=dev).long(),
                parents_buffer=torch.zeros(M, device=dev).long(), position_ids=torch.zeros(M, device=dev).long())


def ref_spec(config, gm_path=None):
    dname, tname, gmp, greedy, T, top_p, M, prefix, max_len = CONFIGS[config]
    return dict(draft=dname, target=tname, growmap=gm_path or gmp, greedy=greedy, T=T, top_p=top_p, M=M, prefix=prefix,
                max_len=max_len, draft_seed=1, target_seed=2)


def run_reference_gpu(config, steps, warmup, n_parity, trace_path, timeout=900):
    """The unmodified reference on this GPU (oracle/ref_gpu.py, separate process).  -> its JSON dict."""
    if not os.path.isfile(os.path.join(ROOT, "oracle", "_ref", "utils.py")):
        return {"impl": "reference_gpu", "unavailable": "oracle/_ref missing (tools/vendor_ref.py runs in the build container)"}
    last = None
    for sdp in ("no_cudnn", "math"):      # a CUDA fault poisons the process: every attempt is a fresh one
        cmd = [sys.executable, os.path.join(ROOT, "oracle", "ref_gpu.py"), "--spec", json.dumps(ref_spec(config)), "--steps",
               str(steps), "--warmup", str(warmup), "--parity", str(n_parity), "--trace", trace_path, "--sdp", sdp]
        try:
            r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=timeout, cwd=ROOT)
            lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            last = json.loads(lines[-1]) if lines else {"impl": "reference_gpu", "unavailable": f"rc={r.returncode}: {r.stderr[-400:]}"}
        except Exception as e:
            last = {"impl": "reference_gpu", "unavailable": f"{type(e).__name__}: {e}"}
        if "unavailable" not in last:
            return last
        last["unavailable"] = f"[sdpa={sdp}] " + last["unavailable"][:300]
        last.pop("traceback", None)
    return last


def first_iteration_trace(new_tree, draft, target, S, prefix, n_prompts):
    """First decode iteration of the first prompts (drafted tree, accept length, accepted tokens): the records
    oracle/ref_gpu.py saves for the reference, from this implementation."""
    out = []
    for pi in range(n_prompts):
        tree = new_tree(pi)
        tree.construct_grow_map()
        tokens = tree.tokens[prefix:prefix + S - 1].cpu().clone()
        valid, a, _, term = tree.verify()
        out.append({"prompt": pi, "tree_tokens": tokens, "accept_len": int(a), "terminal": bool(term),
                    "valid_tokens": valid[:a].cpu().clone()})
        draft.clear_kv()
        target.clear_kv()
    return out


def compare_traces(ours, ref, grow_map):
    """Full-size parity of the first iteration: fraction of identically drafted tree nodes (a node only counts if all its
    ancestors match too -- below a differing node the two runs legitimately sample from different draft contexts) and
    whether the accept walk took the same path."""
    S = grow_map["size"]
    parent = {}
    for p, ch in enumerate(grow_map["Successors"]):
        for c in ch:
            parent[c] = p
    res = []
    for o, r in zip(ours, ref):
        eq = (o["tree_tokens"] == r["tree_tokens"]).tolist()
        ok = [True] * S                                           # node 0 = root
        for k in range(1, S):
            ok[k] = eq[k - 1] and ok[parent[k]]
        comparable = sum(1 for k in range(1, S) if ok[parent[k]])         # nodes whose whole ancestry matched
        same = sum(1 for k in range(1, S) if ok[k])
        res.append({"prompt": o["prompt"], "tree_nodes_identical": round(same / max(S - 1, 1), 4),
                    "identical_given_same_parent": round(same / max(comparable, 1), 4),
                    "accept_len": [o["accept_len"], r["accept_len"]],
                    "accepted_tokens_identical": bool(o["accept_len"] == r["accept_len"] and
                                                      torch.equal(o["valid_tokens"], r["valid_tokens"]))})
    return res


def tp_parity_check(dname, tname, target_tp, grow_map, cls, M, T, top_p, prefix, dev, tp_group, iters=4):
    """Rank 0, before the timed region: the tensor-parallel target against an UNSHARDED copy of the same model on this
    GPU -- two trees in lock-step on the same prompt, seeds and bonus-token noise."""
    from sequoia_b200.engine import GraphInferenceEngine, GraphInferenceEngineTG
    from sequoia_b200.tp import attach_tp
    V = 32000
    target_1 = GraphInferenceEngineTG(M, f"random-init:{tname}:2", device=dev)
    drafts = [GraphInferenceEngine(M, f"random-init:{dname}:1", device=dev) for _ in range(2)]
    attach_tp(drafts[0], target_tp, tp_group)
    prompt = synthetic_prompts(1, prefix)[0].to(dev)
    noise = torch.empty(iters, V, dtype=torch.float16).exponential_(1.0, generator=torch.Generator().manual_seed(5)).to(dev)
    trees = []
    for d, t in ((drafts[0], target_tp), (drafts[1], target_1)):
        torch.manual_seed(4242)
        tr = cls(prefix=prompt, device=dev, temperature=T, top_p=top_p, draft_model_engine=d, target_model_engine=t,
                 max_length=M, max_target_seq=M, grow_map=grow_map, **_buffers(M, dev))
        if hasattr(tr.rt, "external_noise"):
            tr.rt.external_noise = noise
        trees.append(tr)
    max_rel, same_steps, forked = 0.0, 0, False
    for it in range(iters):
        outs = []
        for tr in trees:
            tr.construct_grow_map()
            v, a, _, term = tr.verify()
            outs.append((v.clone(), a, term, tr.rt.target_logits.float().clone()))
        (v0, a0, t0, l0), (v1, a1, t1, l1) = outs
        if not forked:                      # after a fork the two trees hold different tokens: logits no longer comparable
            max_rel = max(max_rel, ((l0 - l1).abs().max() / l1.abs().max()).item())
        if a0 == a1 and t0 == t1 and torch.equal(v0, v1) and not forked:
            same_steps += 1
        else:
            forked = True
        if t0 or t1:
            break
    for tr in trees:
        tr.rt.external_noise = None
    peer = target_tp.engine.runner.peer
    out = {"model": tname, "iters": iters, "max_rel_logit_err": round(max_rel, 6), "accept_seq_identical_steps": same_steps,
           "peer_error": int(peer.error()) if peer is not None else 0,
           "attn_error": int(target_tp.engine.runner.plan.error()),
           "how": "TP target vs an unsharded copy on rank 0, same prompt / seeds / bonus noise, lock-step; logit error "
                  "relative to max |logit| while the two token sequences are still identical"}
    drafts[0].clear_kv(); drafts[1].clear_kv(); target_1.clear_kv(); target_tp.clear_kv()
    from sequoia_b200.tree import clear_runtimes
    clear_runtimes()
    del trees, target_1, drafts
    torch.cuda.empty_cache()
    return out


DUMP_BYTES = 64 * 10**6 - 4096          # all .npy files together, headers included


def dump_outputs(path, tree, valid, accept_len, terminal):
    """Write what the last timed construct_grow_map() + verify() step computed as <path>/<name>.npy: verify()'s return
    values (the accepted sequence incl. the prompt, the accept length, the terminal flag; float64, exact for token ids)
    and the target logits the accept walk decided on (tree.target_logits, float32).  If the logits exceed the DUMP_BYTES
    budget, a fixed seeded sample of their rows is written, with the row indices in target_logits_rows.npy."""
    import numpy as np
    out = {"valid_tokens": valid.cpu().double(), "accept_length": torch.tensor([accept_len], dtype=torch.float64),
           "terminal": torch.tensor([float(terminal)], dtype=torch.float64)}
    logits = tree.target_logits.float().cpu()
    max_rows = (DUMP_BYTES - sum(t.numel() * 8 for t in out.values()) - logits.shape[0] * 8) // (logits.shape[1] * 4)
    if logits.shape[0] > max_rows:
        rows = torch.randperm(logits.shape[0], generator=torch.Generator().manual_seed(0))[:max_rows].sort().values
        out["target_logits_rows"] = rows.double()
        logits = logits[rows]
    out["target_logits"] = logits
    os.makedirs(path, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(path, name + ".npy"), t.numpy())


def run_b200(args):
    import torch.distributed as dist
    from sequoia_b200 import _lib
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    tp_group = None
    if world > 1:
        # NCCL prints its version banner on stdout when the first communicator is created; the contract is ONE JSON line,
        # so create the communicator with fd 1 pointed at /dev/null
        sys.stdout.flush()
        saved_fd, null_fd = os.dup(1), os.open(os.devnull, os.O_WRONLY)
        os.dup2(null_fd, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device(dev))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            os.dup2(saved_fd, 1)
            os.close(null_fd)
            os.close(saved_fd)
        tp_group = dist.group.WORLD
    if args.config == "c5":
        assert world == 1, "the tree-shape sweep is a single-GPU configuration"
        return run_sweep(args, dev)
    dname, tname, gm_path, greedy, T, top_p, M, prefix, max_len = CONFIGS[args.config]
    grow_map = torch.load(os.path.join(ROOT, gm_path))
    S = grow_map["size"]
    from sequoia_b200.engine import GraphInferenceEngine, GraphInferenceEngineTG
    from sequoia_b200.model import NAMED_CONFIGS
    from sequoia_b200.tp import TPFollower, attach_tp, stop_followers
    from sequoia_b200.tree import GreedyTree, SpecTree
    cls = GreedyTree if greedy else SpecTree

    def finish(rc=0):
        sys.stdout.flush()
        sys.stderr.flush()
        if world > 1:
            os._exit(rc)                     # NCCL communicators captured in CUDA graphs: skip the slow teardown
        if rc:
            sys.exit(rc)

    # ---- reference GPU arm first (N=1 only; the reference has no multi-GPU path): nothing of ours is resident yet ---------
    ref_gpu = ref_trace = None
    n_parity = 0 if args.no_reference_gpu else 4
    if world == 1 and not args.no_reference_gpu:
        # the source tree may be read-only: the reference arm's trace goes through a temporary directory
        with tempfile.TemporaryDirectory(prefix="sequoia_bench_") as tmp:
            trace_path = os.path.join(tmp, f"ref_gpu_trace_{args.config}.pt")
            ref_gpu = run_reference_gpu(args.config, min(args.steps, 40), 3, n_parity, trace_path)
            if "unavailable" not in ref_gpu and os.path.exists(trace_path):
                ref_trace = torch.load(trace_path)

    # ---- TP parity on a model that fits unsharded next to a shard (70B: its first 8 layers' worth) ------------------------
    tp_parity = None
    wb = lambda c: 2 * (c.num_hidden_layers * (2 * c.hidden_size * (c.num_attention_heads + c.num_key_value_heads) * c.head_dim
                                              + 3 * c.hidden_size * c.intermediate_size) + 2 * c.vocab_size * c.hidden_size)
    fits = wb(NAMED_CONFIGS[tname]) * (1 + 1 / world) + 2 * wb(NAMED_CONFIGS[dname]) < 150e9
    parity_name = tname if fits else tname + "-8l"
    if world > 1 and not args.no_tp_parity and parity_name != tname:
        small = GraphInferenceEngineTG(M, f"random-init:{parity_name}:2", device=dev, tp_group=tp_group)
        if rank != 0:
            TPFollower(small, grow_map, greedy, M, dev, tp_group).serve()
        else:
            tp_parity = tp_parity_check(dname, parity_name, small, grow_map, cls, M, T, top_p, prefix, dev, tp_group)
            stop_followers(tp_group, dev)
        del small
        torch.cuda.empty_cache()
        dist.barrier()

    torch.manual_seed(17)
    target = GraphInferenceEngineTG(M, f"random-init:{tname}:2", device=dev, tp_group=tp_group)
    prompts = synthetic_prompts(64, prefix)

    def barrier():
        if world > 1:
            target._tp_driver.barrier()      # follower ranks are slaved to rank 0: sync + barrier through the control op
        torch.cuda.synchronize()

    if rank != 0:
        # follower ranks: target shard only, driven by rank 0's broadcasts
        TPFollower(target, grow_map, greedy, M, dev, tp_group).serve()
        finish()
        return
    if world > 1 and not args.no_tp_parity and parity_name == tname:
        tp_parity = tp_parity_check(dname, tname, target, grow_map, cls, M, T, top_p, prefix, dev, tp_group)
    if tp_parity is not None and (tp_parity["peer_error"] or tp_parity["attn_error"]):
        print(json.dumps({"error": "tp_parity: device-side handshake / watchdog error", "tp_parity": tp_parity}))
        stop_followers(tp_group, dev)
        finish(3)
    draft = GraphInferenceEngine(M, f"random-init:{dname}:1", device=dev)
    if world > 1:
        attach_tp(draft, target, tp_group)
    buf = _buffers(M, dev)

    def new_tree(prompt_dev, pi=0):
        torch.manual_seed(1000 + pi)         # per-prompt CPU stream for r / rand: the reference-GPU arm seeds identically
        return cls(prefix=prompt_dev, device=dev, temperature=T, top_p=top_p, draft_kv_len=0, target_kv_len=0,
                   draft_model_engine=draft, target_model_engine=target, max_length=M, max_target_seq=M,
                   grow_map=grow_map, **buf)

    class Loop:
        """tests/testbed.py:45-95 (simulation_fast) with a step budget; timing by CUDA events around each prompt's
        while-loop (construction / prefill excluded exactly as :78-91 does)."""

        def __init__(self):
            self.pi = 0
            self.tree = None
            self.len = 0
            self.terminate = True

        def next_prompt(self, host=False):
            if self.tree is not None:
                draft.clear_kv()
                target.clear_kv()
            p = prompts[self.pi % len(prompts)]
            self.pi += 1
            if host:
                self.h2d += p.numel() * 8 + M * 2 + S * 32000 * 2 + M * 8 + 64
                p = pinned_prompts[(self.pi - 1) % len(prompts)].to(dev, non_blocking=True)
            else:
                p = p.to(dev)
            self.tree = new_tree(p, self.pi - 1)
            self.len = prefix
            self.terminate = False

        h2d = 0
        d2h = 0
        draft_ms = 0.0
        verify_ms = 0.0

        def run_steps(self, k, timed, host=False):
            done = tokens = 0
            ms = 0.0
            while done < k:
                if self.terminate or self.len >= max_len:
                    if host and self.tree is not None:
                        _ = self.tree.tokens[:self.len].to("cpu")        # D2H of the finished sequence
                        self.d2h += self.len * 8
                    self.next_prompt(host)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                while done < k and self.len < max_len and not self.terminate:
                    ea, eb, ec = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                    ea.record()
                    self.tree.construct_grow_map()
                    eb.record()
                    valid, accept_len, _, self.terminate = self.tree.verify()
                    self.last = (valid, accept_len, self.terminate)
                    ec.record()
                    ec.synchronize()
                    if timed:                                         # phase split (tests/testbed.py:144-219 reports the same)
                        self.draft_ms += ea.elapsed_time(eb)
                        self.verify_ms += eb.elapsed_time(ec)
                    tokens += valid.shape[0] - self.len
                    self.len = valid.shape[0]
                    if int(self.tree.rt.host_state[5]) in (0, 2):       # bonus token is EOS / pad (testbed.py:87)
                        self.terminate = True
                    done += 1
                    self.d2h += 64
                e1.record()
                e1.synchronize()
                ms += e0.elapsed_time(e1)
            return tokens, ms

    # ---- full-size parity against the reference-GPU trace (first iteration of the first prompts; untimed) --------------
    parity = None
    if ref_trace is not None:
        ours = first_iteration_trace(lambda pi: new_tree(prompts[pi].to(dev), pi), draft, target, S, prefix, n_parity)
        parity = compare_traces(ours, ref_trace, grow_map)
        ref_gpu["first_iteration_parity"] = parity

    loop = Loop()
    # warm-up: captures the graphs (first prompt) and W untimed steps
    loop.run_steps(max(args.warmup, 3), timed=False)
    lc0 = loop.tree.rt.kernel_launches()
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    t_wall0 = time.time()
    if args.timeline:
        # in-process CUPTI trace of the timed steps (no kernel replay, so it works under tensor parallelism where ncu cannot):
        # per-kernel device time as it runs INSIDE the graphs.  A run with --timeline is a diagnosis, not a bench value.
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            tokens, ms = loop.run_steps(args.steps, timed=True)
            torch.cuda.synchronize()
        write_timeline(prof, args.timeline, args.steps, ms)
    else:
        tokens, ms = loop.run_steps(args.steps, timed=True)
    barrier()
    wall = time.time() - t_wall0
    clocks = sampler.stop()
    launches = loop.tree.rt.kernel_launches() - lc0
    value = tokens / (ms / 1e3)
    acc_per_step = tokens / args.steps
    if args.dump_outputs:                    # before the e2e loop below reuses the runtime's buffers
        dump_outputs(args.dump_outputs, loop.tree, *loop.last)

    # ---- e2e: same metric through the public API from pinned host buffers -------------------------------------------
    pinned_prompts = [p.pin_memory() for p in prompts]
    loop2 = Loop()
    loop2.pi = 1000
    loop2.tree = loop.tree
    loop2.h2d = loop2.d2h = 0
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    tok2, _ = loop2.run_steps(args.steps, timed=True, host=True)
    _ = loop2.tree.tokens[:loop2.len].to("cpu")
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    e2e = {"value": tok2 / (e2e_ms / 1e3), "unit": "tokens/s", "h2d_bytes_per_step": loop2.h2d // args.steps,
           "d2h_bytes_per_step": loop2.d2h // args.steps,
           "note": "includes per-prompt Tree construction (CPU-drawn r/rand as in the reference), prefill, decode"}
    peer = target.engine.runner.peer
    dev_err = {"peer_error": int(peer.error()) if peer is not None else 0,
               "attn_error": int(target.engine.runner.plan.error()) | int(draft.engine.runner.plan.error())}

    # ---- roofline of the verify tree-attention kernel, measured live (CUDA events on the launching stream) ----------
    roof = extra = None
    if not args.no_micro:
        roof = attention_roofline(target, grow_map, prefix, M)
        extra = micro_kernels(draft, target, loop.tree, grow_map)
    draft.clear_kv()
    target.clear_kv()
    if world > 1:
        stop_followers(tp_group, dev)
    out = {
        "metric": METRIC, "value": round(value, 2), "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic (random-init weights, random prompts)",
        "config": {"workload": f"{args.config}: {dname}->{tname}, {os.path.basename(gm_path)} (tree {S}), "
                               f"{'greedy' if greedy else 'stochastic'} T={T} P={top_p} M={M}, prefix {prefix}->{max_len} tokens",
                   "accepted_tokens_per_step": round(acc_per_step, 4), "parallelism": f"target tp{world}, draft on rank 0",
                   "l2": "inputs larger than L2: each step streams the target's %.1f GB of weights" % (target.engine.runner.weight_bytes() / 1e9)},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roof, "kernels": extra,
        "wall_s_timed_region": round(wall, 3), "device_errors": dev_err, "profiled": bool(args.timeline),
        "phases": {"draft_ms_per_step": round(loop.draft_ms / args.steps, 4), "verify_ms_per_step": round(loop.verify_ms / args.steps, 4),
                   "note": "CUDA events around construct_grow_map() (draft tree, rank 0 only) and verify() (target forward over "
                           "all ranks + accept walk + KV compaction + 1-token draft forward) of the timed steps"},
    }
    if tp_parity is not None:
        out["tp_parity"] = tp_parity
    if ref_gpu is not None:
        out["reference_gpu"] = ref_gpu
        if "value" in ref_gpu and ref_gpu["value"]:
            out["reference_gpu"]["speedup_vs_reference_gpu"] = round(value / ref_gpu["value"], 3)
    if not args.no_cpu_baseline and world == 1:
        out["cpu_baseline"] = cpu_reference(args.config, max_seconds=25.0, max_iters=3)
    print(json.dumps(out))
    finish(3 if (dev_err["peer_error"] or dev_err["attn_error"]) else 0)


def write_timeline(prof, path, steps, ms):
    """Markdown table: device time per kernel name over the timed steps, from the profiler's CUDA events."""
    import collections
    import re
    tot = collections.defaultdict(lambda: [0, 0.0])
    t_min, t_max, busy = None, None, 0.0
    for ev in prof.events():
        if ev.device_type is None or "cuda" not in str(ev.device_type).lower():
            continue
        dur = float(getattr(ev, "device_time_total", 0.0) or getattr(ev, "cuda_time_total", 0.0) or 0.0)
        if dur <= 0:
            continue
        name = re.sub(r"\(.*", "", re.sub(r"<.*", "", ev.name)).replace("void ", "")[:70]
        tot[name][0] += 1
        tot[name][1] += dur
        busy += dur
    with open(path, "w") as f:
        f.write(f"In-graph device time per kernel over {steps} timed decode steps (torch.profiler / CUPTI, rank 0; "
                f"CUDA-event time of the same steps {ms:.2f} ms; sum of kernel times {busy / 1e3:.2f} ms).\n\n")
        f.write("| kernel | launches / step | us / step | share of kernel time | avg us |\n|---|---:|---:|---:|---:|\n")
        for k, (c, d) in sorted(tot.items(), key=lambda kv: -kv[1][1]):
            f.write(f"| `{k}` | {c / steps:.1f} | {d / steps:.1f} | {100 * d / max(busy, 1e-9):.1f}% | {d / c:.2f} |\n")


def run_sweep(args, dev):
    """Config c5: tests/run.sh:1-30 of the reference -- tokens/s vs tree shape, SpecInfer policy, 68m -> 7B, M=512."""
    from sequoia_b200.engine import GraphInferenceEngine, GraphInferenceEngineTG
    from sequoia_b200.tree import SpecInferTree, clear_runtimes
    dname, tname, gm_tmpl, _, T, top_p, M, prefix, max_len = CONFIGS["c5"]
    target = GraphInferenceEngineTG(M, f"random-init:{tname}:2", device=dev)
    draft = GraphInferenceEngine(M, f"random-init:{dname}:1", device=dev)
    prompts = synthetic_prompts(64, prefix)
    buf = _buffers(M, dev)
    rows = []
    sampler = ClockSampler(int(dev.split(":")[1]))
    sampler.start()
    total_ms = total_tokens = total_steps = launches = 0
    steps = args.steps
    for shape in SWEEP:
        grow_map = torch.load(os.path.join(ROOT, gm_tmpl.format(shape=shape)))
        pi, done, tokens, ms = 0, 0, 0, 0.0
        warm = 3
        tree = None
        while done < steps + warm:
            torch.manual_seed(1000 + pi)
            if tree is not None:
                draft.clear_kv(); target.clear_kv()
            tree = SpecInferTree(prefix=prompts[pi % 64].to(dev), device=dev, temperature=T, top_p=top_p,
                                 draft_model_engine=draft, target_model_engine=target, max_length=M, max_target_seq=M,
                                 grow_map=grow_map, **buf)
            pi += 1
            length, term = prefix, False
            while done < steps + warm and length < max_len and not term:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                tree.construct_grow_map()
                valid, accept_len, _, verify_term = tree.verify()
                e1.record()
                e1.synchronize()
                if done >= warm:
                    ms += e0.elapsed_time(e1)
                    tokens += valid.shape[0] - length
                length = valid.shape[0]
                term = verify_term or int(tree.rt.host_state[5]) in (0, 2)
                done += 1
        launches += tree.rt.kernel_launches()
        if args.dump_outputs and shape == SWEEP[-1]:
            dump_outputs(args.dump_outputs, tree, valid, accept_len, verify_term)
        rows.append({"tree": shape, "size": int(grow_map["size"]), "levels": len(grow_map["roots"]),
                     "tokens_per_s": round(tokens / (ms / 1e3), 1), "ms_per_step": round(ms / steps, 3),
                     "accepted_tokens_per_step": round(tokens / steps, 3)})
        total_ms += ms; total_tokens += tokens; total_steps += steps
        draft.clear_kv(); target.clear_kv()
        clear_runtimes()
        torch.cuda.empty_cache()
    clocks = sampler.stop()
    best = max(rows, key=lambda r: r["tokens_per_s"])
    out = {"metric": METRIC, "value": best["tokens_per_s"], "unit": "tokens/s", "n_gpus": 1, "steps": steps, "warmup": 3,
           "ms_per_step": best["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f16", "data": "synthetic (random-init weights, random prompts)",
           "config": {"workload": f"c5: {dname}->{tname}, tree-shape sweep tests/run.sh:1-30 ({len(SWEEP)} KxL trees, SpecInfer "
                                  f"policy, T={T} P={top_p} M={M}); value = best shape ({best['tree']})",
                      "accepted_tokens_per_step": best["accepted_tokens_per_step"], "parallelism": "target tp1",
                      "l2": "inputs larger than L2: each step streams the target's 13.5 GB of weights"},
           "clocks": clocks, "gpu_launches": int(launches), "sweep": rows,
           "sweep_mean_tokens_per_s": round(total_tokens / (total_ms / 1e3), 1)}
    print(json.dumps(out))


def _timeit(fn, iters=20, warm=3, reps=5):
    """Average device time (us) of one fn() call: `iters` calls are captured into a CUDA graph (so host launch overhead
    is excluded, as inside the real decode graphs) and the graph is replayed `reps` times between CUDA events."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(warm):
            fn()
        s.synchronize()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(iters):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / (iters * reps) * 1e3   # us


def _sha16(path):
    import hashlib
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()[:16]


def attention_roofline(target, grow_map, prefix, M):
    """Verify attention (Engine/Llama_modules.py:220-248) of the steady-state shape: q = S tree rows, kv = P-1+S with the
    mid-decode P (193 for prefix 128 -> 256 tokens: kv = 320 for config 2 as in SURVEY.md 8d); cycles through all layers
    so K/V come from HBM (cache >> L2 at 7B).  HBM-bound when the arithmetic intensity is below the measured ridge
    (configs 2/3), tensor-pipe-bound otherwise (config 4's GQA shape)."""
    from sequoia_b200 import ops
    from sequoia_b200.tree import pack_tree_mask
    rn = target.engine.runner
    S = grow_map["size"]
    P = min(193, M - S + 1)
    kv = P - 1 + S
    bits = pack_tree_mask(grow_map["mask"]).to(rn.device)
    state = torch.zeros(16, dtype=torch.int32, device=rn.device)
    state[0] = P
    rn.qkv.normal_(0, 1)
    rn.k_cache.normal_(0, 1)
    rn.v_cache.normal_(0, 1)
    layer = [0]

    def call():
        ops.tree_attn(rn.plan, layer[0] % rn.L, S, state=state, n0=0, kv_end=S, tree_bits=bits, tree_words=bits.shape[1],
                      tree_size=S, impl=0)
        layer[0] += 1

    us = _timeit(call, iters=4 * rn.L, warm=rn.L)
    D = rn.D
    alg_bytes = 2 * D * 2 * (rn.Hkv * kv + rn.H * S)           # K+V read once, Q read + O write (SURVEY.md 8d)
    flops = 4 * rn.H * S * kv * D
    peak, how = load_peaks()
    tf_peak = load_tf_peak()
    # measured DRAM traffic: only if the committed ncu capture is of THIS kernel source and THIS shape
    traffic = None
    tp = os.path.join(ROOT, "profiles", "attn_traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            t = json.load(f)
        if t.get("kernel_sha16") == _sha16(os.path.join(ROOT, "sequoia_b200", "csrc", "sq_attn.cu")) and \
                t.get("shape") == [rn.H, rn.Hkv, S, kv, D]:
            traffic = t.get("dram_bytes_per_launch")
    rn.k_cache.zero_()
    rn.v_cache.zero_()
    gbs, tfs = alg_bytes / (us * 1e-6) / 1e9, flops / (us * 1e-6) / 1e12
    tensor_bound = flops / alg_bytes > tf_peak * 1e12 / (peak * 1e9)
    out = {"kernel": "tree_attn_tc_kernel<%d> (verify attention, whole launch incl. split-KV reduction; H=%d Hkv=%d q=%d kv=%d)"
                     % (D, rn.H, rn.Hkv, S, kv),
           "bound": "tensor" if tensor_bound else "hbm",
           "achieved": round(tfs if tensor_bound else gbs, 2), "peak": tf_peak if tensor_bound else peak,
           "unit": "TFLOP/s" if tensor_bound else "GB/s",
           "frac": round((tfs / tf_peak) if tensor_bound else (gbs / peak), 4), "traffic": traffic, "peak_source": how,
           "algorithmic_bytes": alg_bytes, "algorithmic_flops": flops, "us_per_launch": round(us, 3),
           "GBps": round(gbs, 1), "tflops": round(tfs, 2)}
    return out


def micro_kernels(draft, target, tree, grow_map):
    """Per-kernel device times (us) of the other hot-path kernels at this config's shapes, for DESIGN.md's table."""
    from sequoia_b200 import ops
    rt = tree.rt
    S = grow_map["size"]
    out = {}
    lv = max(range(len(rt.st.levels)), key=lambda i: rt.st.levels[i]["n_parents"])
    rows = rt.st.levels[lv]["n_parents"]
    us = _timeit(lambda: rt.op_sample(lv))
    out["sample_level"] = {"us": round(us, 2), "rows": rows, "GBps": round(rows * 32000 * 4 / us / 1e3, 1)}
    snap_t, snap_p, snap_s = rt.tokens.clone(), rt.position_ids.clone(), rt.state.clone()

    def acc():
        rt.state.copy_(snap_s)
        rt.op_accept()
    us = _timeit(acc)
    out["accept_walk(+state copy)"] = {"us": round(us, 2)}
    rt.tokens.copy_(snap_t); rt.position_ids.copy_(snap_p); rt.state.copy_(snap_s)
    st = torch.zeros(16, dtype=torch.int32, device=rt.device)
    st[3], st[4] = 5, 150
    idx = torch.tensor([160, 170, 180, 190, 200, 0, 0, 0], dtype=torch.int32, device=rt.device)
    kvc = target.engine.kv_cache
    us = _timeit(lambda: kvc.gather_from_state(idx, st, 8))
    L, _, Hkv, _, D = kvc.k_cache.shape
    out["kv_gather(target,n=5)"] = {"us": round(us, 2), "GBps": round(2 * 2 * L * Hkv * 5 * D * 2 / us / 1e3, 1)}
    rn = target.engine.runner
    us = _timeit(lambda: ops.add_rmsnorm(rn.hidden, rn.proj, rn.norm, rn.normed, S, rn.eps))
    out["add_rmsnorm(S rows)"] = {"us": round(us, 2), "GBps": round(S * rn.h * 2 * 4 / us / 1e3, 1)}
    st2 = torch.zeros(16, dtype=torch.int32, device=rt.device)
    st2[0] = 150
    us = _timeit(lambda: ops.rope_kv_append(rn.qkv, rn.H, rn.Hkv, rn.D, rn.cos, rn.sin, rt.position_ids, rt.storage_ids, S,
                                            rn.k_cache[0], rn.v_cache[0], rn.M, state=st2, n0=0))
    b = S * (rn.H + 2 * rn.Hkv) * rn.D * 2 + S * (rn.H + 2 * rn.Hkv) * rn.D * 2      # read qkv, write q + K + V
    out["rope_kv_append(S rows)"] = {"us": round(us, 2), "GBps": round(b / us / 1e3, 1)}
    us = _timeit(lambda: ops.silu_mul(rn.gate_up, rn.act, S))
    out["silu_mul(S rows)"] = {"us": round(us, 2), "GBps": round(S * rn.I * 2 * 3 / us / 1e3, 1)}
    if rn.peer is not None and rt.tp is not None:
        # every rank must issue the same launches (each one handshakes with its peers): followers mirror via OP_MICRO
        from sequoia_b200.tp import OP_MICRO, micro_allreduce
        k = 64
        rt.tp.send_ctrl(OP_MICRO, k, S)
        micro_allreduce(rn, k, S)                        # warm-up round
        torch.cuda.synchronize()
        rt.tp.send_ctrl(OP_MICRO, k, S)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        micro_allreduce(rn, k, S)
        e1.record()
        e1.synchronize()
        us = e0.elapsed_time(e1) / k * 1e3
        N = rn.tp.size
        out["tp_allreduce_add_rmsnorm(S rows)"] = {"us": round(us, 2), "ranks": N,
                                                   "nvlink_rx_GBps": round((N - 1) * S * rn.h * 2 / us / 1e3, 1),
                                                   "note": "eager back-to-back launches incl. host launch gaps"}
    rn.k_cache[0].zero_(); rn.v_cache[0].zero_()
    return out


# ----------------------------------------------------------------------------------------------------------------------
def pick_cpu_threads():
    """torch's fp16 CPU GEMM does not scale to every core count (128 threads were 10x slower than 8 on the build box):
    try powers of two up to os.cpu_count() on one 7B-shaped linear and keep the fastest, i.e. all the threads the
    reference's CPU path can actually use."""
    n = os.cpu_count() or 1
    x = torch.randn(128, 4096).half()
    w = torch.randn(4096, 4096).half()
    best, best_t = 1, float("inf")
    c = 1
    cands = []
    while c < n:
        cands.append(c)
        c *= 2
    cands.append(n)
    for c in cands[-5:]:
        torch.set_num_threads(c)
        torch.nn.functional.linear(x, w)
        t0 = time.time()
        for _ in range(3):
            torch.nn.functional.linear(x, w)
        dt = time.time() - t0
        if dt < best_t:
            best, best_t = c, dt
    return best


def cpu_reference(config, max_seconds, max_iters, warm_iters=1):
    """The reference's algorithm on the host cores: the torch-CPU oracle port (oracle/sequoia_oracle.py) on the same
    shapes.  To keep host init bounded, all target layers alias ONE layer's random weights (identical FLOPs/bytes per
    layer; the working set still exceeds the caches).  Returns tokens/s over the timed iterations."""
    from oracle import sequoia_oracle as O
    from sequoia_b200.model import NAMED_CONFIGS
    dname, tname, gm_path, greedy, T, top_p, M, prefix, max_len = CONFIGS[config]
    ncores = pick_cpu_threads()
    torch.set_num_threads(ncores)
    grow_map = torch.load(os.path.join(ROOT, gm_path))

    def weights(name, seed):
        """The SAME random-init model the GPU arms use: drawn by sequoia_b200.model._RandomInit's seeded CUDA generator
        (tensor by tensor, copied to host).  Without a CUDA device (build container) fall back to the oracle's own CPU
        init with one layer's tensors aliased across layers (bounded init time) and say so."""
        c = NAMED_CONFIGS[name]
        cfg = O.LlamaCfg(c.hidden_size, c.intermediate_size, c.num_hidden_layers, c.num_attention_heads,
                         c.num_key_value_heads, c.vocab_size, c.rms_norm_eps, c.rope_theta, c.max_position_embeddings)
        if torch.cuda.is_available():
            from sequoia_b200.model import _RandomInit, full_state_dict
            gen = _RandomInit(c, seed, torch.device("cuda:0"))

            class ToHost:
                def get(self, n, shape):
                    return gen.get(n, shape).cpu()
            return cfg, full_state_dict(c, ToHost()), True
        one = O.LlamaCfg(c.hidden_size, c.intermediate_size, 1, c.num_attention_heads, c.num_key_value_heads,
                         c.vocab_size, c.rms_norm_eps, c.rope_theta, c.max_position_embeddings)
        w1 = O.init_llama_weights(one, seed)
        w = dict(w1)
        for l in range(1, c.num_hidden_layers):
            for k, v in w1.items():
                if k.startswith("model.layers.0."):
                    w[k.replace("model.layers.0.", f"model.layers.{l}.")] = v
        return cfg, w, False

    t0 = time.time()
    dcfg, dw, same_d = weights(dname, 1)
    tcfg, tw, same_t = weights(tname, 2)
    draft = O.EngineOracle(O.LlamaOracle(dcfg, dw, M, "FI"))
    target = O.EngineOracle(O.LlamaOracle(tcfg, tw, M, "TG"))
    torch.manual_seed(1000)                          # prompt 0's seed in the GPU arms
    prompt = synthetic_prompts(1, prefix)[0]
    tree = (O.GreedyTreeOracle(draft, target, prompt, grow_map, max_length=M) if greedy else
            O.SpecTreeOracle(draft, target, prompt, grow_map, temperature=T, top_p=top_p, max_length=M))
    length = prefix
    for _ in range(warm_iters):                      # first iteration = prefill of the target (untimed, like the GPU arm)
        tree.construct_grow_map()
        valid, _, _, term = tree.verify()
        length = valid.shape[0]
    init_s = time.time() - t0
    iters = tokens = 0
    t1 = time.time()
    while iters < max_iters and (time.time() - t1) < max_seconds and not term and length < max_len:
        tree.construct_grow_map()
        valid, _, _, term = tree.verify()
        tokens += valid.shape[0] - length
        length = valid.shape[0]
        iters += 1
    dt = time.time() - t1
    return {"value": round(tokens / dt, 4) if dt > 0 and iters else None, "unit": "tokens/s", "cores": ncores,
            "kind": "port", "ms_per_step": round(dt / max(iters, 1) * 1e3, 1), "steps_timed": iters,
            "accepted_tokens_per_step": round(tokens / max(iters, 1), 3),
            "same_weights_as_gpu_arm": bool(same_d and same_t),
            "sample": f"{iters} steady decode iteration(s) of the torch-CPU oracle (fp16, {ncores} threads) on the same "
                      f"shapes/growmap/prompt after 1 untimed prefill iteration; "
                      + ("same random-init weights as the GPU arm" if same_d and same_t else
                         "no CUDA device: target layers alias one layer's CPU-drawn weights") + f" (init {init_s:.0f}s)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dname, tname, gm_path, greedy, T, top_p, M, prefix, max_len = CONFIGS[args.config]
    S = torch.load(os.path.join(ROOT, gm_path))["size"]
    cb = cpu_reference(args.config, max_seconds=150.0, max_iters=max(args.steps, 1), warm_iters=1)
    out = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "tokens/s",
           "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f16", "data": "synthetic (random-init weights, random prompts)",
           "config": {"workload": f"{args.config}: {dname}->{tname}, {os.path.basename(gm_path)} (tree {S}), "
                                  f"{'greedy' if greedy else 'stochastic'} T={T} P={top_p} M={M}, prefix {prefix}->{max_len} tokens",
                      "accepted_tokens_per_step": cb["accepted_tokens_per_step"], "parallelism": "host CPU"},
           "cpu_baseline": cb, "gpu_launches": 0,
           "e2e": {"value": cb["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=list(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-micro", action="store_true", help="skip the per-kernel micro timings (for ncu launch lists)")
    ap.add_argument("--no-reference-gpu", action="store_true", help="skip the reference-on-this-GPU arm (N=1)")
    ap.add_argument("--no-tp-parity", action="store_true", help="skip the TP-vs-unsharded parity check (N>1)")
    ap.add_argument("--timeline", default=None, help="write a per-kernel in-graph device-time table (markdown) of the timed "
                                                     "steps to this file (torch.profiler; the run's value is then not a bench number)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
