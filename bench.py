#!/usr/bin/env python
"""bench.py - the SAM-Decoding draft-retrieval hot path on B200 (see DESIGN.md, "Measurement").

Headline workload (BASELINE.json configs[1], "c2"): 1024 concurrent requests, 8192-token prompts;
every step each request appends 1-8 accepted tokens to its dynamic suffix automaton and then
performs one suffix-match + draft query (DraftModel.update + DraftModel.lookup of the reference).
  value  = queries/s, inputs resident in HBM, the K timed steps replayed as one CUDA graph
  e2e    = the same through the public API with host buffers (H2D of tokens/counts/start tokens
           and D2H of the drafts inside the timed region, one sync per step)
Extra objects on the same JSON line: `verify` (config c4: fused verify + KV compaction,
us/step and GB/s against the HBM roofline) and `static` (config c3 at a host-buildable corpus size).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
With --dump-outputs the headline's last timed step (drafts, lengths, sources, match lengths, state indices) goes to
DIR/<name>.npy; the inputs are seeded, so two builds run with the same arguments can be compared array for array.
Under torchrun (N > 1) every rank runs the same per-GPU workload on its own requests (weak
scaling, no data-path collective); rank 0 prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(REPO, "sam-decoding_b200"))

METRIC = "suffix_match_draft_queries_per_sec"
UNIT = "queries/s"
N_PREDICTS = 16
LEN_BIAS = 5
LEN_THRESHOLD = 5
VOCAB = 32000


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--requests", type=int, default=1024)
    ap.add_argument("--prompt", type=int, default=8192)
    ap.add_argument("--no-extras", action="store_true", help="skip the c3 / c4 side measurements")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--kv-len", type=int, default=2048, help="KV cache length of the c4 side measurement")
    ap.add_argument("--verify-vocab", type=int, default=32000)
    ap.add_argument("--static-tokens", type=int, default=50_000_000, help="corpus size of the c3 side measurement")
    ap.add_argument("--only-static", action="store_true", help="run only the c3 static-SAM measurement (e.g. at 50M tokens)")
    ap.add_argument("--check-static", action="store_true", help="with --only-static: compare 4 steps x 4096 queries with the C oracle")
    ap.add_argument("--l2-mb", type=int, default=0, help="with --only-static: also time with this many MB of state records pinned in L2")
    ap.add_argument("--only-verify", action="store_true", help="profiling aid: run only the c4 verify loop")
    ap.add_argument("--only-step", action="store_true", help="profiling aid: run only the c2 device loop")
    ap.add_argument("--only-c1", action="store_true", help="run only the c1 (one request) measurement")
    ap.add_argument("--only-tree", action="store_true", help="run only the sam_only static tree drafter measurement")
    ap.add_argument("--scouts", type=int, default=2, help="profiling aid: scout warps of the step kernel (0 none, 1 cursor scouts, 2 all)")
    ap.add_argument("--tma", type=int, default=None, help="tuning aid: 1 bulk-copy staged / 0 register staged logits stream of the verify kernel")
    ap.add_argument("--even-items", type=int, default=None, help="tuning aid: 1 even / 0 all-warps phase-1 item split of the verify kernel")
    ap.add_argument("--overlap", type=int, default=None, help="tuning aid: 1 overlapped / 0 two-barrier flow of the verify kernel")
    ap.add_argument("--lean", type=int, default=None, help="tuning aid: 1 lean / 0 wide build of the step kernel (default: by batch size)")
    ap.add_argument("--ngram", type=int, default=None, help="tuning aid: depth of the short-context scouts (-1 off)")
    ap.add_argument("--prewalk", type=int, default=None, help="tuning aid: draft tokens the scouts walk ahead for the next step")
    ap.add_argument("--variant", type=int, default=1, help="step kernel variant: 1 = one thread per request (default), 0 = warp-cooperative (round 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of the headline workload as DIR/<name>.npy (float64)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and (a.impl != "ours" or a.only_verify or a.only_static or a.only_tree or a.only_c1):
        ap.error("--dump-outputs needs the headline workload of --impl ours")
    return a


# --------------------------------------------------------------------------------------
# synthetic workload (shared by both arms)
# --------------------------------------------------------------------------------------
def _gen_stream(args):
    from samd_b200 import synth
    r, total, seed0 = args
    return synth.copy_mix(total, VOCAB, seed0 + r).astype(np.int32)


def make_workload(n_requests, prompt, n_steps, seed0, procs=None):
    """streams [R, total]; counts [S, R] ~ U{1..8}; per-step token blocks and start tokens."""
    from multiprocessing import Pool
    total = prompt + 8 * n_steps + 1
    procs = procs or min(os.cpu_count() or 1, 32)
    jobs = [(r, total, seed0) for r in range(n_requests)]
    if procs > 1 and n_requests >= 64:
        with Pool(procs) as pool:
            streams = pool.map(_gen_stream, jobs, chunksize=max(1, n_requests // (procs * 4)))
    else:
        streams = [_gen_stream(j) for j in jobs]
    streams = np.stack(streams)
    rng = np.random.default_rng(seed0 + 777)
    counts = rng.integers(1, 9, size=(n_steps, n_requests)).astype(np.int32)
    ends = prompt + np.cumsum(counts, axis=0)                      # position after each step
    begins = ends - counts
    tokens = np.zeros((n_steps, n_requests, 8), dtype=np.int32)
    cols = np.arange(8)[None, None, :]
    idx = np.minimum(begins[:, :, None] + cols, total - 1)
    rows = np.arange(n_requests)[None, :, None]
    tokens = np.where(cols < counts[:, :, None], streams[rows, idx], 0).astype(np.int32)
    start = streams[np.arange(n_requests)[None, :], ends].astype(np.int32)
    return streams, counts, tokens, start


def _gate():
    """A short spin kernel (about 200 us) in front of a device-timed region: the stream stays busy while the host enqueues the
    start event and the graph launch, so the start event's timestamp is taken when the work is ready to run - device
    time, not the host's cudaGraphLaunch latency (which a 20-step run would otherwise carry as 1.2 us per step)."""
    import torch
    torch.cuda._sleep(int(os.environ.get("SAMD_BENCH_GATE_CYCLES", "400000")))


# --------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# --------------------------------------------------------------------------------------
class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.lines, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()

    def summary(self, t0=None, t1=None):
        sm, smax, reasons = [], [], set()
        for ts, line in self.lines:
            if t0 is not None and not (t0 - 0.15 <= ts <= t1 + 0.15):
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's Python path (oracle/samd_oracle.py)
# --------------------------------------------------------------------------------------
def _cpu_worker(job):
    """One worker = a block of requests: untimed prefill, then timed steps (extend + lookup + draft)."""
    sys.path.insert(0, os.path.join(REPO, "oracle"))
    import samd_oracle as O
    streams, counts, tokens, start, prompt, w0, w1 = job
    sams = []
    for s in streams:
        a = O.Automaton()
        a.extend(s[:prompt].tolist())
        sams.append(a)
    R = len(sams)

    def run(step_lo, step_hi):
        t0 = time.perf_counter()
        for s in range(step_lo, step_hi):
            for r in range(R):
                a = sams[r]
                a.extend(tokens[s, r, :counts[s, r]].tolist())
                O.select_samd(a, None, int(start[s, r]), N_PREDICTS, LEN_BIAS, LEN_THRESHOLD)
        return time.perf_counter() - t0

    run(0, w0)
    return run(w0, w1)


class _NoTree:
    """Stand-in for the tree-model fallback of samd's DraftModel (Token Recycle / EAGLE are outside the c2 metric; the GPU
    arm also only reports `type = tree model` for those queries): gen_draft answers at once."""

    def reset(self):
        pass

    def update(self, **kwargs):
        pass

    def gen_draft(self, start_token):
        return [start_token], {}


def _cpu_worker_ref(job):
    """The same block of work through the reference's OWN classes (samd.DynSAM + samd.DraftModel.lookup), loaded
    unmodified from baseline/_ref."""
    import contextlib
    import io
    sys.path.insert(0, os.path.join(REPO, "oracle"))
    import ref_loader
    assert ref_loader.use_staged(), "baseline/_ref is missing: python baseline/stage_reference.py"
    with contextlib.redirect_stdout(io.StringIO()):
        ns = ref_loader.load()
        cfg = ns.samd_config.SamdConfig(n_predicts=N_PREDICTS, len_bias=LEN_BIAS, len_threshold=LEN_THRESHOLD)
    streams, counts, tokens, start, prompt, w0, w1 = job
    drafts = []
    for s in streams:
        d = ns.samd_draft.DraftModel(cfg, tree_model=_NoTree(), lm=None, device="cpu")     # NullStaticSAM, fresh DynSAM
        d.reset()
        d.sam_dyn.add_tokens(s[:prompt].tolist())
        drafts.append(d)
    R = len(drafts)

    def run(step_lo, step_hi):
        t0 = time.perf_counter()
        for s in range(step_lo, step_hi):
            for r in range(R):
                d = drafts[r]
                tk = tokens[s, r, :counts[s, r]].tolist()
                d.sam_dyn.add_tokens(tk)               # DraftModel.update (samd/draft.py:65-79) minus the tree model
                d.sam_static.transfer_tokens(tk)
                d.lookup(int(start[s, r]))             # samd/draft.py:52-63
        return time.perf_counter() - t0

    run(0, w0)
    return run(w0, w1)


def _cpu_worker_c(job):
    """Same block of work through the oracle's C restatement (oracle/sam_oracle.c)."""
    import ctypes as C
    sys.path.insert(0, os.path.join(REPO, "oracle"))
    import c_oracle as CO
    streams, counts, tokens, start, prompt, w0, w1 = job
    R = len(streams)
    sams = [CO.CSam(streams.shape[1] + 8) for _ in range(R)]
    for a, s in zip(sams, streams):
        a.extend(s[:prompt])
    arr = (CO.vp * R)(*[a.h for a in sams])
    tk = np.ascontiguousarray(tokens.transpose(0, 1, 2), dtype=np.int32)
    ct = np.ascontiguousarray(counts, dtype=np.int32)
    st = np.ascontiguousarray(start, dtype=np.int32)
    run = lambda lo, hi: CO.lib().so_run_steps(arr, R, CO._p(tk), CO._p(ct), CO._p(st), lo, hi, N_PREDICTS, LEN_BIAS, LEN_THRESHOLD)
    run(0, w0)
    t0 = time.perf_counter()
    run(w0, w1)
    return time.perf_counter() - t0


def cpu_arm(n_sample, prompt, steps, warmup, seed0, cores, worker=None):
    """Returns (queries/s, per-worker max wall seconds, description) on a bounded sample."""
    from multiprocessing import Pool
    streams, counts, tokens, start = make_workload(n_sample, prompt, steps + warmup, seed0, procs=1)
    per = max(1, n_sample // cores)
    jobs = []
    for c in range(0, n_sample, per):
        sl = slice(c, min(n_sample, c + per))
        jobs.append((streams[sl], counts[:, sl], tokens[:, sl], start[:, sl], prompt, warmup, warmup + steps))
    with Pool(len(jobs)) as pool:
        walls = pool.map(worker or _cpu_worker, jobs)
    wall = max(walls)
    return n_sample * steps / wall, wall, len(jobs)


def have_staged_reference():
    return os.path.isdir(os.path.join(REPO, "baseline", "_ref", "samd", "sam"))


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = min(os.cpu_count() or 1, 32)
    real = have_staged_reference()
    # bounded sample: a step of the reference arm is one pass over `n_sample` requests of the c2 workload
    n_sample = cores * (16 if real else 64)
    steps, warm = a.steps, a.warmup
    t0 = time.time()
    qps, wall, used = cpu_arm(n_sample, a.prompt, steps, warm, 2000, cores, worker=_cpu_worker_ref if real else None)
    if real:
        kind = "reference"
        what = ("the reference's own classes, unmodified, from baseline/_ref: samd.DraftModel with a fresh samd.DynSAM and "
                "NullStaticSAM per request - sam_dyn.add_tokens + sam_static.transfer_tokens + DraftModel.lookup per step (the "
                "tree-model fallback stubbed out, as in the GPU arm), one Python process per core")
    else:
        kind = "port"
        what = ("baseline/_ref not staged on this machine: oracle/samd_oracle.py, the Python port of samd DynSAM + "
                "DraftModel.lookup, one process per core")
    out = {
        "impl": "reference", "metric": METRIC, "value": qps, "unit": UNIT, "n_gpus": a.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": wall / steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic",
        "config": workload_config(a, a.requests),   # the GPU arm's config; the bounded sample is described in cpu_baseline
        "cpu_baseline": {"value": qps, "unit": UNIT, "cores": used, "kind": kind,
                         "sample": f"{n_sample} requests x {steps} steps of the c2 workload (prefill untimed); {what}"},
        "e2e": {"value": qps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.time() - t0,
    }
    print(json.dumps(out))


def workload_config(a, requests):
    return {"workload": f"c2: batched dynamic SAM, {requests} concurrent requests x {a.prompt}-token prompts, "
                        f"1-8 accepted tokens appended per step then one suffix-match+draft query "
                        f"(samd flavour, n_predicts={N_PREDICTS}, len_bias={LEN_BIAS}, len_threshold={LEN_THRESHOLD})",
            "requests_per_gpu": requests, "prompt_tokens": a.prompt, "vocab": VOCAB,
            "l2": "no flush: per-GPU arena working set (~1.4 GB) exceeds the 126 MB L2",
            "parallelism": f"requests sharded over {a.gpus} GPU(s), no collective"}


# --------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------
def run_ours(a):
    import torch
    import torch.distributed as dist
    from samd_b200 import _cabi as K, engine as E

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # keep stdout to the single JSON line
        dist.init_process_group("nccl", device_id=dev)
    K.require_device()
    K.lib().samd_step_set_variant(a.variant)
    K.lib().samd_step_set_scouts(a.scouts)
    if a.prewalk is not None:
        K.lib().samd_step_set_prewalk(a.prewalk)
    if a.ngram is not None:
        K.lib().samd_step_set_ngram(a.ngram)
    if a.lean is not None:
        K.lib().samd_step_set_lean(a.lean)
    if a.overlap is not None:
        K.lib().samd_verify_set_overlap(a.overlap)
    if a.even_items is not None:
        K.lib().samd_verify_set_even_items(a.even_items)
    if a.tma is not None:
        K.lib().samd_verify_set_tma(a.tma)
    launches0 = E.launch_count()
    if a.only_verify:                         # profiling aid (ncu): just the c4 loop
        print(json.dumps({"verify": bench_verify(a, dev, 6458.1, iters=6, warm=2)}))
        return
    if a.only_static:
        print(json.dumps({"static": bench_static(a, dev, n_corpus=a.static_tokens, check=a.check_static, l2_mb=a.l2_mb)}))
        return
    if a.only_tree:
        print(json.dumps({"sam_only_tree": bench_tree_drafter(a, dev)}))
        return
    if a.only_c1:
        print(json.dumps({"c1": bench_c1(a, dev)}))
        return
    if a.only_step:
        a.no_extras = a.no_cpu = True
    R, N, S, W = a.requests, a.prompt, a.steps, a.warmup
    t_setup = time.time()
    streams, counts, tokens, start = make_workload(R, N, S + W, 2000 + 100000 * rank)
    max_tokens = N + 8 * (S + W) + 16
    dyn = E.DynSamBatch(R, max_tokens, dev)
    snap = E.DynSamBatch(R, max_tokens, dev)
    eng = E.DraftEngine(dyn, None, K.FLAVOUR_SAMD, n_predicts=N_PREDICTS, len_bias=LEN_BIAS, len_threshold=LEN_THRESHOLD)
    d_tokens = torch.as_tensor(tokens).to(dev)
    d_counts = torch.as_tensor(counts).to(dev)
    d_start = torch.as_tensor(start).to(dev)
    # prefill (untimed): DraftModel.update(prompt) for every request
    d_prompt = torch.as_tensor(streams[:, :N]).to(dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    eng.step(d_prompt, None, None)
    ev1.record()
    torch.cuda.synchronize()
    prefill_ms = ev0.elapsed_time(ev1)
    del d_prompt

    def step(s):
        eng.step(d_tokens[s], d_counts[s], d_start[s])

    # The arenas as the prefill left them: every measured pass below starts from this snapshot and runs its W warm-up
    # steps (real steps 0..W-1) right before its K timed ones (steps W..W+K-1), so that the timed region never follows
    # the 2.8 GB restore copy directly (that copy leaves the TLBs and the L2 cold: +40 us on a first device step, +80-120 us
    # on a first host-path step - an artefact that a short run (K = 20) would mostly measure).
    snap.copy_from(dyn)
    torch.cuda.synchronize()

    def warm():
        dyn.copy_from(snap)
        for s in range(W):                   # warm-up steps 0..W-1, eager
            step(s)
        torch.cuda.synchronize()

    # the K timed steps as one CUDA graph; one dry replay (untimed) instantiates and uploads it
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for s in range(W, W + S):
            step(s)
    g.replay()
    torch.cuda.synchronize()

    clocks = Clocks(local)
    clocks.start()
    time.sleep(0.3)
    warm()
    stats0 = dyn.stats()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    wall0 = time.time()
    _gate()
    ev0.record()
    g.replay()
    ev1.record()
    torch.cuda.synchronize()
    wall1 = time.time()
    if world > 1:
        dist.barrier()
    dev_ms = ev0.elapsed_time(ev1)
    stats1 = dyn.stats()
    assert stats1["overflowed"] == 0, "arena overflow in the timed region"
    draft_checksum = int(eng.draft.sum().item())
    last_step = step_outputs(eng) if a.dump_outputs and rank == 0 else None

    # per-launch duration of the step kernel, measured live with CUDA events (eager launches)
    warm()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(S)]
    for i, s in enumerate(range(W, W + S)):
        evs[i][0].record()
        step(s)
        evs[i][1].record()
    torch.cuda.synchronize()
    kern_ms = float(np.mean([x.elapsed_time(y) for x, y in evs]))

    # e2e: host buffers in, drafts out, through the public engine API (DraftEngine.step_host): per step the caller
    # stages its inputs (counts | start tokens | accepted tokens) in a pinned buffer; one staging-copy kernel
    # (samd_stage_copy: 16-byte coalesced PCIe reads) brings them into a device block, the step kernel reads that and
    # writes every output (type, match lengths, state indices, draft length, draft tokens) straight into mapped pinned
    # host memory; then the stream is synchronised.  Measured host to host: 35.8 us this way, 39.8 fully zero-copy,
    # 38.6 with a copy kernel on both sides, 49.7 with copy-engine memcpys.  h2d / d2h bytes are the sizes of those two
    # host buffers.
    inp, res = eng.host_buffers(8)
    h_in = torch.empty(W + S, inp.numel(), dtype=torch.int32).pin_memory()
    h_in[:, :R] = torch.as_tensor(counts)
    h_in[:, R:2 * R] = torch.as_tensor(start)
    h_in[:, 2 * R:] = torch.as_tensor(tokens).reshape(W + S, R * 8)
    inp_np, h_np = inp.numpy(), h_in.numpy()
    staged = [h_np[s] for s in range(W + S)]     # (row views made outside the timed loop; the copies are inside)
    # The pre-generated input rows are read once so that the per-step staging copy finds them in the CPU cache, as a
    # caller's freshly produced tokens would be (cold rows cost 4 us per step more: a property of pre-generating 11 MB
    # of inputs, not of the path).
    h_in_checksum = int(h_in.sum())
    dyn.copy_from(snap)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    for s in range(W):                       # the W warm-up steps (0..W-1) through the host path itself
        np.copyto(inp_np, staged[s])
        eng.step_host(inp, res)
    e2e_t0 = time.perf_counter()
    ev0.record()
    diag_ts = [] if os.environ.get("SAMD_BENCH_E2E_DIAG") else None
    for s in range(W, W + S):
        np.copyto(inp_np, staged[s])         # the caller's host-side staging of this step's inputs (40 KB into the pinned buffer)
        eng.step_host(inp, res)
        if diag_ts is not None:
            diag_ts.append(time.perf_counter())
    ev1.record()
    torch.cuda.synchronize()
    e2e_wall = time.perf_counter() - e2e_t0
    e2e_ms = max(ev0.elapsed_time(ev1), e2e_wall * 1e3)
    clocks.stop()
    assert int(res[6 * R:].sum().item()) == draft_checksum, "e2e and device runs disagree"
    if os.environ.get("SAMD_BENCH_E2E_DIAG"):
        d = np.diff(np.array([e2e_t0] + diag_ts)) * 1e6
        print("e2e diag first pass per-step us: p10 %.1f p50 %.1f p90 %.1f p99 %.1f max %.1f; first 8:" % tuple(np.percentile(d, [10, 50, 90, 99, 100])),
              np.round(d[:8], 1), "steps > 60 us:", np.nonzero(d > 60)[0].tolist(), np.round(d[d > 60], 0).tolist(), file=sys.stderr)
        for rep in range(3):
            dyn.copy_from(snap)
            torch.cuda.synchronize()
            for s in range(W):
                np.copyto(inp_np, staged[s])
                eng.step_host(inp, res)
            t0 = time.perf_counter()
            for s in range(W, W + S):
                np.copyto(inp_np, staged[s])
                eng.step_host(inp, res)
            print("e2e diag rep", rep, (time.perf_counter() - t0) / S * 1e6, "us/step; first pass", e2e_wall / S * 1e6, e2e_ms / S * 1e3, file=sys.stderr)
    h2d = inp.numel() * 4
    d2h = res.numel() * 4

    # max over ranks
    if world > 1:
        t = torch.tensor([dev_ms, e2e_ms, kern_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_ms, kern_ms = (float(x) for x in t.tolist())
    queries = R * S * world
    value = queries / (dev_ms * 1e-3)
    e2e_value = queries / (e2e_ms * 1e-3)

    # algorithmic bytes per launch from the kernel's own counters (DESIGN.md "algorithmic bytes")
    d = {k: stats1[k] - stats0[k] for k in stats1}
    appended = d["tokens"]
    a_tok = 20 * appended + 16 * d["n_edges"] + 16 * d["n_clones"] + 28 * d["extend_probes"]
    a_q = R * S * (4 * (N_PREDICTS - 1) + 4 * N_PREDICTS + 16 + 12) + 28 * d["lookup_probes"]
    alg_bytes_per_launch = (a_tok + a_q) / S
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "B200_PROFILING.md fallback 6650"
    # launch duration = graph-replayed step time (pure device time; the eager per-launch events above also
    # contain host enqueue gaps and are reported separately)
    launch_ms = dev_ms / S
    achieved = alg_bytes_per_launch / (launch_ms * 1e-3) / 1e9
    traffic = {}
    try:
        traffic = json.load(open(os.path.join(REPO, "profiles", "traffic.json")))
    except Exception:
        pass
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": S, "warmup": W,
        "ms_per_step": dev_ms / S, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic", "config": workload_config(a, R),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms / S, "gpu_launches_per_step": 2, "host_mode": eng.HOST_MODE},
        "gpu_launches": None,
        "roofline": {"kernel": "sam_step_scalar_kernel" if a.variant == 1 else "sam_step_kernel", "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                     "frac": achieved / hbm_peak, "traffic": traffic.get("sam_step_scalar_kernel" if a.variant == 1 else "sam_step_kernel", {}).get("bytes_per_launch"),
                     "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg_bytes_per_launch, "launch_us": launch_ms * 1e3,
                     "note": "latency-bound pointer chase: queries/s and probes/query are the figures of merit"},
        "step_kernel": {"us_per_launch_events": kern_ms * 1e3, "us_per_step_graph": dev_ms / S * 1e3,
                        "appended_tokens_per_step": appended / S, "probes_per_appended_token": d["extend_probes"] / max(1, appended),
                        "edge_inserts_per_token": d["n_edges"] / max(1, appended), "clones_per_token": d["n_clones"] / max(1, appended),
                        "probes_per_lookup": d["lookup_probes"] / (R * S), "prefill_ms": prefill_ms,
                        "prefill_tokens_per_s": R * N / (prefill_ms * 1e-3), "arena_bytes": dyn.nbytes},
        "clocks": clocks.summary(wall0, wall1),
        "clocks_whole_run": clocks.summary(),
        "setup_s": time.time() - t_setup,
    }
    del g, snap, h_in, d_tokens
    torch.cuda.empty_cache()
    if rank == 0 and world == 1 and not a.no_extras:
        try:
            out["verify"] = bench_verify(a, dev, hbm_peak)
            out["verify"]["roofline"]["traffic"] = traffic.get("verify_compact_kernel", {}).get("bytes_per_launch")
        except Exception as e:  # side measurement must not kill the headline line
            out["verify"] = {"error": repr(e)}
        try:                                  # config c5's verification half: Llama-3 vocabulary and KV shape
            torch.cuda.empty_cache()
            out["verify_c5"] = bench_verify(a, dev, hbm_peak, vocab=128256, heads=8, kv_len=8192, name="c5", recycle=False)
        except Exception as e:
            out["verify_c5"] = {"error": repr(e)}
        torch.cuda.empty_cache()
        try:
            out["static"] = bench_static(a, dev, n_corpus=a.static_tokens)
        except Exception as e:
            out["static"] = {"error": repr(e)}
        try:
            out["c2_concurrent"] = bench_c2_concurrent(a, dev, (streams, counts, tokens, start))
        except Exception as e:
            out["c2_concurrent"] = {"error": repr(e)}
        try:
            out["c2_sam_only"] = bench_c2_sam_only(a, dev, (streams, counts, tokens, start))
        except Exception as e:
            out["c2_sam_only"] = {"error": repr(e)}
        try:
            out["c1"] = bench_c1(a, dev)
        except Exception as e:
            out["c1"] = {"error": repr(e)}
        try:
            out["sam_only_tree"] = bench_tree_drafter(a, dev)
        except Exception as e:
            out["sam_only_tree"] = {"error": repr(e)}
    if rank == 0 and world == 1 and not a.no_cpu:
        # the CPU baseline beside it (rank 0, N = 1 only): the reference's own classes when baseline/_ref is staged, on a
        # bounded sample of the same workload; the Python port and the C restatement of the oracle follow for context
        cores = min(os.cpu_count() or 1, 32)
        if have_staged_reference():
            n_ref = cores * 16
            qps, wall, used = cpu_arm(n_ref, N, 64, 2, 2000, cores, worker=_cpu_worker_ref)
            out["cpu_baseline"] = {"value": qps, "unit": UNIT, "cores": used, "kind": "reference",
                                   "sample": f"{n_ref} requests x 64 steps of the same workload (prefill untimed, {wall:.2f} s of work "
                                             f"per core): the reference's own samd.DynSAM / samd.DraftModel, unmodified, from "
                                             f"baseline/_ref, one Python process per core"}
        n_sample = cores * 64
        qps_p, wall_p, used_p = cpu_arm(n_sample, N, 256, 4, 2000, cores)
        port = {"value": qps_p, "unit": UNIT, "cores": used_p, "kind": "port",
                "sample": f"{n_sample} requests x 256 steps of the same workload (prefill untimed, {wall_p:.2f} s "
                          f"of work per core), Python port of the reference path (oracle/samd_oracle.py)"}
        if "cpu_baseline" in out:
            out["cpu_baseline_port"] = port
        else:
            out["cpu_baseline"] = port
        try:
            qps_c, wall_c, used_c = cpu_arm(n_sample, N, 256, 4, 2000, cores, worker=_cpu_worker_c)
            out["cpu_baseline_c"] = {"value": qps_c, "unit": UNIT, "cores": used_c, "kind": "port",
                                     "sample": f"same sample through the oracle's plain-C restatement (oracle/sam_oracle.c), "
                                               f"{wall_c:.3f} s per core; reported for context - the reference itself is Python"}
        except Exception as e:
            out["cpu_baseline_c"] = {"error": repr(e)}
    if world > 1 and not a.no_extras:
        try:
            res = bench_sharded_static(a, dev, rank, world)
            if rank == 0:
                out["sharded_static"] = res
        except Exception as e:
            if rank == 0:
                out["sharded_static"] = {"error": repr(e)}
    # the whole metric inside `roofline` (BASELINE's metric is a triple: queries/s; verify+KV us/step; GB/s)
    others = {}
    v = out.get("verify")
    if isinstance(v, dict) and "us_per_step" in v:
        others["c4_verify_kv"] = {"us_per_step": v["us_per_step"], "achieved_gbs": v["roofline"]["achieved"], "frac": v["roofline"]["frac"],
                                  "us_verify_only": v["us_per_step_verify_only"], "frac_verify_only": v["roofline_verify_only"]["frac"],
                                  "us_with_token_recycle_top8": v["token_recycle"]["us_per_step_with_top8_table_update"],
                                  "traffic": v["roofline"].get("traffic"), "traffic_note": traffic.get("verify_compact_kernel", {}).get("workload")}
    v = out.get("verify_c5")
    if isinstance(v, dict) and "us_per_step" in v:
        others["c5_verify_kv"] = {"us_per_step": v["us_per_step"], "achieved_gbs": v["roofline"]["achieved"], "frac": v["roofline"]["frac"],
                                  "us_verify_only": v["us_per_step_verify_only"], "frac_verify_only": v["roofline_verify_only"]["frac"]}
    v = out.get("static")
    if isinstance(v, dict) and "queries_per_s" in v:
        others["c3_static_50m"] = {"queries_per_s": v["queries_per_s"], "us_per_step": v["us_per_step"],
                                   "sectors_per_query": traffic.get("static_lookup", {}).get("l1_sectors_per_query"),
                                   "l2_hit": traffic.get("static_lookup", {}).get("l2_hit_rate"),
                                   "l2_window": v.get("l2_window")}
    v = out.get("c2_concurrent")
    if isinstance(v, dict) and "queries_per_s" in v:
        others["c2_concurrent"] = {"queries_per_s": v["queries_per_s"], "us_per_step_per_batch": v["us_per_step_per_batch"],
                                   "e2e_queries_per_s": v["e2e_queries_per_s"]}
    v = out.get("c1")
    if isinstance(v, dict) and "gpu_us_per_step" in v:
        others["c1"] = {k: v[k] for k in v if k != "workload"}
    v = out.get("c2_sam_only")
    if isinstance(v, dict) and "queries_per_s" in v:
        others["c2_sam_only"] = {k: v[k] for k in v if k != "workload"}
    v = out.get("sam_only_tree")
    if isinstance(v, dict) and "trees_per_s" in v:
        others["sam_only_static_tree"] = {k: v[k] for k in v if k != "workload"}
    v = out.get("sharded_static")
    if isinstance(v, dict) and "queries_per_s" in v:
        others["c5_sharded_static"] = {"queries_per_s": v["queries_per_s"], "p2p": v.get("p2p"), "nccl": v.get("nccl"),
                                       "matches_oracle": v.get("matches_oracle")}
    out["roofline"]["others"] = others
    out["roofline"]["sectors_per_query"] = traffic.get("sam_step_lookup", {}).get("l1_sectors_per_query")
    out["roofline"]["l2_hit"] = traffic.get("sam_step_lookup", {}).get("l2_hit_rate")
    out["gpu_launches"] = S          # kernels of ours inside the timed region: one sam_step_kernel per step
    out["gpu_launches_total_process"] = E.launch_count() - launches0
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if last_step is not None:
        save_outputs(a.dump_outputs, last_step)
    if rank == 0:
        print(json.dumps(out))


DUMP_LIMIT_BYTES = 63_000_000      # under 64 MB with the .npy headers


def step_outputs(eng):
    """What DraftEngine.step hands its caller, per request, as float64 (the int32 values are exact): the draft
    [R, n_predicts], its length, the draft source, and match length and state index in the dynamic and static automata."""
    fields = {"draft": eng.draft, "draft_len": eng.draft_len, "type": eng.out_type, "match_dyn": eng.match_dyn,
              "match_static": eng.match_static, "index_dyn": eng.index_dyn, "index_static": eng.index_static}
    return {name: t.cpu().numpy().astype(np.float64) for name, t in fields.items()}


def save_outputs(path, arrays):
    """DIR/<name>.npy for every array; above DUMP_LIMIT_BYTES only a fixed, seeded sample of the requests is kept and
    their indices go to request_index.npy."""
    n = len(arrays["draft"])
    row_bytes = sum(v.nbytes for v in arrays.values()) // n
    if n * row_bytes > DUMP_LIMIT_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT_BYTES // (row_bytes + 8), replace=False))
        arrays = {k: v[keep] for k, v in arrays.items()}
        arrays["request_index"] = keep.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(path, name + ".npy"), v)


def bench_verify(a, dev, hbm_peak, iters=40, warm=5, vocab=None, heads=32, kv_len=None, name="c4", recycle=True):
    """Config c4: fused verify + KV compaction, Vicuna-7B shape (B=64, T=61, V=32000, bf16;
    KV 64 tensors [64,32,kv_len,128] bf16).  Rotates 4 logits buffers (1 GB > L2) between iterations."""
    import torch
    from samd_b200 import engine as E, synth
    B, T, V = 64, 61, vocab or a.verify_vocab
    L, H, DH, ML = 32, heads, 128, max(kv_len or a.kv_len, 256)
    ri_np = synth.tree_retrieve_indices(synth.token_recycle_tree())
    rng = np.random.default_rng(4000)
    tree_tokens = rng.integers(3, V, size=(B, T)).astype(np.int32)
    nbuf = 4
    logits = []
    for i in range(nbuf):
        lg, _ = synth.planted_logits(B, T, V, tree_tokens, ri_np, seed=4000 + i, device=dev)
        logits.append(lg)
    free_b, _ = torch.cuda.mem_get_info(dev)
    kv_bytes = 2 * L * B * H * ML * DH * 2
    if kv_bytes > free_b * 0.8:
        ML = max(256, int(ML * free_b * 0.8 / kv_bytes) // 64 * 64)
    kv_all = torch.empty(2 * L, B, H, ML, DH, dtype=torch.bfloat16, device=dev)
    kv_all.view(torch.int16).random_(0, 30000)
    kv = [kv_all[i] for i in range(2 * L)]
    ver = E.Verifier(B, T, dev)
    ver.bind_kv(kv)
    d_tok = torch.as_tensor(tree_tokens).to(dev)
    d_ri = torch.as_tensor(ri_np).to(dev)
    cache0 = cache_len = res = None

    def run(n, move, recycle=None):
        """n launches (rotating logits buffers) captured as ONE CUDA graph and replayed: per-launch time is pure
        device time, free of host enqueue gaps.  cache_len keeps growing inside a replay (reset between replays)."""
        outs = [ver.verify(logits[i], d_tok, d_ri, cache_len=cache_len, move_kv=move, recycle=recycle) for i in range(nbuf)]   # warm + allocate
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for i in range(n):
                ver.verify(logits[i % nbuf], d_tok, d_ri, cache_len=cache_len, move_kv=move, out=outs[i % nbuf], recycle=recycle)
        times = []
        for rep in range(7):
            cache_len.copy_(cache0)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            _gate()
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / n)
        cache_len.copy_(cache0)
        res_local = ver.verify(logits[0], d_tok, d_ri, cache_len=cache_len, move_kv=move, out=outs[0], recycle=recycle)
        torch.cuda.synchronize()
        return times[2:], res_local

    n_graph = 16
    cache0 = torch.randint(min(256, ML // 4), max(min(1900, ML - 80) - 6 * n_graph, min(256, ML // 4) + 1), (B,),
                           dtype=torch.int32, device=dev)
    cache_len = cache0.clone()
    t_full, res = run(n_graph, True)
    t_nokv, _ = run(n_graph, False)
    # Token Recycle's top-8 table update riding on the same pass (SURVEY 8f row 2), and what it replaces: a second
    # full read of the logits by torch.topk
    table = E.RecycleTable(synth.token_recycle_tree(), V, dev)
    t_rec = [float("nan")]
    if recycle:
        t_rec, _ = run(n_graph, True, recycle=table)
    tk = []
    for i in range(6 if recycle else 0):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        logits[i % nbuf].topk(8)
        e1.record()
        tk.append((e0, e1))
    torch.cuda.synchronize()
    us_torch_topk = float(np.median([x.elapsed_time(y) for x, y in tk][2:])) * 1e3 if recycle else float("nan")
    cache_len.copy_(cache0)
    res = ver.verify(logits[0], d_tok, d_ri, cache_len=cache_len, move_kv=True, out=res)
    torch.cuda.synchronize()
    # the same row moves through the stand-alone compaction entry point (samd_kv_compact), for attribution
    from samd_b200 import _cabi as K
    m = ver._kv_meta
    t_kv = []
    for i in range(iters):
        cache_len.copy_(cache0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        K.check(K.lib().samd_kv_compact(ver._kv_ptrs.data_ptr(), m["n_kv"], m["n_heads"], m["row_bytes"], m["batch_stride"],
                                        m["head_stride"], m["pos_stride"], res["indices"].data_ptr(), res["indices"].shape[1],
                                        res["accept_len"].data_ptr(), cache_len.data_ptr(), B, K.stream_ptr()))
        e1.record()
        t_kv.append((e0, e1))
    torch.cuda.synchronize()
    us_kv_alone = float(np.median([x.elapsed_time(y) for x, y in t_kv])) * 1e3
    acc = res["accept_len"].cpu().numpy()
    idx = res["indices"].cpu().numpy()
    moved = int(sum(int((idx[b, :acc[b]] != np.arange(acc[b])).sum()) for b in range(B)))
    row_bytes = 2 * L * H * DH * 2
    logit_bytes = B * T * V * 2 + B * T * 4 + ri_np.size * 4
    kv_bytes_moved = 2 * moved * row_bytes
    us_full, us_nokv = float(np.median(t_full)) * 1e3, float(np.median(t_nokv)) * 1e3
    gbs_full = (logit_bytes + kv_bytes_moved) / (us_full * 1e-6) / 1e9
    gbs_nokv = logit_bytes / (us_nokv * 1e-6) / 1e9
    return {"workload": f"{name}: fused tree verification + KV compaction, B={B} T={T} V={V} bf16, 30x6 path table, "
                        f"KV {2 * L}x[{B},{H},{ML},{DH}] bf16; 4 rotating logits buffers (1 GB > L2)",
            "us_per_step": us_full, "us_per_step_p10": float(np.percentile(t_full, 10)) * 1e3,
            "us_per_step_p90": float(np.percentile(t_full, 90)) * 1e3, "us_per_step_verify_only": us_nokv,
            "algorithmic_bytes": logit_bytes + kv_bytes_moved, "logits_bytes": logit_bytes, "kv_bytes_moved": kv_bytes_moved,
            "kv_rows_moved": moved, "mean_accept_len": float(acc.mean()), "us_kv_compact_standalone": us_kv_alone,
            "kv_standalone_gbs": kv_bytes_moved / (us_kv_alone * 1e-6) / 1e9,
            "roofline": {"kernel": "verify_compact_kernel", "bound": "hbm", "achieved": gbs_full, "peak": hbm_peak,
                         "unit": "GB/s", "frac": gbs_full / hbm_peak, "traffic": None},
            "roofline_verify_only": {"achieved": gbs_nokv, "peak": hbm_peak, "unit": "GB/s", "frac": gbs_nokv / hbm_peak},
            "gpu_launches_per_step": 1,
            "token_recycle": {"us_per_step_with_top8_table_update": float(np.median(t_rec)) * 1e3,
                              "us_torch_topk_separate_pass": us_torch_topk,
                              "note": "top-8 of all B*T rows + table[token] update fused into the verify launch"}}


def bench_c2_sam_only(a, dev, workload):
    """c2 in the samd_sam_only flavour (SURVEY 8d: max_predicts = 40, alpha = 4): same streams and steps as the headline,
    the draft is the unpadded continuation of up to 40 tokens (samd_sam_only/sam/dyn_sam.py gen_draft)."""
    import torch
    from samd_b200 import _cabi as K, engine as E
    streams, counts, tokens, start = workload
    R, N, S, W = a.requests, a.prompt, a.steps, a.warmup
    d_tokens, d_counts, d_start = (torch.as_tensor(x).to(dev) for x in (tokens, counts, start))
    dyn = E.DynSamBatch(R, N + 8 * (S + W) + 16, dev)
    eng = E.DraftEngine(dyn, None, K.FLAVOUR_SAM_ONLY, n_predicts=40, len_bias=LEN_BIAS, len_threshold=LEN_THRESHOLD, alpha=4.0)
    eng.step(torch.as_tensor(streams[:, :N]).to(dev), None, None)
    torch.cuda.synchronize()
    snap = E.DynSamBatch(R, dyn.max_tokens, dev)
    snap.copy_from(dyn)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for s in range(W, W + S):
            eng.step(d_tokens[s], d_counts[s], d_start[s])
    g.replay()                               # dry replay, then the arenas as the prefill left them and the W warm-up steps
    dyn.copy_from(snap)
    for s in range(W):
        eng.step(d_tokens[s], d_counts[s], d_start[s])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    _gate()
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    return {"workload": f"c2, samd_sam_only flavour: {R} requests x {N}-token prompts, max_predicts 40, alpha 4",
            "queries_per_s": R * S / (ms * 1e-3), "us_per_step": ms / S * 1e3,
            "mean_draft_len": float(eng.draft_len.float().mean().item())}


def bench_c2_concurrent(a, dev, workload, n_streams=4):
    """Context for the headline: the step kernel is a latency-bound pointer chase that keeps ~6 % of the SM
    warp slots busy, so independent 1024-request batches overlap almost perfectly.  n_streams batches (own
    arenas, same token streams) run as n_streams CUDA graphs on n_streams streams; aggregate queries/s."""
    import torch
    from samd_b200 import _cabi as K, engine as E
    streams, counts, tokens, start = workload
    R, N, S, W = a.requests, a.prompt, a.steps, a.warmup
    d_tokens, d_counts, d_start = (torch.as_tensor(x).to(dev) for x in (tokens, counts, start))
    d_prompt = torch.as_tensor(streams[:, :N]).to(dev)
    cuda_streams = [torch.cuda.Stream(dev) for _ in range(n_streams)]
    engines, graphs = [], []
    for cs in cuda_streams:
        with torch.cuda.stream(cs):
            dyn = E.DynSamBatch(R, N + 8 * (S + W) + 16, dev)
            eng = E.DraftEngine(dyn, None, K.FLAVOUR_SAMD, n_predicts=N_PREDICTS, len_bias=LEN_BIAS, len_threshold=LEN_THRESHOLD)
            eng.step(d_prompt, None, None)
        engines.append(eng)
    torch.cuda.synchronize()
    snaps = []
    for eng in engines:                      # the arenas as the prefill left them
        snap = E.DynSamBatch(R, N + 8 * (S + W) + 16, dev)
        snap.copy_from(eng.dyn)
        snaps.append(snap)
    for eng, cs in zip(engines, cuda_streams):
        with torch.cuda.stream(cs):
            for s in range(W):               # warm-up steps right before the timed ones
                eng.step(d_tokens[s], d_counts[s], d_start[s])
    torch.cuda.synchronize()
    for eng, cs in zip(engines, cuda_streams):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=cs):
            for s in range(W, W + S):
                eng.step(d_tokens[s], d_counts[s], d_start[s])
        graphs.append(g)
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True)
    ends = [torch.cuda.Event(enable_timing=True) for _ in cuda_streams]
    _gate()
    e0.record()
    for g, cs, ev in zip(graphs, cuda_streams, ends):
        cs.wait_event(e0)
        with torch.cuda.stream(cs):
            g.replay()
            ev.record()
    torch.cuda.synchronize()
    ms = max(e0.elapsed_time(ev) for ev in ends)
    # the same through the host-buffer entry: per step every batch stages its inputs in its pinned buffer and calls
    # step_host(sync=False) on its own stream; the streams are synchronised before the buffers are reused
    for eng, snap in zip(engines, snaps):
        eng.dyn.copy_from(snap)
    del graphs, snaps
    torch.cuda.synchronize()
    h_in = torch.empty(W + S, R * 10, dtype=torch.int32).pin_memory()
    h_in[:, :R] = torch.as_tensor(counts)
    h_in[:, R:2 * R] = torch.as_tensor(start)
    h_in[:, 2 * R:] = torch.as_tensor(tokens).reshape(W + S, R * 8)
    bufs = [eng.host_buffers(8) for eng in engines]
    for s in range(W):                       # the W warm-up steps through the host path (the first call captures its graph)
        for (inp, res), eng, cs in zip(bufs, engines, cuda_streams):
            inp.copy_(h_in[s])
            with torch.cuda.stream(cs):
                eng.step_host(inp, res, sync=False)
        for cs in cuda_streams:
            cs.synchronize()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for s in range(W, W + S):
        for (inp, res), eng, cs in zip(bufs, engines, cuda_streams):
            inp.copy_(h_in[s])
            with torch.cuda.stream(cs):
                eng.step_host(inp, res, sync=False)
        for cs in cuda_streams:
            cs.synchronize()
    host_s = time.perf_counter() - t0
    return {"workload": f"{n_streams} independent c2 batches ({R} requests each) in flight on {n_streams} streams",
            "queries_per_s": n_streams * R * S / (ms * 1e-3), "us_per_step_per_batch": ms / S * 1e3, "n_streams": n_streams,
            "e2e_queries_per_s": n_streams * R * S / host_s, "e2e_us_per_step": host_s / S * 1e6,
            "e2e_note": "host buffers in and out every step for every batch (step_host, zero-copy), one host thread"}


def bench_c1(a, dev, prompt=4096, steps=256):
    """Config c1 (the reference demo's shape, tests/test_samd_sam_only.py): ONE request, 4k-token prompt, samd_sam_only
    flavour (max_predicts 40, alpha 4).  Latency comparison: a single warp walks the chain, so this is the regime
    where a CPU core is competitive - reported for completeness, next to the Python / C ports on one core."""
    import torch
    from samd_b200 import _cabi as K, engine as E, synth
    sys.path.insert(0, os.path.join(REPO, "oracle"))
    stream = synth.copy_mix(prompt + 8 * steps + 1, VOCAB, 1000).astype(np.int32)
    rng = np.random.default_rng(1001)
    counts = rng.integers(1, 9, size=steps).astype(np.int32)
    ends = prompt + np.cumsum(counts)
    dyn = E.DynSamBatch(1, prompt + 8 * steps + 16, dev)
    eng = E.DraftEngine(dyn, None, K.FLAVOUR_SAM_ONLY, n_predicts=40, len_bias=5, alpha=4.0)
    d_prompt = torch.as_tensor(stream[None, :prompt]).to(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    eng.step(d_prompt, None, None)
    e1.record()
    torch.cuda.synchronize()
    build_ms = e0.elapsed_time(e1)
    toks = [torch.as_tensor(stream[None, ends[i] - counts[i]:ends[i]]).to(dev) for i in range(steps)]
    starts = [torch.as_tensor(stream[ends[i]:ends[i] + 1]).to(dev) for i in range(steps)]
    g = torch.cuda.CUDAGraph()
    snap = E.DynSamBatch(1, dyn.max_tokens, dev)
    snap.copy_from(dyn)
    with torch.cuda.graph(g):
        for i in range(steps):
            eng.step(toks[i], None, starts[i])
    g.replay()
    torch.cuda.synchronize()
    dyn.copy_from(snap)
    torch.cuda.synchronize()
    _gate()
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    gpu_us = e0.elapsed_time(e1) / steps * 1e3
    # one CPU core: Python port and C restatement on the same stream
    import samd_oracle as O
    import c_oracle as CO
    t0 = time.perf_counter()
    po = O.Automaton()
    po.extend(stream[:prompt].tolist())
    py_build = time.perf_counter() - t0
    empty = O.Automaton()
    t0 = time.perf_counter()
    for i in range(steps):
        po.extend(stream[ends[i] - counts[i]:ends[i]].tolist())
        O.select_sam_only(po, empty, None, int(stream[ends[i]]), 40, 4.0, 8, 5)
    py_us = (time.perf_counter() - t0) / steps * 1e6
    co = CO.CSam(len(stream) + 8)
    t0 = time.perf_counter()
    co.extend(stream[:prompt])
    c_build = time.perf_counter() - t0
    # the same loop through the DROP-IN classes (samd_sam_only.DraftModel.update / lookup: one launch each, the lookup's
    # result read back with one device-to-host copy - what a caller of the reference's API sees, syncs included)
    import samd_sam_only as SO
    dm = SO.DraftModel(SO.SamdConfig(max_predicts=40, alpha=4.0, K=8, len_bias=5), device=str(dev))
    dm.reset()
    dm.update(torch.as_tensor(stream[:prompt]).to(dev))
    torch.cuda.synchronize()
    n_warm = 16                               # first calls allocate the pinned I/O buffers and build the argument blocks
    for i in range(n_warm):
        dm.update(toks[i][0])
        dm.lookup(int(stream[ends[i]]))
    t0 = time.perf_counter()
    for i in range(n_warm, steps):
        dm.update(toks[i][0])
        dm.lookup(int(stream[ends[i]]))
    dropin_us = (time.perf_counter() - t0) / (steps - n_warm) * 1e6
    return {"workload": f"c1: one request, {prompt}-token prompt, {steps} steps of 1-8 appended tokens + lookup + draft "
                        f"(samd_sam_only flavour, max_predicts 40, alpha 4)",
            "gpu_build_tokens_per_s": prompt / (build_ms * 1e-3), "gpu_us_per_step": gpu_us,
            "cpu_python_port_build_tokens_per_s": prompt / py_build, "cpu_python_port_us_per_step": py_us,
            "cpu_c_port_build_tokens_per_s": prompt / c_build, "cores": 1,
            "dropin_api_us_per_step": dropin_us, "dropin_api_steps_per_s": 1e6 / dropin_us,
            "dropin_note": "samd_sam_only.DraftModel.update + lookup per step through the reference's class API "
                           "(two launches and one device-to-host read per step)"}


def bench_static(a, dev, n_corpus=2_000_000, n_q=4096, steps=64, warm=8, check=False, l2_mb=None):
    """Config c3: static SAM lookups over a corpus built on the host inside the run, 4096 persistent cursors advanced
    1-8 tokens per step, then lookup + 16-token draft.  `check`: the first 4 steps of all 4096 queries are compared with
    the oracle's C restatement built over the same documents (state index, match length, draft).  `l2_mb`: the same
    measurement again with the first l2_mb MB of the state records pinned in L2 (access-policy window)."""
    import torch
    from samd_b200 import _cabi as K, engine as E, synth
    t0 = time.time()
    docs = synth.make_corpus(n_corpus, VOCAB, 3000, singletons=True)
    st = E.StaticSamDevice.build(docs, synth.EOS, with_counts=False, device=dev)
    build_s = time.time() - t0
    q = synth.corpus_queries(docs, n_q, 8 * (steps + warm) + 1, VOCAB, 3001).astype(np.int32)
    rng = np.random.default_rng(3002)
    counts = rng.integers(1, 9, size=(steps + warm, n_q)).astype(np.int32)
    ends = np.cumsum(counts, axis=0)
    begins = ends - counts
    cols = np.arange(8)[None, None, :]
    rows = np.arange(n_q)[None, :, None]
    tokens = np.where(cols < counts[:, :, None], q[rows, np.minimum(begins[:, :, None] + cols, q.shape[1] - 1)], 0).astype(np.int32)
    start = q[np.arange(n_q)[None, :], ends].astype(np.int32)
    dyn = E.DynSamBatch(n_q, 8 * (steps + warm) * 2 + 64, dev)
    eng = E.DraftEngine(dyn, st, K.FLAVOUR_SAMD, n_predicts=N_PREDICTS, len_bias=0, len_threshold=0)
    d_tok, d_cnt, d_st = (torch.as_tensor(x).to(dev) for x in (tokens, counts, start))
    parity = None
    if check:
        sys.path.insert(0, os.path.join(REPO, "oracle"))
        import c_oracle as CO
        t1 = time.time()
        ref = CO.CSam.build(docs, synth.EOS)
        ref_build_s = time.time() - t1
        cur = np.zeros((n_q, 2), dtype=np.int32)
        n_cmp = n_static = 0
        for s in range(4):
            eng.step(d_tok[s], d_cnt[s], d_st[s])
            torch.cuda.synchronize()
            ref.batch_advance(cur, tokens[s], counts[s])
            r_state, r_len, r_draft = ref.batch_lookup(cur, start[s], N_PREDICTS)
            assert np.array_equal(eng.index_static.cpu().numpy(), r_state), f"c3 parity: static state index differs at step {s}"
            assert np.array_equal(eng.match_static.cpu().numpy(), r_len), f"c3 parity: static match length differs at step {s}"
            assert np.array_equal(eng.static_cursor.cpu().numpy(), cur), f"c3 parity: static cursor differs at step {s}"
            is_static = (eng.out_type == K.DRAFT_STATIC_SEQ).cpu().numpy()
            assert np.array_equal(eng.draft.cpu().numpy()[is_static], r_draft[is_static]), f"c3 parity: draft differs at step {s}"
            n_cmp += n_q
            n_static += int(is_static.sum())
        parity = {"queries_compared": n_cmp, "static_drafts_compared": n_static, "oracle": "oracle/sam_oracle.c built over the same documents",
                  "oracle_build_s": ref_build_s, "identical": True}
        del ref
        eng.reset()
    for s in range(warm):
        eng.step(d_tok[s], d_cnt[s], d_st[s])
    torch.cuda.synchronize()
    snap_cur = eng.static_cursor.clone()
    snap = E.DynSamBatch(n_q, dyn.max_tokens, dev)
    snap.copy_from(dyn)

    def timed():
        dyn.copy_from(snap)
        eng.static_cursor.copy_(snap_cur)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for s in range(warm, warm + steps):
                eng.step(d_tok[s], d_cnt[s], d_st[s])
        g.replay()
        torch.cuda.synchronize()
        dyn.copy_from(snap)
        eng.static_cursor.copy_(snap_cur)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        _gate()
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), int(eng.draft.sum().item())

    ms, checksum = timed()
    src = torch.bincount(eng.out_type, minlength=4).tolist()
    out = {"workload": f"c3: static SAM over {st.n_tokens} tokens ({st.n_states} states, {st.n_edges} edges, "
                       f"{st.nbytes / 1e9:.2f} GB flat) + per-request dynamic SAM, {n_q} cursors, 1-8 tokens/step, draft 16",
           "queries_per_s": n_q * steps / (ms * 1e-3), "us_per_step": ms / steps * 1e3, "host_build_s": build_s,
           "host_build_tokens_per_s": st.n_tokens / build_s, "mean_match_static": float(eng.match_static.float().mean()),
           "draft_source_hist": {"dyn": src[0], "static": src[1], "tree_model": src[2]}}
    if parity is not None:
        out["parity"] = parity
    if l2_mb:
        st.set_l2_window(int(l2_mb) << 20)
        ms_w, checksum_w = timed()
        st.set_l2_window(0)
        out["l2_window"] = {"mb_requested": int(l2_mb), "us_per_step": ms_w / steps * 1e3, "queries_per_s": n_q * steps / (ms_w * 1e-3),
                            "us_per_step_without": ms / steps * 1e3, "results_identical": checksum_w == checksum}
    return out


def bench_tree_drafter(a, dev, n_corpus=5_000_000, n_q=4096, steps=32, warm=4):
    """samd_sam_only's static tree drafter (samd_sam_only/sam/static_sam.py:182-215: best-first search over occurrence
    counts with CPython-heapq order, then the mask / position / retrieve buffers): 4096 cursors over a count-annotated
    static automaton, every query drafts a tree of up to 40 nodes per step.  Trees per second."""
    import torch
    from samd_b200 import _cabi as K, engine as E, synth
    docs = synth.make_corpus(n_corpus, VOCAB, 3100, singletons=True)
    st = E.StaticSamDevice.build(docs, synth.EOS, with_counts=True, device=dev)
    q = synth.corpus_queries(docs, n_q, 8 * (steps + warm) + 1, VOCAB, 3101).astype(np.int32)
    rng = np.random.default_rng(3102)
    counts = rng.integers(1, 9, size=(steps + warm, n_q)).astype(np.int32)
    ends = np.cumsum(counts, axis=0)
    begins = ends - counts
    cols = np.arange(8)[None, None, :]
    rows = np.arange(n_q)[None, :, None]
    tokens = np.where(cols < counts[:, :, None], q[rows, np.minimum(begins[:, :, None] + cols, q.shape[1] - 1)], 0).astype(np.int32)
    start = q[np.arange(n_q)[None, :], ends].astype(np.int32)
    dyn = E.DynSamBatch(n_q, 8 * (steps + warm) * 2 + 64, dev)
    eng = E.DraftEngine(dyn, st, K.FLAVOUR_SAM_ONLY, n_predicts=40, len_bias=-(1 << 20), alpha=4.0)   # the static tree always wins
    d_tok, d_cnt, d_st = (torch.as_tensor(x).to(dev) for x in (tokens, counts, start))

    def step(s):
        eng.step(d_tok[s], d_cnt[s], d_st[s])
        eng.tree_draft(d_st[s], K_top=8)

    for s in range(warm):
        step(s)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i, s in enumerate(range(warm, warm + steps)):
        ev[i][0].record()
        eng.step(d_tok[s], d_cnt[s], d_st[s])
        ev[i][1].record()
        eng.tree_draft(d_st[s], K_top=8)
        ev[i][2].record()
    torch.cuda.synchronize()
    us_step = float(np.median([x.elapsed_time(y) for x, y, _ in ev])) * 1e3
    us_tree = float(np.median([y.elapsed_time(z) for _, y, z in ev])) * 1e3
    n_tree = int((eng.out_type == K.DRAFT_STATIC_TREE).sum().item())
    return {"workload": f"samd_sam_only static tree drafter: {st.n_tokens}-token corpus with counts ({st.n_states} states), {n_q} queries/step, "
                        f"max_predicts 40, alpha 4, K 8",
            "us_per_step_tree_kernel": us_tree, "trees_per_s": n_tree / (us_tree * 1e-6), "trees_per_step": n_tree,
            "mean_tree_nodes": float(eng.tree_n.float().mean()), "us_per_step_lookup_kernel": us_step}


def bench_sharded_static(a, dev, rank, world, tokens_per_shard=2_000_000, n_q=4096, steps=64, warm=8):
    """Config c5's retrieval half at a host-buildable size: the static corpus is split by document over the
    ranks; per step every rank advances ALL query cursors on its shard, computes packed keys, one NCCL
    all-reduce-max (Q x 8 bytes) merges them and the draft is read from the replicated corpus tokens."""
    import torch
    import torch.distributed as dist
    from samd_b200 import dist as D, synth
    docs = synth.make_corpus(tokens_per_shard * world, VOCAB, 5000, singletons=True)       # same corpus on every rank
    t0 = time.time()
    sh = D.ShardedStaticSam(docs, synth.EOS, rank, world, n_q, dev)
    build_s = time.time() - t0
    q = synth.corpus_queries(docs, n_q, 8 * (steps + warm) + 1, VOCAB, 5001).astype(np.int32)
    rng = np.random.default_rng(5002)
    counts = rng.integers(1, 9, size=(steps + warm, n_q)).astype(np.int32)
    ends = np.cumsum(counts, axis=0)
    begins = ends - counts
    cols = np.arange(8)[None, None, :]
    rows = np.arange(n_q)[None, :, None]
    tokens = np.where(cols < counts[:, :, None], q[rows, np.minimum(begins[:, :, None] + cols, q.shape[1] - 1)], 0).astype(np.int32)
    start = q[np.arange(n_q)[None, :], ends].astype(np.int32)
    d_tok, d_cnt, d_st = (torch.as_tensor(x).to(dev) for x in (tokens, counts, start))

    def timed(p2p, graph):
        """warm-up steps, then `steps` timed steps; eager launches or one captured graph (p2p only: NCCL stays eager)"""
        sh.reset()
        out = (torch.empty(n_q, dtype=torch.int32, device=dev), torch.empty(n_q, N_PREDICTS, dtype=torch.int32, device=dev))

        def step(s):
            return sh.lookup_draft(d_st[s], N_PREDICTS, p2p=p2p, out=out if p2p else None, tokens=d_tok[s], counts=d_cnt[s])

        for s in range(warm):
            res = step(s)
        torch.cuda.synchronize()
        dist.barrier()
        g = None
        if graph:
            cur0 = sh.cursor.clone()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for s in range(warm, warm + steps):
                    res = step(s)
            sh.cursor.copy_(cur0)
            torch.cuda.synchronize()
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if g is not None:
            _gate()
        e0.record()
        if g is not None:
            g.replay()
        else:
            for s in range(warm, warm + steps):
                res = step(s)
        e1.record()
        torch.cuda.synchronize()
        dist.barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), res[0].clone(), res[1].clone()

    def oracle_check():
        """The merged result of 4 steps x all queries against ONE automaton over the whole corpus (the oracle's C
        restatement, built on rank 0): match length and draft must be identical - the queries are EOS-free, so no match can
        span a shard boundary (SURVEY 8e).  Both exchange paths are checked, not against each other but against the oracle."""
        ok = {"nccl": True, "p2p": None}
        ref = cur = None
        if rank == 0:
            sys.path.insert(0, os.path.join(REPO, "oracle"))
            import c_oracle as CO
            ref = CO.CSam.build(docs, synth.EOS)
        for path in ("nccl", "p2p"):
            if path == "p2p" and sh._xchg is None:
                continue
            sh.reset()
            cur = np.zeros((n_q, 2), dtype=np.int32)
            good = True
            for s in range(4):
                m, d = sh.lookup_draft(d_st[s], N_PREDICTS, p2p=(path == "p2p"), tokens=d_tok[s], counts=d_cnt[s])
                torch.cuda.synchronize()
                if rank == 0:
                    ref.batch_advance(cur, tokens[s], counts[s])
                    r_state, r_len, r_draft = ref.batch_lookup(cur, start[s], N_PREDICTS)
                    hit = r_len > 0
                    good = good and bool(np.array_equal(m.cpu().numpy(), r_len)) and \
                        bool(np.array_equal(d.cpu().numpy()[hit], r_draft[hit]))
            flag = torch.tensor([1 if good else 0], device=dev, dtype=torch.int32)
            dist.broadcast(flag, 0)
            ok[path] = bool(flag.item())
        return ok

    ms, match, draft = timed(False, False)
    out = {"workload": f"c5 (reduced corpus): static SAM over {sh.n_corpus} tokens split by document over {world} GPUs "
                       f"({sh.sam.n_tokens} tokens on rank 0), {n_q} queries/step advanced 1-8 tokens, packed-u64 "
                       f"max-reduce ({n_q * 8} B) per step, draft {N_PREDICTS} from the replicated corpus",
           "nccl": {"queries_per_s": n_q * steps / (ms * 1e-3), "us_per_step": ms / steps * 1e3, "gpu_launches_per_step": 3,
                    "collectives_per_step": 1, "note": "cursor walk, look-up kernel, NCCL all-reduce-max, draft kernel; eager launches"},
           "host_build_s": build_s, "mean_match": float(match.float().mean())}
    try:                                      # the same step with the reduction done by the look-up kernel over NVLink peer memory
        if not sh.connect_peers():
            raise RuntimeError("peer mapping failed on some rank")
        ms_p, match_p, draft_p = timed(True, False)
        same = bool(torch.equal(match_p, match) and torch.equal(draft_p, draft))
        ms_g, match_g, draft_g = timed(True, True)
        same = same and bool(torch.equal(match_g, match) and torch.equal(draft_g, draft))
        out["p2p"] = {"queries_per_s": n_q * steps / (ms_p * 1e-3), "us_per_step": ms_p / steps * 1e3,
                      "graph_queries_per_s": n_q * steps / (ms_g * 1e-3), "graph_us_per_step": ms_g / steps * 1e3,
                      "gpu_launches_per_step": 2, "collectives_per_step": 0, "identical_to_nccl": same, "peers_ok": sh.peers_ok(),
                      "note": "cursor walk + look-up kernel with remote atomicMax into every rank's buffer, draft kernel waiting on "
                              "peer flags; eager, and all steps captured in one CUDA graph"}
        out["queries_per_s"] = max(out["nccl"]["queries_per_s"], out["p2p"]["queries_per_s"], out["p2p"]["graph_queries_per_s"])
    except Exception as e:
        out["p2p"] = {"error": repr(e)}
        out["queries_per_s"] = out["nccl"]["queries_per_s"]
    try:
        out["matches_oracle"] = oracle_check()
    except Exception as e:
        out["matches_oracle"] = {"error": repr(e)}
    return out


def main():
    a = parse()
    # stdout carries exactly one JSON line: file descriptor 1 is re-pointed at stderr, so whatever a native library
    # prints there (NCCL's version banner, ...) cannot get in front of it, and Python's own stdout keeps the real one
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w", buffering=1)
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
    sys.stdout.flush()


if __name__ == "__main__":
    main()
