#!/usr/bin/env python3
"""bench.py — exposure-path traversals/sec on a synthetic estate (BASELINE.json's metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload L|M2|M1|S] [--mode exposure|enumerate] [--impl b200|reference]
                    [--dump-outputs DIR]

One *traversal* = for one finding node f: ``impact_of(f, max_depth=4)`` + f's derived exposure paths (SURVEY.md §8d).
``--mode enumerate`` (BASELINE config 5) adds, per finding, ``bfs(f, max_depth=4, traversable_only=True)`` path
enumeration (order + first-discoverer parents) and ``traverse_subgraph([f], max_depth=4)`` under four relationship masks
({all}, {uses, depends_on, contains, provides_tool}, the lateral set, static-only).

One *step* = one pass of that hot path over every finding of the estate.  The CSR is replicated by a one-time NCCL
broadcast, sources are sharded by depth-1 frontier signature (all members of a frontier group on one rank), there is no
collective on the data path → total work is fixed by the estate: ``"scaling": "strong"``.

Numbers on the JSON line
  value         traversals/s with inputs (finding list, CSR) resident in HBM, CUDA-event timed over K steps, max over ranks.
  e2e           the same through the host API (``DeviceGraph.exposure_many`` → C ABI ``abb_exposure_host``): H2D of the finding
                ids, the signature sharding at N>1, D2H of every result array, all inside the timed region.  ``first_call_ms``
                is the same call before the library has a size hint (cold arenas); ``python_zero_copy`` wraps the pinned
                result blocks as numpy views.  The exposure-path rows cross PCIe in their factorised form (links + templates).
  roofline      frontier-expansion (walk) kernels: ALGORITHMIC bytes of the traversals actually EXECUTED (one per frontier
                group + the individually walked sources; oracle counters 8·N_exp + 6·M_scan + 8·N_disc over every executed
                traversal) ÷ CUDA-event time of the walk launches ÷ measured HBM peak.  ``per_source_equivalent`` applies the
                same formula to every source unshared (it may exceed the peak: shared traversals are not re-executed).
  cpu_baseline  the CPU port (oracle/oracle.c, OpenMP, explicit thread count) on a bounded sample + the unmodified Python
                reference's numbers measured in the build container (profiles/r02_reference_python.json).
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "exposure-path traversals/sec"
UNIT = "traversals/s"
WORKLOADS = {
    # name: (agents, description)
    "L": (215_000, "10M-node/100M-edge synthetic estate"),
    "M2": (20_700, "1M-node/10M-edge synthetic estate"),
    "M1": (2_000, "100K-node/1M-edge synthetic estate"),
    "S": (300, "16K-node/150K-edge synthetic estate (smoke)"),
}
MAX_DEPTH = 4
DYN = (1 << 26) | (1 << 27) | (1 << 28)                       # invoked, accessed, delegated_to (container.py:777)
REACH4 = (1 << 1) | (1 << 2) | (1 << 7) | (1 << 3)            # uses, depends_on, contains, provides_tool (dependency_reach.py:44-51)
LATERAL = (1 << 13) | (1 << 14) | (1 << 15)                   # lateral set (container.py:687-696)
MASKS = (("all", 0, False), ("reach4", REACH4, False), ("lateral", LATERAL, False), ("static_only", 0, True))


_JSON_OUT = None


def claim_stdout() -> None:
    """Keep the process's real stdout for the ONE JSON line: file descriptor 1 is pointed at stderr for everything else
    (NCCL's version banner, library chatter of child threads), the JSON line goes to a duplicate of the original."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict) -> None:
    out = _JSON_OUT or sys.stdout
    print(json.dumps(line), file=out, flush=True)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:  # pragma: no cover
        return os.cpu_count() or 1


def hbm_peak() -> tuple[float, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    FIELDS = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines: list[str] = []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *exc):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self) -> dict:
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ── estate / oracle helpers ─────────────────────────────────────────────────────────────────────────────────────────────
def generate_estate(workload: str, seed: int):
    from agent_bom_b200 import estate

    agents, desc = WORKLOADS[workload]
    t0 = time.perf_counter()
    est = estate.generate(agents, seed, estate.BENCH_KNOBS, exact_rank=False)
    log(f"[bench] estate {workload}: {est.n_nodes:,} nodes / {est.n_edges:,} edges / {len(est.findings):,} findings (generate {time.perf_counter() - t0:.1f}s)")
    return est, desc


def device_csr(est):
    """CSR for upload, built by the product's own counting sort (libabb200.so)."""
    from agent_bom_b200.graph import csr as csrmod

    t0 = time.perf_counter()
    host = csrmod.from_arrays(None, est.node_type, est.src, est.dst, est.rel, est.flags, node_rank=est.node_rank)
    log(f"[bench] CSR build: {host.n_entries:,} adjacency entries per direction ({time.perf_counter() - t0:.1f}s)")
    return host


def oracle_graph_from(host):
    """The oracle walks the host CSR the device gets (the library's builder is parity-tested against the oracle's own in tests/)."""
    from oracle import oracle as orc

    return orc.OracleGraph(n_nodes=host.n_nodes, fwd_off=host.fwd_off, fwd_nbr=host.fwd_nbr, fwd_meta=host.fwd_meta, fwd_eid=host.fwd_eid,
                           rev_off=host.rev_off, rev_nbr=host.rev_nbr, rev_meta=host.rev_meta, rev_eid=host.rev_eid, node_type=host.node_type)


def cpu_traversals(og, findings: np.ndarray, node_rank: np.ndarray, threads: int, mode: str = "exposure"):
    """One CPU pass of the hot path over `findings`; returns (seconds, impact WalkResult)."""
    from oracle import oracle as orc

    t0 = time.perf_counter()
    w = orc.impact_many(og, findings, MAX_DEPTH, threads=threads)
    orc.derived_paths(og, findings, node_rank, threads=threads)
    if mode == "enumerate":
        orc.bfs_many(og, findings, MAX_DEPTH, True, threads=threads)
        ro = np.arange(len(findings) + 1, dtype=np.int64)
        for _name, mask, static in MASKS:
            m = (mask or 0xFFFFFFFF) & (~DYN if static else 0xFFFFFFFF)
            orc.traverse_many(og, findings, ro, direction=1, max_depth=MAX_DEPTH, rel_mask=m, threads=threads)
    return time.perf_counter() - t0, w


def sample_for_budget(og, findings, node_rank, budget_s: float, threads: int, mode: str = "exposure", min_frac: float = 0.0):
    """Largest evenly spaced sample of `findings` whose CPU pass fits ~budget_s (probe first), at least `min_frac` of them."""
    probe = findings[:: max(1, len(findings) // 4000)][:4000]
    dt, _ = cpu_traversals(og, probe, node_rank, threads, mode)
    rate = len(probe) / max(dt, 1e-6)
    n = int(min(len(findings), max(len(probe), rate * budget_s, min_frac * len(findings))))
    stride = max(1, len(findings) // n)
    return np.ascontiguousarray(findings[::stride][:n])


def forecast_weight(host, depth: int = 3) -> np.ndarray:
    """Per node: number of reverse walks of length `depth`+1 starting there = candidates its depth-`depth` frontier would scan.
    Used to put the heaviest sources into the parity gate (the tiers' hand-offs are exercised by exactly those)."""
    roff = host.rev_off.astype(np.int64)
    nbr = host.rev_nbr
    w = np.diff(roff).astype(np.float64)
    for _ in range(depth):
        c = np.concatenate([[0.0], np.cumsum(w[nbr])])
        w = c[roff[1:]] - c[roff[:-1]]
    return w


def reference_python_numbers():
    p = ROOT / "profiles" / "r02_reference_python.json"
    if not p.exists():
        return None
    try:
        doc = json.loads(p.read_text())
        return {"source": "profiles/r02_reference_python.json (unmodified Python reference, build container, oracle/time_reference_python.py)",
                "host_cpu_count": doc["host"]["cpu_count"],
                "impact_of": [{"agents": e["agents"], "nodes": e["nodes"], "edges": e["edges"], "findings_per_s_single_process": e["impact_of"]["findings_per_s_single_process"],
                               "findings_per_s_fork_pool": e["impact_of"]["fork_pool"]["findings_per_s"], "processes": e["impact_of"]["fork_pool"]["processes"]} for e in doc["impact"]],
                "traversals_incl_derived_paths": [{"agents": e["agents"], "edges": e["edges"], "traversals_per_s_single_process": e["traversals_per_s_single_process"]} for e in doc["derived_paths"]]}
    except Exception:
        return None


# ── --impl reference ────────────────────────────────────────────────────────────────────────────────────────────────────
def run_reference(args) -> int:
    """The reference algorithm's CPU port on the host cores (rank 0 only; the Python reference cannot travel to this box).
    Needs nothing of the product library: the CSR comes from the oracle's own numpy restatement of add_edge."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle as orc

    threads = host_threads()            # explicit: torchrun exports OMP_NUM_THREADS=1 to its children
    est, desc = generate_estate(args.workload, args.seed)
    t0 = time.perf_counter()
    og = orc.build_csr(est.n_nodes, est.src, est.dst, est.rel, est.flags, est.node_type)
    log(f"[bench] oracle CSR build {time.perf_counter() - t0:.1f}s; {threads} OpenMP threads")
    # every pass is a bounded sample: the whole --steps K --warmup W run stays within a few minutes (≈150 s of timed CPU work in total)
    per_pass = max(2.0, min(args.cpu_budget, 150.0 / (args.steps + args.warmup)))
    sample = sample_for_budget(og, est.findings, est.node_rank, per_pass, threads, args.mode, min_frac=0.10 if args.workload != "L" else 0.0)
    times = []
    for i in range(args.warmup + args.steps):
        dt, _w = cpu_traversals(og, sample, est.node_rank, threads, args.mode)
        if i >= args.warmup:
            times.append(dt)
    total = sum(times)
    value = len(sample) * len(times) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * total / len(times), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": f"{desc}, all finding nodes as sources", "mode": args.mode, "estate": est.summary() | {"edges_by_relationship": None}, "max_depth": MAX_DEPTH},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{len(sample):,} of {len(est.findings):,} findings (every {max(1, len(est.findings) // len(sample))}th = {100.0 * len(sample) / len(est.findings):.1f} %), "
                                   f"{total / len(times):.1f}s per pass, oracle/oracle.c with {threads} OpenMP threads",
                         "reference_python": reference_python_numbers()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


# ── parity gate ─────────────────────────────────────────────────────────────────────────────────────────────────────────
def parity_gate(dg, og, est, host, my_host, args, mode: str) -> str:
    """An invalid run must not print a number: `--check` evenly spaced findings + the `--check-heavy` heaviest of this rank
    (by forecast degree) go through the host API and are compared with the oracle, bit for bit."""
    from oracle import oracle as orc

    nq = len(my_host)
    k = min(args.check, nq)
    sel = my_host[:: max(1, nq // k)][:k]
    if args.check_heavy > 0:
        w = forecast_weight(host)[my_host]
        heavy = my_host[np.argsort(-w, kind="stable")[: min(args.check_heavy, nq)]]
        sel = np.unique(np.concatenate([sel, heavy])).astype(np.int32)
    got_w, got_p = dg.exposure_many(sel, MAX_DEPTH)
    want_w = orc.impact_many(og, sel, MAX_DEPTH, threads=host_threads())
    want_p = orc.derived_paths(og, sel, est.node_rank, threads=host_threads())
    ok = np.array_equal(got_w.count, np.diff(want_w.off).astype(np.int32)) and np.array_equal(got_w.hist, want_w.hist) and np.array_equal(got_w.maxd, want_w.maxd)
    for q in range(len(sel)):
        if not ok:
            break
        a, b = int(want_w.off[q]), int(want_w.off[q + 1])
        ok = np.array_equal(got_w.slice(q), want_w.nodes[a:b])
    ok = ok and np.array_equal(got_p.hops, want_p.hops) and np.array_equal(got_p.rels, want_p.rels) and np.array_equal(got_p.ncred, want_p.ncred)
    what = "impact_of + exposure-path rows"
    if ok and mode == "enumerate":
        gb = dg.bfs_many(sel, MAX_DEPTH, True)
        wb = orc.bfs_many(og, sel, MAX_DEPTH, True, threads=host_threads())
        ok = np.array_equal(gb.count, np.diff(wb.off).astype(np.int32))
        for q in range(len(sel)):
            if not ok:
                break
            a, b = int(wb.off[q]), int(wb.off[q + 1])
            ok = np.array_equal(gb.slice(q), wb.nodes[a:b]) and np.array_equal(gb.aux(q, "parent") - 1, wb.aux[a:b])
        ro = np.arange(len(sel) + 1, dtype=np.int64)
        for _name, mask, static in MASKS:
            if not ok:
                break
            m = (mask or 0xFFFFFFFF) & (~DYN if static else 0xFFFFFFFF)
            wt = orc.traverse_many(og, sel, ro, direction=1, max_depth=MAX_DEPTH, rel_mask=m, threads=host_threads())
            gt = dg.walk(dg.spec_traverse(1, MAX_DEPTH, -1, -1, False, mask, static, False, True), sel, ro)
            ok = np.array_equal(gt.count, np.diff(wt.off).astype(np.int32)) and np.array_equal(gt.ecount, np.diff(wt.eoff))
            for q in range(len(sel)):
                if not ok:
                    break
                a, b = int(wt.off[q]), int(wt.off[q + 1])
                ea, eb = int(wt.eoff[q]), int(wt.eoff[q + 1])
                ok = np.array_equal(gt.slice(q), wt.nodes[a:b]) and np.array_equal(gt.aux(q, "depth"), wt.aux[a:b]) and np.array_equal(gt.edge_slice(q), wt.edges[ea:eb])
        what += " + bfs order/parents + 4 masked traverse_subgraph (nodes, depths, recorded edges)"
    if not ok:
        raise SystemExit("[bench] PARITY FAILURE against the CPU oracle — refusing to report a number")
    msg = f"{len(sel):,} findings ({k:,} evenly spaced + the {args.check_heavy} heaviest by forecast degree) bit-identical to the oracle: {what}"
    log(f"[bench] parity gate: {msg}")
    return msg


# ── --dump-outputs ──────────────────────────────────────────────────────────────────────────────────────────────────────
# The results of one step at L run to gigabytes, so a seeded sample of the findings is written: for each sampled finding its
# complete per-query answers and the first entries of its node / edge lists and exposure-path rows (all layout-independent:
# arena offsets are not written).  Everything is float64, which holds every int32 id exactly.
DUMP_BYTES = 64 << 20             # all files together
DUMP_QUERIES = 2048               # sampled findings
DUMP_ROWS = 64                    # exposure-path rows kept per sampled finding
DUMP_LIST_VALUES = 6 << 20        # list entries kept over all sampled findings and all walks of the step


def _capped_index(start, count, cap: int):
    """Positions start[i] .. start[i] + min(count[i], cap) - 1, concatenated over i."""
    import torch

    pos = torch.arange(cap, device=start.device)
    keep = pos[None, :] < count[:, None]
    return (start[:, None] + pos[None, :])[keep]


def dump_outputs(out_dir: Path, roots, sel, walks, paths) -> None:
    """Write what the device buffers of `walks` ((name, DeviceWalk) pairs) and `paths` (DevicePaths) hold for the queries `sel`
    of the batch `roots` as `out_dir/<name>.npy`."""
    import torch

    from agent_bom_b200.graph.schema import N_ENTITY_TYPES

    dev = roots.device
    q = torch.from_numpy(sel).to(dev)
    n_lists = sum(1 + (w.parent is not None) + (w.depth is not None) + (w.edges is not None) for _, w in walks)
    cap = min(1024, DUMP_LIST_VALUES // (len(sel) * n_lists))
    out = {"sources": roots[q]}
    for name, w in walks:
        p = name.replace("[", "_").rstrip("]")
        count = w.q_count[q].long()
        out[f"{p}_count"], out[f"{p}_maxd"], out[f"{p}_flags"] = count, w.q_maxd[q], w.q_flags[q]
        if w.q_hist is not None:
            out[f"{p}_hist"] = w.q_hist.view(-1, N_ENTITY_TYPES)[q]
        ix = _capped_index(w.q_start[q], count, cap)
        for field in ("nodes", "parent", "depth"):
            if getattr(w, field) is not None:
                out[f"{p}_{field}"] = getattr(w, field)[ix]
        if w.edges is not None:
            out[f"{p}_ecount"] = w.q_ecount[q]
            out[f"{p}_edges"] = w.edges[_capped_index(w.q_estart[q], w.q_ecount[q], cap)]
    first = paths.f_off[q]
    rows = paths.f_off[q + 1] - first
    ix = _capped_index(first, rows, DUMP_ROWS)
    out["paths_count"], out["paths_hops"], out["paths_rels"] = rows, paths.hops.view(-1, 4)[ix], paths.rels.view(-1, 4)[ix, :3]
    out["paths_ncred"], out["paths_ntool"] = paths.ncred[ix], paths.ntool[ix]
    arrays = {k: v.cpu().numpy().astype(np.float64) for k, v in out.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise SystemExit(f"[bench] --dump-outputs: {total:,} bytes exceed the {DUMP_BYTES:,}-byte bound")
    out_dir.mkdir(parents=True, exist_ok=True)
    for k, a in arrays.items():
        np.save(out_dir / f"{k}.npy", a)
    log(f"[bench] outputs of the last timed step: {len(sel):,} of {roots.shape[0]:,} findings, lists cut at {cap} entries and "
        f"{DUMP_ROWS} path rows, {len(arrays)} arrays ({total / 1e6:.1f} MB) -> {out_dir}")


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="L", choices=sorted(WORKLOADS))
    ap.add_argument("--mode", default="exposure", choices=["exposure", "enumerate"])
    ap.add_argument("--seed", type=int, default=2145)
    ap.add_argument("--batch", type=int, default=1 << 22, help="findings per launch batch (one batch de-duplicates shared frontiers best)")
    ap.add_argument("--cpu-budget", type=float, default=20.0, help="seconds of CPU work per CPU-baseline pass")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--check", type=int, default=2000, help="evenly spaced findings checked against the oracle before timing")
    ap.add_argument("--check-heavy", type=int, default=200, help="heaviest findings (by forecast degree) added to the parity gate")
    ap.add_argument("--no-overlap", dest="overlap", action="store_false", help="run the exposure-path pipeline after the walk instead of next to it (second stream)")
    ap.add_argument("--dump-outputs", type=Path, metavar="DIR",
                    help=f"after the timed steps write what the last one computed for a seeded sample of {DUMP_QUERIES} findings as DIR/<name>.npy "
                         "(float64; rank 0's shard with several GPUs; the step must be one batch)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    if args.warmup < 3:
        args.warmup = 3
    claim_stdout()
    if args.impl == "reference":
        return run_reference(args)

    import torch

    from agent_bom_b200 import _lib, dist as abdist
    from agent_bom_b200.engine import DeviceGraph
    from agent_bom_b200.torch_api import DevicePaths, DeviceWalk, frontier_signatures, shard_by_signature

    # keep stdout to the single JSON line: NCCL's version banner / debug output goes to a file
    os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/abb200_nccl.%h.%p.log")
    info = abdist.init_from_env("nccl" if int(os.environ.get("WORLD_SIZE", "1")) > 1 else None)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback (use --impl reference for the CPU port)")
    torch.cuda.set_device(info.local_rank)
    device = torch.device("cuda", info.local_rank)
    lib = _lib.load()
    mode = args.mode

    # ---- load path (untimed by the metric, reported): rank 0 generates + builds the CSR, one packed NCCL broadcast replicates it
    est = host = None
    desc = WORKLOADS[args.workload][1]
    if info.rank == 0:
        est, desc = generate_estate(args.workload, args.seed)
        host = device_csr(est)
    abdist.warm_up(info, device)
    t0 = time.perf_counter()
    tensors, n_nodes, n_entries, bstats = abdist.broadcast_csr(host, info, device, return_stats=True)
    findings_all = abdist.broadcast_array(est.findings if info.rank == 0 else None, info, device)
    torch.cuda.synchronize()
    t_bcast = time.perf_counter() - t0
    dg = DeviceGraph.adopt(tensors, n_nodes, n_entries, info.local_rank)
    spec = DeviceGraph.spec_impact_of(MAX_DEPTH)

    def shard_of(all_findings):
        """This rank's findings: every finding of one depth-1 frontier group lands on the same rank, so each shared traversal runs
        once in the whole job (a positional split would repeat the heavy groups on every rank)."""
        if info.world == 1:
            return all_findings
        sig = frontier_signatures(dg, spec, all_findings)
        return all_findings[shard_by_signature(sig, info.world, info.rank)].contiguous()

    my = shard_of(findings_all)
    my_host = my.cpu().numpy()
    nq = int(my.shape[0])
    batch = max(1, min(args.batch, nq))
    batches = [(s, min(s + batch, nq)) for s in range(0, nq, batch)]
    if args.dump_outputs and len(batches) > 1:
        raise SystemExit(f"[bench] --dump-outputs needs the step in one batch: --batch {batch:,} < {nq:,} findings (the buffers keep only the last batch)")
    log(f"[bench] rank {info.rank}/{info.world}: {nq:,} findings in {len(batches)} batches of <= {batch:,}; CSR replicate {t_bcast:.3f}s ({dg.nbytes / 1e9:.2f} GB, {bstats})")

    # ---- cold first call through the host API (no size hint yet): arenas are sized on the fly, the walk may run twice
    t0 = time.perf_counter()
    dg.exposure_many(my_host[batches[0][0]: batches[0][1]], MAX_DEPTH, collect=False)
    first_call_ms = 1000.0 * (time.perf_counter() - t0)

    # ---- device-resident leg: buffers sized by a first fitted pass
    walk = DeviceWalk(dg, spec, batch, node_cap=1 << 20)
    paths = DevicePaths(dg, batch)
    extra = []          # (name, DeviceWalk) of the enumerate mode
    if mode == "enumerate":
        extra.append(("bfs", DeviceWalk(dg, DeviceGraph.spec_bfs(MAX_DEPTH, True), batch, node_cap=1 << 20)))
        for name, mask, static in MASKS:
            extra.append((f"traverse[{name}]", DeviceWalk(dg, DeviceGraph.spec_traverse(1, MAX_DEPTH, -1, -1, False, mask, static, False, True), batch,
                                                         node_cap=1 << 20, edge_cap=1 << 20)))
    need_nodes = need_rows = tot_nodes = tot_rows = 0
    extra_tot = {name: [0, 0] for name, _ in extra}
    for s, e in batches:
        n_need, _ = walk.launch_fitted(my[s:e])
        rows = paths.run_fitted(my[s:e])
        need_nodes, need_rows = max(need_nodes, n_need), max(need_rows, rows)
        tot_nodes += n_need; tot_rows += rows
        for name, w in extra:
            nn, ne = w.launch_fitted(my[s:e])
            extra_tot[name][0] += nn; extra_tot[name][1] += ne
    walk.reserve(need_nodes); paths.reserve(need_rows)
    torch.cuda.synchronize()

    # ---- parity gate against the oracle (rank 0)
    og = None
    parity = None
    if info.rank == 0 and (args.check > 0 or not args.no_cpu_baseline):
        from oracle import oracle as orc

        og = oracle_graph_from(host)
    if info.rank == 0 and args.check > 0:
        parity = parity_gate(dg, og, est, host, my_host, args, mode)

    main_stream = torch.cuda.current_stream()
    side_stream = torch.cuda.Stream(device=device) if args.overlap else None

    def one_step(timers=None, overlap=False):
        """One pass of the hot path.  `overlap`: the exposure-path pipeline (independent of the walk's results) runs on a second
        stream next to the walk and fills the SMs the walk's tail leaves idle; the step ends when both have finished."""
        for s, e in batches:
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(3 + len(extra))] if timers is not None else None
            if evs: evs[0].record()
            if overlap:
                side_stream.wait_stream(main_stream)
                walk.launch(my[s:e])
                paths.count(my[s:e], stream=side_stream)
                paths.fill(my[s:e], stream=side_stream)
                main_stream.wait_stream(side_stream)
                if evs: evs[1].record(); evs[2].record()
            else:
                walk.launch(my[s:e])
                if evs: evs[1].record()
                paths.count(my[s:e])
                paths.fill(my[s:e])
                if evs: evs[2].record()
            for i, (_name, w) in enumerate(extra):
                w.launch(my[s:e])
                if evs: evs[3 + i].record()
            if evs: timers.append(evs)

    clocks = ClockSampler(info.local_rank)
    clocks.__enter__()                       # sampled from the warm-up through the end of the e2e leg (all under load)
    for _ in range(args.warmup):
        one_step()
    torch.cuda.synchronize()
    abdist.barrier(info)
    # kernel-time breakdown (walk / paths / extra walks) from a sequential pass: this is what the roofline uses
    timers: list = []
    for _ in range(args.steps):
        one_step(timers)
    torch.cuda.synchronize()
    walk_ms = sum(ev[0].elapsed_time(ev[1]) for ev in timers) / args.steps
    paths_ms = sum(ev[1].elapsed_time(ev[2]) for ev in timers) / args.steps
    seq_ms = sum(ev[0].elapsed_time(ev[-1]) for ev in timers) / args.steps
    if args.overlap:
        for _ in range(args.warmup):
            one_step(overlap=True)
        torch.cuda.synchronize()
    abdist.barrier(info)
    launches0 = lib.abb_launch_count()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(args.steps):
        one_step(overlap=args.overlap)
    end.record()
    torch.cuda.synchronize()
    if args.dump_outputs and info.rank == 0:
        sel = np.sort(np.random.default_rng(args.seed).choice(nq, size=min(DUMP_QUERIES, nq), replace=False))
        dump_outputs(args.dump_outputs, my, sel, [("impact", walk), *extra], paths)
    abdist.barrier(info)
    launches = lib.abb_launch_count() - launches0
    dev_ms = start.elapsed_time(end)
    extra_ms = {name: sum(ev[2 + i].elapsed_time(ev[3 + i]) for ev in timers) / args.steps for i, (name, _w) in enumerate(extra)}
    # the walk the statistics below describe is the impact walk
    walk.launch(my[batches[-1][0]: batches[-1][1]])
    torch.cuda.synchronize()
    walk_stats = dg.last_walk_stats()
    tier_counts = dg.last_walk_tier_counts()
    dev_ms_max = abdist.max_over_ranks(dev_ms, info, device)
    total_findings = int(findings_all.shape[0])
    value = total_findings * args.steps / (dev_ms_max / 1000.0)
    per_rank = abdist.gather_floats([walk_ms, paths_ms, dev_ms / args.steps, float(nq)], info, device)

    # ---- end-to-end leg: host finding ids in, every result array out, through the C-ABI host call
    all_host = findings_all.cpu().numpy()

    def e2e_step():
        h2d = d2h = 0
        if info.world > 1:                   # the shard selection is part of the call a user makes: H2D of all ids, signatures, mask, D2H of this rank's ids
            mine = shard_of(torch.from_numpy(all_host).to(device)).cpu().numpy()
            h2d += all_host.nbytes; d2h += mine.nbytes
        else:
            mine = my_host
        for s, e in batches:
            w, p = dg.exposure_many(mine[s:e], MAX_DEPTH, collect=False)
            h2d += w[1] + p[1]; d2h += w[2] + p[2]
            if mode == "enumerate":
                for _name, wk in extra:
                    r = dg.walk(wk.spec, mine[s:e], zero_copy=True)
                    h2d += r.h2d_bytes; d2h += r.d2h_bytes
                    del r
        return h2d, d2h

    for _ in range(args.warmup):
        e2e_step()
    torch.cuda.synchronize()
    abdist.barrier(info)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        h2d, d2h = e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    abdist.barrier(info)
    # the same through numpy views of the pinned result blocks (what UnifiedGraph.impact_of_many / exposure callers hold)
    t0 = time.perf_counter()
    touched = 0
    for _ in range(args.steps):
        for s, e in batches:
            w, p = dg.exposure_many(my_host[s:e], MAX_DEPTH, zero_copy=True)
            touched += int(w.count[:16].sum()) + int(p.off[-1])    # touch the views
            del w, p
    e2e_py_s = time.perf_counter() - t0
    abdist.barrier(info)
    clocks.__exit__(None, None, None)
    e2e_s_max = abdist.max_over_ranks(e2e_s, info, device)
    e2e_py_max = abdist.max_over_ranks(e2e_py_s, info, device)
    first_call_max = abdist.max_over_ranks(first_call_ms, info, device)
    e2e_value = total_findings * args.steps / e2e_s_max
    h2d_all = abdist.sum_over_ranks(h2d, info, device)
    d2h_all = abdist.sum_over_ranks(d2h, info, device)

    # ---- roofline of the frontier-expansion (impact walk) launches + CPU baseline, rank 0
    roofline = cpu_baseline = None
    peak, peak_src = hbm_peak()
    threads = host_threads()
    if info.rank == 0:
        if og is not None and not args.no_cpu_baseline:
            # executed traversals of this rank: one representative per frontier group (exact: every one is walked by the oracle)
            sig_np = frontier_signatures(dg, spec, my).cpu().numpy()
            _, first_idx = np.unique(sig_np, return_index=True)
            leaders = np.sort(my_host[first_idx])
            n_exp = m_scan = n_disc = 0
            t0 = time.perf_counter()
            for a in range(0, len(leaders), 250_000):
                lw = orc.impact_many(og, leaders[a: a + 250_000], MAX_DEPTH, threads=threads)
                n_exp += lw.n_exp; m_scan += lw.m_scan; n_disc += lw.n_disc
                del lw
            exec_bytes = 8 * n_exp + 6 * m_scan + 8 * n_disc
            log(f"[bench] executed-traversal byte count: {len(leaders):,} traversals, {exec_bytes / 1e9:.2f} GB algorithmic ({time.perf_counter() - t0:.1f}s of oracle)")
            # CPU baseline proper (N=1 only) and the per-source (unshared) byte figure from the same sample
            budget = args.cpu_budget if info.world == 1 else min(args.cpu_budget, 3.0)
            sample = sample_for_budget(og, my_host, est.node_rank, budget, threads, mode, min_frac=0.10 if args.workload != "L" else 0.0)
            dt, w = cpu_traversals(og, sample, est.node_rank, threads, mode)
            bytes_per_source = w.algorithmic_bytes / len(sample)
            if info.world == 1:
                cpu_baseline = {"value": len(sample) / dt, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": f"{len(sample):,} of {nq:,} findings (evenly spaced, {100.0 * len(sample) / nq:.1f} %), oracle/oracle.c with {threads} OpenMP threads, {dt:.1f}s",
                                "reference_python": reference_python_numbers()}
            achieved = exec_bytes / (walk_ms / 1000.0) / 1e9
            traffic = traffic_note = None
            tfile = ROOT / "profiles" / "ncu_traffic.json"          # DRAM bytes of the walk kernels from an `ncu --set full` capture (commit recorded in the file)
            if tfile.exists() and args.workload == "L" and info.world == 1 and mode == "exposure":
                try:
                    tdoc = json.loads(tfile.read_text())
                    traffic = float(tdoc["walk_dram_bytes_per_launch"])
                    traffic_note = f"ncu --set full capture at commit {tdoc.get('commit', '?')} ({tdoc.get('captured', '?')})"
                except Exception:
                    traffic = None
            roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_note,
                        "kernel": "frontier-expansion kernels of abb_walk_launch (walk_smem_kernel S1, walk_block_kernel mid/big, walk_global_kernel G1/GX) + de-duplication passes",
                        "algorithmic_bytes_per_launch": exec_bytes, "executed_traversals": int(len(leaders)),
                        "algorithmic_bytes_per_executed_traversal": exec_bytes / max(1, len(leaders)),
                        "bytes_counted_by": "oracle counters (8*N_exp + 6*M_scan + 8*N_disc) over every executed traversal, exact",
                        "walk_ms_per_step": walk_ms, "peak_source": peak_src,
                        "per_source_equivalent": {"achieved": bytes_per_source * nq / (walk_ms / 1000.0) / 1e9, "frac": bytes_per_source * nq / (walk_ms / 1000.0) / 1e9 / peak,
                                                  "algorithmic_bytes_per_source": bytes_per_source, "estimated_from": f"{len(sample):,} sampled findings",
                                                  "note": "every source counted unshared (SURVEY 8d); exceeds the peak because sources with an identical depth-1 frontier share one traversal"},
                        "sharing": {"sources": nq, "frontier_groups": walk_stats["groups"], "individual": walk_stats["individual"],
                                    "result_nodes_stored": tot_nodes,
                                    "result_nodes_referenced": int(walk.q_count[:nq].sum(dtype=torch.int64).item()) if len(batches) == 1 else None},
                        }
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": info.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {
                "workload": f"{desc}, all finding nodes as sources, sharded across {info.world} GPU(s) by frontier signature", "mode": mode,
                "nodes": n_nodes, "adjacency_entries_per_direction": n_entries, "findings": total_findings, "max_depth": MAX_DEPTH, "batch": batch, "seed": args.seed,
                "estate_knobs": "creds_per_server=20, cred_bucket=80, vulns_per_server=8 (agent_bom_b200.estate.BENCH_KNOBS)",
                "l2": "inputs larger than L2 (CSR >> 126 MB; no flush)" if dg.nbytes > 400e6 else "CSR smaller than L2; no flush (reported as is)",
                "reached_nodes_per_step_rank0": tot_nodes, "path_rows_per_step_rank0": tot_rows,
                "csr_replicate_s": t_bcast, "csr_broadcast": bstats,
            },
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d_all), "d2h_bytes_per_step": int(d2h_all), "ms_per_step": 1000.0 * e2e_s_max / args.steps,
                    "first_call_ms": first_call_max, "python_zero_copy": {"value": total_findings * args.steps / e2e_py_max, "ms_per_step": 1000.0 * e2e_py_max / args.steps},
                    "includes": "H2D of finding ids, frontier-signature sharding (N>1), walk (in 8 signature-partitioned pieces above 2 M sources, each piece's arena DMA-copied behind the next piece's walk) + path kernels, D2H of per-source slices/packed histograms and of the factorised exposure-path rows "
                                "(links + templates; the flat rows are expanded on the host on first access and are not part of this figure)"},
            "gpu_launches": int(launches),
            "walk_ms_per_step": walk_ms, "paths_ms_per_step": paths_ms, "sequential_ms_per_step": seq_ms,
            "streams": "walk on the main stream, exposure-path pipeline on a second stream (independent inputs), joined at the end of every step" if args.overlap else "one stream",
            "per_rank": {"walk_ms": [r[0] for r in per_rank], "paths_ms": [r[1] for r in per_rank], "step_ms": [r[2] for r in per_rank], "sources": [int(r[3]) for r in per_rank]},
            "tier_handoffs": tier_counts,
            "parity": parity,
            "clocks": clocks.summary(),
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
        }
        if mode == "enumerate":
            line["enumerate"] = {"per_walk_ms": extra_ms, "emitted_per_step_rank0": {k: {"nodes": v[0], "edges": v[1]} for k, v in extra_tot.items()},
                                 "unit_of_work": "impact_of + exposure paths + bfs(depth 4, traversable_only) + traverse_subgraph(depth 4) x {all, reach4, lateral, static_only} per finding"}
        emit(line)
    abdist.barrier(info)
    if info.world > 1:
        import torch.distributed as tdist

        tdist.destroy_process_group()
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
