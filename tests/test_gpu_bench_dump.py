"""bench.py --dump-outputs on the GPU: the arrays it writes are the CPU oracle's answers for the sampled findings, two runs with
the same inputs write the same arrays, and --steps sets the number of timed steps."""

from __future__ import annotations

import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from oracle import oracle as orc

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]
AGENTS, SEED = 20_700, 2145         # bench.py --workload M2 and its default --seed


def run_bench(out: Path, steps: int):
    proc = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "M2", "--steps", str(steps), "--warmup", "3", "--no-cpu-baseline",
                           "--dump-outputs", str(out)], capture_output=True, text=True, timeout=1800)
    assert proc.returncode == 0, proc.stderr[-3000:]
    return json.loads(proc.stdout), {p.stem: np.load(p) for p in sorted(out.glob("*.npy"))}


def capped(flat, off, cap):
    return np.concatenate([flat[off[i]: off[i] + min(cap, off[i + 1] - off[i])] for i in range(len(off) - 1)])


def test_dumped_outputs_equal_the_oracle_and_steps_set_the_timed_steps(tmp_path):
    import bench
    from agent_bom_b200 import estate

    one, got = run_bench(tmp_path / "one", 1)
    three, again = run_bench(tmp_path / "three", 3)
    assert (one["steps"], three["steps"]) == (1, 3)
    assert three["gpu_launches"] == 3 * one["gpu_launches"] > 0          # library launches inside the timed region
    assert got.keys() == again.keys()
    for name in got:
        np.testing.assert_array_equal(got[name], again[name], err_msg=name)
    assert all(a.dtype == np.float64 for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= bench.DUMP_BYTES

    est = estate.generate(AGENTS, SEED, estate.BENCH_KNOBS, exact_rank=False)
    og = orc.build_csr(est.n_nodes, est.src, est.dst, est.rel, est.flags, est.node_type)
    src = got["sources"].astype(np.int32)
    assert len(src) == bench.DUMP_QUERIES < len(est.findings) and np.isin(src, est.findings).all() and np.all(np.diff(src) > 0)

    want = orc.impact_many(og, src, bench.MAX_DEPTH)
    np.testing.assert_array_equal(got["impact_count"], np.diff(want.off))
    np.testing.assert_array_equal(got["impact_maxd"], want.maxd)
    np.testing.assert_array_equal(got["impact_hist"], want.hist)
    cap = min(1024, bench.DUMP_LIST_VALUES // len(src))
    assert got["impact_count"].max() > cap                                 # the cut is exercised
    np.testing.assert_array_equal(got["impact_nodes"], capped(want.nodes, want.off, cap))

    rows = orc.derived_paths(og, src, est.node_rank)
    owner = np.searchsorted(src, rows.hops[:, 3])                          # rows come finding by finding, in input order
    assert np.all(np.diff(owner) >= 0)
    off = np.concatenate([[0], np.cumsum(np.bincount(owner, minlength=len(src)))])
    np.testing.assert_array_equal(got["paths_count"], np.diff(off))
    np.testing.assert_array_equal(got["paths_hops"], capped(rows.hops, off, bench.DUMP_ROWS))
    np.testing.assert_array_equal(got["paths_rels"], capped(rows.rels, off, bench.DUMP_ROWS))
    np.testing.assert_array_equal(got["paths_ncred"], capped(rows.ncred, off, bench.DUMP_ROWS))
    np.testing.assert_array_equal(got["paths_ntool"], capped(rows.ntool, off, bench.DUMP_ROWS))
