"""Differential check of the CPU oracle against the UNMODIFIED reference engine on random estates.

The other fixtures under tests/golden/ pin the oracle on fixed known-answer graphs and generator estates; this test adds one
random graph per seed (oracle/make_golden.py ``random_estate``) — an estate-shaped core (agents → servers → packages →
vulnerabilities, credentials, tools) plus noise edges of every relationship type, bidirectional and non-traversable edges,
duplicates, self loops and ghost endpoints — with the reference's own `impact_of / bfs / reachable_from / shortest_path /
traverse_subgraph / compute_dependency_reach / _derived_attack_paths` answers on each (``make_golden.py --live-only`` runs the
reference and writes them to ``tests/golden/live/estates.json.xz``), and holds the oracle to the same answers through the checks
of tests/test_oracle_golden.py.  CPU-only."""

from __future__ import annotations

import gzip
import json
import lzma

import pytest

import golden_util

BUNDLE = golden_util.GOLDEN / "live" / "estates.json.xz"


@pytest.fixture(scope="module")
def live(tmp_path_factory):
    """Unpack the bundle into one fixture file per seed, where golden_util.load looks for them."""
    docs = json.loads(lzma.decompress(BUNDLE.read_bytes()))
    out = tmp_path_factory.mktemp("live_golden")
    for doc in docs:
        with gzip.open(out / f"{doc['name']}.json.gz", "wb") as fh:
            fh.write(json.dumps(doc).encode())
    saved = golden_util.GOLDEN
    golden_util.GOLDEN = out
    try:
        yield [doc["name"] for doc in docs]
    finally:
        golden_util.GOLDEN = saved


@pytest.mark.parametrize("check", ["test_adjacency_model", "test_impact_of", "test_bfs_paths_exact_order", "test_reachable_from", "test_shortest_path",
                                   "test_traverse_subgraph", "test_dependency_reach", "test_derived_attack_paths"])
def test_oracle_equals_the_reference_on_fresh_random_estates(live, check):
    import test_oracle_golden as tog

    fn = getattr(tog, check)
    assert len(live) == 16
    for name in live:
        fn(name)
