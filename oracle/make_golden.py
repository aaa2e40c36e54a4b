#!/usr/bin/env python3
"""Generate tests/golden/*.json.gz by running the UNMODIFIED reference engine.

Runs only in the build container (imports ``/root/reference/src``; the GPU box
has no reference tree).  The emitted fixtures pin the CPU oracle
(tests/test_oracle_golden.py) and, through it and directly, the CUDA engine.

    python oracle/make_golden.py            # writes every fixture

Each fixture holds one graph (dense indices: node order = ``graph.nodes``
insertion order, ghosts — edge endpoints without a node record — appended in
first-seen order; edge order = ``graph.edges``) and the reference's answers
for a battery of queries, all in index space.

Known-answer graphs are rebuilt from the reference's own tests:
  tests/test_graph_schema.py:328-386 (+ assertions :408-441, :895-946)
  tests/test_dependency_reach.py:26-161
  tests/test_graph_wave1.py:135-169 (impact_of / sources_of)
  tests/test_graph_api.py:1585-1633 (derived path hops + edges)
plus probes from SURVEY.md §8(a') and estates from the reference's generator
(scripts/generate_graph_benchmark_estate.py) through the reference builder.
"""

from __future__ import annotations

import gzip
import importlib.util
import json
import lzma
import random
import sys
from pathlib import Path

REF = Path("/root/reference")
sys.path.insert(0, str(REF / "src"))
ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from agent_bom.api.routes.graph import _derived_attack_paths  # noqa: E402
from agent_bom.graph import (  # noqa: E402
    EntityType,
    RelationshipType,
    UnifiedEdge,
    UnifiedGraph,
    UnifiedNode,
    build_unified_graph_from_report,
    compute_dependency_reach,
)

from agent_bom_b200.graph.schema import ENTITY_CODE, REL_CODE, REL_CODE_OTHER, enum_value  # noqa: E402

OUT = ROOT / "tests" / "golden"

AG, SRV, PKG, TOOL, VULN, CRED, MIS, PROV, USER = (
    EntityType.AGENT, EntityType.SERVER, EntityType.PACKAGE, EntityType.TOOL, EntityType.VULNERABILITY,
    EntityType.CREDENTIAL, EntityType.MISCONFIGURATION, EntityType.PROVIDER, EntityType.USER,
)
R = RelationshipType


def mk(nodes, edges) -> UnifiedGraph:
    """nodes: (id, type[, severity, risk_score[, label]]); edges: (src, dst, rel[, direction[, traversable]])."""
    g = UnifiedGraph(scan_id="golden")
    for n in nodes:
        nid, et = n[0], n[1]
        sev = n[2] if len(n) > 2 else ""
        risk = n[3] if len(n) > 3 else 0.0
        label = n[4] if len(n) > 4 else nid
        g.add_node(UnifiedNode(id=nid, entity_type=et, label=label, severity=sev, risk_score=risk))
    for e in edges:
        g.add_edge(UnifiedEdge(source=e[0], target=e[1], relationship=e[2], direction=e[3] if len(e) > 3 else "directed",
                               traversable=e[4] if len(e) > 4 else True))
    return g


# ── known-answer graphs ─────────────────────────────────────────────────────

def kat_schema():  # tests/test_graph_schema.py:328-386
    return mk(
        [("agent:a", AG, "", 0, "agent-a"), ("agent:b", AG, "", 0, "agent-b"), ("server:a:fs", SRV, "", 0, "mcp-fs"),
         ("server:b:fs", SRV, "", 0, "mcp-fs"), ("vuln:CVE-2024-1", VULN, "critical", 9.0, "CVE-2024-1"), ("cred:API_KEY", CRED, "", 0, "API_KEY")],
        [("agent:a", "server:a:fs", R.USES), ("agent:b", "server:b:fs", R.USES), ("server:a:fs", "vuln:CVE-2024-1", R.VULNERABLE_TO),
         ("server:a:fs", "cred:API_KEY", R.EXPOSES_CRED), ("agent:a", "agent:b", R.SHARES_SERVER, "bidirectional")],
    )


def kat_directed():  # tests/test_graph_schema.py:926-946
    return mk([("a", AG), ("s", SRV), ("v", VULN)], [("a", "s", R.USES), ("s", "v", R.VULNERABLE_TO)])


def kat_chain():  # tests/test_dependency_reach.py:26-83 (chain + second agent)
    return mk(
        [("agent:cursor", AG), ("server:mcp-fs", SRV), ("pkg:direct@1.0", PKG), ("pkg:transitive@2.0", PKG), ("vuln:CVE-2026-0001", VULN),
         ("agent:claude", AG), ("server:other", SRV), ("vuln:CVE-2026-0002", VULN)],
        [("agent:cursor", "server:mcp-fs", R.USES), ("server:mcp-fs", "pkg:direct@1.0", R.DEPENDS_ON), ("pkg:direct@1.0", "pkg:transitive@2.0", R.DEPENDS_ON),
         ("pkg:transitive@2.0", "vuln:CVE-2026-0001", R.VULNERABLE_TO), ("agent:claude", "server:other", R.USES),
         ("server:other", "pkg:transitive@2.0", R.DEPENDS_ON), ("pkg:direct@1.0", "vuln:CVE-2026-0002", R.VULNERABLE_TO)],
    )


def kat_reach_misc():  # tests/test_dependency_reach.py:86-161 (island, affects, dangling, lateral) in one graph
    return mk(
        [("agent:cursor", AG), ("pkg:orphan@1", PKG), ("vuln:CVE-2026-9999", VULN), ("server:mcp", SRV), ("pkg:p", PKG), ("vuln:CVE-2026-1234", VULN),
         ("vuln:CVE-2026-0042", VULN), ("agent:a", AG), ("agent:b", AG), ("pkg:lateral@1", PKG)],
        [("pkg:orphan@1", "vuln:CVE-2026-9999", R.VULNERABLE_TO), ("agent:cursor", "server:mcp", R.USES), ("server:mcp", "pkg:p", R.DEPENDS_ON),
         ("vuln:CVE-2026-1234", "pkg:p", R.AFFECTS), ("agent:a", "agent:b", R.SHARES_SERVER), ("agent:b", "pkg:lateral@1", R.SHARES_SERVER)],
    )


def kat_derived():  # tests/test_graph_api.py:1585-1633 shape: agent -> server -> package -> vuln (+ creds/tools, server-level vuln, orphan)
    return mk(
        [("agent:a", AG), ("server:a:fs", SRV), ("pkg:npm:form-data", PKG), ("vuln:cve", VULN, "high", 0.0, "CVE-X"),
         ("cred:TOKEN", CRED, "", 0, "TOKEN"), ("tool:read", TOOL, "", 0, "read"), ("tool:write", TOOL, "", 0, "write"),
         ("user:u", USER), ("server:lonely", SRV), ("vuln:srv", VULN, "", 7.5, ""), ("mis:m", MIS, "low"), ("vuln:orphan", VULN, "critical")],
        [("agent:a", "server:a:fs", R.USES), ("server:a:fs", "pkg:npm:form-data", R.DEPENDS_ON), ("pkg:npm:form-data", "vuln:cve", R.VULNERABLE_TO),
         ("server:a:fs", "cred:TOKEN", R.EXPOSES_CRED), ("server:a:fs", "tool:read", R.PROVIDES_TOOL), ("server:a:fs", "tool:write", R.PROVIDES_TOOL),
         ("user:u", "server:a:fs", R.USES), ("server:a:fs", "vuln:srv", R.VULNERABLE_TO), ("server:lonely", "vuln:srv", R.VULNERABLE_TO),
         ("server:lonely", "pkg:npm:form-data", R.DEPENDS_ON), ("vuln:cve", "mis:m", R.TRIGGERS), ("server:a:fs", "mis:m", R.VULNERABLE_TO),
         ("agent:a", "user:u", R.SHARES_CRED, "bidirectional"), ("server:a:fs", "agent:a", R.MANAGES)],
    )


def kat_probe():  # SURVEY §8(a'): order ties, non-traversable, bidirectional, ghost endpoint, self loop, dynamic rels
    g = mk(
        [("s", AG), ("b", SRV), ("a", SRV), ("c", PKG), ("d", VULN, "medium"), ("e", TOOL), ("f", CRED), ("z", AG)],
        [("s", "b", R.USES), ("s", "a", R.USES), ("a", "c", R.DEPENDS_ON), ("b", "c", R.DEPENDS_ON), ("c", "d", R.VULNERABLE_TO, "directed", False),
         ("a", "d", R.SHARES_CRED, "bidirectional"), ("d", "e", R.EXPLOITABLE_VIA), ("e", "e", R.ACCESSED), ("s", "e", R.INVOKED),
         ("f", "f", R.SHARES_SERVER, "bidirectional"), ("z", "s", R.DELEGATED_TO), ("b", "ghost:1", R.CONTAINS), ("ghost:2", "c", R.CONTAINS),
         ("e", "f", R.REACHES_TOOL, "bidirectional", False)],
    )
    return g


def load_generator():
    spec = importlib.util.spec_from_file_location("ref_gen", REF / "scripts" / "generate_graph_benchmark_estate.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def densify(report, c: int, b: int, v: int):
    """Density post-processing probed in SURVEY.md §8(d) (only fields the builder reads)."""
    for ai, agent in enumerate(report["agents"]):
        for si, server in enumerate(agent["mcp_servers"]):
            for ti, tool in enumerate(server["tools"]):
                tool["capabilities"] = ["execute" if ti % 5 == 0 else "read"]
            server["credential_env_vars"] = [f"TEAM{ai // b:05d}_TOKEN_{k}" for k in range(c)]
            for pi, pkg in enumerate(server["packages"][:v]):
                pkg["vulnerabilities"] = [{"id": f"CVE-2027-{ai:06d}{si:02d}{pi:02d}", "severity": ("critical", "high", "medium", "low")[(ai + pi) % 4]}]
    return report


def estate(agents: int, dense=None):
    gen = load_generator()
    report, _ = gen.generate_estate(agents=agents, seed=2145, vulnerable_package_rate=0.08)
    if dense:
        densify(report, *dense)
    return build_unified_graph_from_report(report)


def mesh_inventory():
    """examples/agent-mesh-inventory.json + pinned blast-radius overlay (SURVEY §8d config 1)."""
    inv = json.loads((REF / "examples" / "agent-mesh-inventory.json").read_text())
    rows = []
    sev = ("critical", "high", "medium", "low")
    k = 0
    for agent in inv.get("agents", []):
        for server in agent.get("mcp_servers", []):
            for pkg in server.get("packages", []):
                rows.append({
                    "vulnerability_id": f"CVE-2030-{k:04d}", "severity": sev[k % 4], "package": pkg.get("name", ""),
                    "package_name": pkg.get("name", ""), "package_version": pkg.get("version", ""), "ecosystem": pkg.get("ecosystem", ""),
                    "risk_score": (k % 7) * 1.5,
                })
                k += 1
    inv["blast_radius"] = rows
    return build_unified_graph_from_report(inv)


# ── extraction ──────────────────────────────────────────────────────────────

class Indexer:
    def __init__(self, g: UnifiedGraph):
        self.ids = list(g.nodes.keys())
        self.idx = {nid: i for i, nid in enumerate(self.ids)}
        self.n_real = len(self.ids)
        for e in g.edges:
            for end in (e.source, e.target):
                if end not in self.idx:
                    self.idx[end] = len(self.ids)
                    self.ids.append(end)

    def __call__(self, nid):
        return self.idx[nid]


def graph_arrays(g: UnifiedGraph, ix: Indexer):
    node_types = [ENTITY_CODE[enum_value(n.entity_type)] for n in g.nodes.values()] + [255] * (len(ix.ids) - ix.n_real)
    edges = []
    for e in g.edges:
        flags = (1 if e.traversable else 0) | (2 if e.is_bidirectional else 0)
        edges.append([ix(e.source), ix(e.target), REL_CODE.get(enum_value(e.relationship), REL_CODE_OTHER), flags])
    # cross-check the adjacency model itself (a1): list order of adjacency / reverse_adjacency
    adj = {ix(u): [[ix(e.target), REL_CODE.get(enum_value(e.relationship), REL_CODE_OTHER)] for e in lst] for u, lst in g.adjacency.items() if lst}
    radj = {ix(u): [[ix(e.source), REL_CODE.get(enum_value(e.relationship), REL_CODE_OTHER)] for e in lst] for u, lst in g.reverse_adjacency.items() if lst}
    return node_types, edges, adj, radj


def run_battery(name: str, g: UnifiedGraph, rng: random.Random, small: bool, derived: bool = True):
    doc = battery_doc(name, g, rng, small, derived)
    OUT.mkdir(parents=True, exist_ok=True)
    path = OUT / f"{name}.json.gz"
    with gzip.GzipFile(path, "wb", mtime=0) as fh:
        fh.write(json.dumps(doc, separators=(",", ":"), sort_keys=True).encode())
    print(f"{name}: {doc['n_real']} nodes (+{len(doc['node_ids']) - doc['n_real']} ghosts) {len(doc['edges'])} edges, "
          f"{len(doc['findings'])} findings -> {path.name} {path.stat().st_size / 1024:.0f} KiB")


def battery_doc(name: str, g: UnifiedGraph, rng: random.Random, small: bool, derived: bool = True) -> dict:
    ix = Indexer(g)
    node_types, edges, adj, radj = graph_arrays(g, ix)
    ids = ix.ids
    real = ids[: ix.n_real]
    findings = [n.id for n in g.nodes.values() if enum_value(n.entity_type) in ("vulnerability", "misconfiguration")]
    agents = [n.id for n in g.nodes.values() if enum_value(n.entity_type) == "agent"]

    def sample(pop, k):
        pop = list(pop)
        return pop if len(pop) <= k else rng.sample(pop, k)

    cases: dict = {}

    # impact_of
    imp_sources = (real if small else findings + sample([r for r in real if r not in set(findings)], 300))
    imp = []
    for depth in ((4, 1, 2, 0) if small else (4, 2)):
        for s in imp_sources:
            r = g.impact_of(s, max_depth=depth)
            imp.append({"s": ix(s), "d": depth, "nodes": sorted(ix(x) for x in r["affected_nodes"]), "by_type": r["affected_by_type"],
                        "count": r["affected_count"], "maxd": r["max_depth_reached"]})
    r = g.impact_of("no-such-node")
    cases["impact_missing"] = r
    cases["impact"] = imp

    # bfs (ordered paths)
    bfs_sources = real if small else agents + sample(findings, 50) + sample(real, 100)
    bfs = []
    for depth, trav in (((4, True), (2, True), (3, False), (0, True)) if small else ((4, True), (2, False))):
        for s in bfs_sources:
            bfs.append({"s": ix(s), "d": depth, "t": trav, "paths": [[ix(x) for x in p] for p in g.bfs(s, max_depth=depth, traversable_only=trav)]})
    cases["bfs"] = bfs

    # reachable_from
    rf = []
    for depth, trav, inc in (((6, False, True), (2, True, False), (1, False, True)) if small else ((6, False, True), (3, True, False))):
        for s in (real if small else sample(real, 200) + agents[:50]):
            rf.append({"s": ix(s), "d": depth, "t": trav, "inc": inc,
                       "nodes": sorted(ix(x) for x in g.reachable_from(s, max_depth=depth, traversable_only=trav, include_source=inc))})
    cases["reachable"] = rf

    # shortest_path
    sp = []
    pairs = [(a, b) for a in real for b in real] if small else (
        [(rng.choice(real), rng.choice(real)) for _ in range(300)] + [(rng.choice(agents), rng.choice(findings)) for _ in range(200) if agents and findings])
    for a, b in pairs:
        p = g.shortest_path(a, b)
        sp.append({"a": ix(a), "b": ix(b), "path": None if p is None else [ix(x) for x in p]})
    cases["shortest"] = sp

    # traverse_subgraph
    lateral = {R.SHARES_SERVER, R.SHARES_CRED, R.LATERAL_PATH}
    reach4 = {R.USES, R.DEPENDS_ON, R.CONTAINS, R.PROVIDES_TOOL}
    configs = []
    for direction in ("forward", "reverse", "both"):
        for kw in (
            {}, {"traversable_only": True}, {"relationship_types": reach4}, {"relationship_types": lateral, "max_depth": 2},
            {"static_only": True}, {"dynamic_only": True}, {"include_roots": False}, {"include_roots": False, "max_depth": 2},
            {"max_nodes": 3}, {"max_edges": 4}, {"max_nodes": 7, "max_edges": 30, "max_depth": 6}, {"max_depth": 10, "max_nodes": 100000, "max_edges": 10**9},
            {"max_depth": 0}, {"max_depth": 1, "max_nodes": 1},
        ):
            configs.append((direction, kw))
    root_sets = []
    pool = real
    for _ in range(6 if small else 25):
        root_sets.append([rng.choice(pool)])
    for _ in range(4 if small else 10):
        k = rng.randint(2, 4)
        rs = [rng.choice(pool) for _ in range(k)]
        root_sets.append(rs)
    root_sets.append([pool[0], pool[0], "missing:root", pool[-1]])
    if findings:
        root_sets.append(findings[:3])
    if len(ids) > ix.n_real:
        root_sets.append([ids[ix.n_real]])  # ghost root: skipped by the reference
    trav = []
    for direction, kw in configs:
        for rs in root_sets:
            call = dict(direction=direction, max_depth=4, max_nodes=500, max_edges=10_000)
            call.update(kw)
            sub, depth_by, truncated = g.traverse_subgraph(list(rs), **call)
            rec = {
                "roots": [ix.idx.get(x, -1) for x in rs], "direction": direction,
                "kw": {k: (sorted(REL_CODE[enum_value(r)] for r in v) if k == "relationship_types" else v) for k, v in kw.items()},
                "nodes": sorted(ix(x) for x in sub.nodes), "depth": sorted([ix(k), v] for k, v in depth_by.items()), "truncated": truncated,
                "edges": sorted([ix(e.source), ix(e.target), REL_CODE.get(enum_value(e.relationship), REL_CODE_OTHER)] for e in sub.edges),
            }
            trav.append(rec)
    cases["traverse"] = trav

    # compute_dependency_reach
    rep = compute_dependency_reach(g)
    cases["dependency_reach"] = {
        "packages": [[ix(p.package_id), [ix(a) for a in p.reachable_from], p.min_hop_distance] for p in rep.packages.values()],
        "vulnerabilities": [[ix(v.vulnerability_id), [ix(p) for p in v.package_ids], [ix(a) for a in v.reachable_from], v.min_hop_distance]
                            for v in rep.vulnerabilities.values()],
    }

    # _derived_attack_paths (final, risk-sorted order)
    if derived:
        paths = _derived_attack_paths(g)
        cases["derived_paths"] = [
            {"hops": [ix(h) for h in p.hops], "edges": [REL_CODE[e] for e in p.edges], "risk": p.composite_risk,
             "creds": p.credential_exposure, "tools": p.tool_exposure, "vuln_ids": p.vuln_ids, "source": ix(p.source), "target": ix(p.target)}
            for p in paths
        ]

    doc = {
        "name": name,
        "n_real": ix.n_real,
        "node_ids": ids,
        "node_types": node_types,
        "node_labels": [n.label for n in g.nodes.values()],
        "node_risk": [float(n.risk_score or 0.0) for n in g.nodes.values()],
        "node_severity": [n.severity for n in g.nodes.values()],
        "edges": edges,
        "adjacency": {str(k): v for k, v in adj.items()} if small else None,
        "reverse_adjacency": {str(k): v for k, v in radj.items()} if small else None,
        "findings": [ix(f) for f in findings],
        "agents": [ix(a) for a in agents],
        "cases": cases,
    }
    return doc


def estate_identity():
    """Pin agent_bom_b200.estate: its direct-to-arrays graph must equal what the reference builder makes of its report JSON."""
    from agent_bom_b200 import estate as est_mod

    docs = []
    for agents, knobs, label in ((150, est_mod.Knobs(), "shipped-shape"), (60, est_mod.Knobs.dense(6, 8, 3), "dense-6-8-3"), (90, est_mod.BENCH_KNOBS, "bench-knobs")):
        est = est_mod.generate(agents, 2145, knobs, exact_rank=True)
        g = build_unified_graph_from_report(est.report_json())
        ix = Indexer(g)
        node_types, edges, _, _ = graph_arrays(g, ix)
        docs.append({"label": label, "agents": agents, "seed": 2145, "knobs": dict(knobs.__dict__), "node_ids": ix.ids, "node_types": node_types, "edges": edges,
                     "node_severity": [n.severity for n in g.nodes.values()], "node_labels": [n.label for n in g.nodes.values()]})
        print(f"estate_identity {label}: {len(ix.ids)} nodes {len(edges)} edges")
    path = OUT / "identity" / "estate_identity.json.gz"
    path.parent.mkdir(parents=True, exist_ok=True)
    with gzip.GzipFile(path, "wb", mtime=0) as fh:
        fh.write(json.dumps(docs, separators=(",", ":"), sort_keys=True).encode())
    print(f"-> {path} {path.stat().st_size / 1024:.0f} KiB")


def builder_identity():
    """Pin agent_bom_b200.graph.build_unified_graph_from_report against the reference builder on the same reports.

    The two keyword tables the reference keeps outside its graph package (tool classification, credential-key patterns)
    are captured as lookup tables of the reference's own answers for the names occurring in each report."""
    from agent_bom.constants import is_credential_key
    from agent_bom.risk_analyzer import classify_tool
    from agent_bom_b200 import estate as est_mod

    inv = json.loads((REF / "examples" / "agent-mesh-inventory.json").read_text())
    rows, k = [], 0
    for agent in inv.get("agents", []):
        for server in agent.get("mcp_servers", []):
            for pkg in server.get("packages", []):
                rows.append({"vulnerability_id": f"CVE-2030-{k:04d}", "severity": ("critical", "high", "medium", "low")[k % 4], "package": pkg.get("name", ""),
                             "package_name": pkg.get("name", ""), "package_version": pkg.get("version", ""), "ecosystem": pkg.get("ecosystem", ""),
                             "risk_score": (k % 7) * 1.5})
                k += 1
    mesh = dict(inv, blast_radius=rows)
    reports = [
        ("estate-dense", est_mod.generate(40, 3, est_mod.Knobs.dense(4, 8, 2), exact_rank=True).report_json()),
        ("estate-shipped", est_mod.generate(90, 3, est_mod.Knobs(), exact_rank=True).report_json()),
        ("mesh-inventory", inv),
        ("mesh-inventory+blast-overlay", mesh),
    ]
    docs = []
    for label, report in reports:
        g = build_unified_graph_from_report(json.loads(json.dumps(report)))
        tool_caps, cred_keys = {}, []
        for agent in report.get("agents", []):
            for server in agent.get("mcp_servers", []):
                for tool in server.get("tools", []):
                    key = f"{tool.get('name', '')}|#|{tool.get('description', '')}"
                    tool_caps[key] = [c.value for c in classify_tool(str(tool.get("name", "")), str(tool.get("description", "")))]
                env = server.get("env", {})
                if isinstance(env, dict):
                    cred_keys.extend(k2 for k2 in env if is_credential_key(k2))
        docs.append({
            "label": label, "report": report, "tool_caps": tool_caps, "cred_keys": sorted(set(cred_keys)),
            "nodes": [[n.id, enum_value(n.entity_type), n.label, n.severity, float(n.risk_score or 0.0)] for n in g.nodes.values()],
            "edges": [[e.source, e.target, enum_value(e.relationship), e.direction, bool(e.traversable)] for e in g.edges],
        })
        print(f"builder_identity {label}: {len(g.nodes)} nodes {len(g.edges)} edges")
    path = OUT / "identity" / "builder_identity.json.gz"
    with gzip.GzipFile(path, "wb", mtime=0) as fh:
        fh.write(json.dumps(docs, separators=(",", ":"), sort_keys=True).encode())
    print(f"-> {path} {path.stat().st_size / 1024:.0f} KiB")


def snapshot_identity():
    """Pin agent_bom_b200.graph.snapshot.load_snapshot: a SQLite file written by the reference's own save_graph, and what the
    reference's load_graph makes of every (tenant, scan) in it — node order, edge order, records, materialised paths."""
    import sqlite3
    import tempfile

    from agent_bom.db import graph_store as ref_db

    out_dir = OUT / "snapshot"
    out_dir.mkdir(parents=True, exist_ok=True)
    tmp = Path(tempfile.mkdtemp()) / "graph.sqlite"
    conn = sqlite3.connect(str(tmp))
    conn.row_factory = sqlite3.Row
    ref_db._init_db(conn)

    def stamped(g, scan, tenant, created):
        g.scan_id, g.tenant_id, g.created_at = scan, tenant, created
        return g

    mesh = stamped(mesh_inventory(), "scan-a", "default", "2026-01-01T00:00:00+00:00")
    ref_db.save_graph(conn, mesh)
    dense = stamped(estate(12, dense=(4, 8, 2)), "scan-b", "default", "2026-02-01T00:00:00+00:00")
    dense.attack_paths = _derived_attack_paths(dense)[:40]          # materialised rows win over derived ones
    ref_db.save_graph(conn, dense)
    # scan-a saved again with one node and its edges gone and the rest re-inserted: INSERT OR REPLACE moves the surviving rows
    mesh2 = stamped(mesh_inventory(), "scan-a", "default", "2026-01-01T00:00:00+00:00")
    victim = next(nid for nid, n in mesh2.nodes.items() if enum_value(n.entity_type) == "package")
    del mesh2.nodes[victim]
    ref_db.save_graph(conn, mesh2)
    probe = stamped(kat_probe(), "scan-a", "acme", "2026-03-01T00:00:00+00:00")
    ref_db.save_graph(conn, probe)
    blank = stamped(kat_derived(), "scan-z", "", "2026-04-01T00:00:00+00:00")   # blank tenant -> "default", becomes the newest there
    ref_db.save_graph(conn, blank)
    conn.commit()

    cases = []
    for tenant, scan in (("default", "scan-a"), ("default", "scan-b"), ("default", ""), ("", "scan-z"), ("acme", ""), ("acme", "scan-a"), ("acme", "missing"), ("nobody", "")):
        g = ref_db.load_graph(conn, tenant_id=tenant, scan_id=scan)
        nodes = list(g.nodes.values())
        sample_nodes = nodes[:: max(1, len(nodes) // 12)]
        sample_edges = g.edges[:: max(1, len(g.edges) // 12)]
        cases.append({
            "tenant": tenant, "scan": scan, "scan_id": g.scan_id, "tenant_id": g.tenant_id, "created_at": g.created_at if g.scan_id else "",
            "nodes": [[n.id, enum_value(n.entity_type), n.label, n.severity, float(n.risk_score or 0.0)] for n in nodes],
            "edges": [[e.source, e.target, enum_value(e.relationship), e.direction, bool(e.traversable), float(e.weight)] for e in g.edges],
            "attack_paths": [p.to_dict() for p in g.attack_paths],
            "interaction_risks": [r.to_dict() for r in g.interaction_risks],
            "node_dicts": [n.to_dict() for n in sample_nodes],
            "edge_dicts": [e.to_dict() for e in sample_edges],
        })
        print(f"snapshot_identity {tenant!r}/{scan!r}: -> {g.scan_id!r} {len(g.nodes)} nodes {len(g.edges)} edges {len(g.attack_paths)} paths")
    conn.close()
    with gzip.GzipFile(out_dir / "graph.sqlite.gz", "wb", mtime=0) as fh:
        fh.write(tmp.read_bytes())
    with gzip.GzipFile(out_dir / "expected.json.gz", "wb", mtime=0) as fh:
        fh.write(json.dumps(cases, separators=(",", ":"), sort_keys=True, default=str).encode())
    print(f"-> {out_dir} {sum(f.stat().st_size for f in out_dir.iterdir()) / 1024:.0f} KiB")


def _ctx_doc(name, graph, scores, extra_nodes=()):
    """Serialise a reference ContextGraph (only the fields effective-reach scoring reads) with the reference's answers."""
    keep_node = ("capabilities", "agent", "cvss_score", "epss_score", "is_kev")
    nodes = [[n.id, n.kind.value if hasattr(n.kind, "value") else str(n.kind), n.label, {k: n.metadata[k] for k in keep_node if k in n.metadata}]
             for n in graph.nodes.values()]
    edges = [[e.source, e.target, e.kind.value if hasattr(e.kind, "value") else str(e.kind), {k: e.metadata[k] for k in ("server",) if k in e.metadata}]
             for e in graph.edges]
    adjacency = {nid: [[e.source, e.target, e.kind.value if hasattr(e.kind, "value") else str(e.kind)] for e in lst] for nid, lst in graph.adjacency.items() if lst}
    return {"name": name, "nodes": nodes, "edges": edges, "adjacency": adjacency,
            "scores": {nid: s.as_breakdown() for nid, s in scores.items()},
            "edge_scores": [e.metadata.get("effective_reach_score") for e in graph.edges],
            "extra": [[nid, sc.as_breakdown()] for nid, sc in extra_nodes]}


def effective_reach_golden():
    """Pin agent_bom_b200.effective_reach against the reference's annotate_graph / compute on ContextGraphs built by the
    reference (its own test fixtures, a seeded synthetic fleet with shared servers, and hand-wired corner cases)."""
    import copy

    from agent_bom.context_graph import ContextGraph, EdgeKind, GraphEdge, GraphNode, NodeKind, build_context_graph
    from agent_bom.effective_reach import annotate_graph, compute

    spec = importlib.util.spec_from_file_location("ref_test_effective_reach", REF / "tests" / "test_effective_reach.py")
    ref_tests = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_tests)
    docs = []
    for name, builder in (("low_reach", ref_tests._low_reach_fixture), ("high_reach", ref_tests._high_reach_fixture)):
        agents, blast = builder()
        g = build_context_graph(agents, blast)
        docs.append(_ctx_doc(name, g, annotate_graph(g)))
    agents, blast = ref_tests._high_reach_fixture()
    blast[0]["affected_agents"] = ["claude-desktop"]                     # tests/test_effective_reach.py:175-186
    g = build_context_graph(agents, blast)
    docs.append(_ctx_doc("high_reach_one_listed_agent", g, annotate_graph(g)))
    snapshots = json.loads((REF / "tests" / "fixtures" / "effective_reach_snapshots.json").read_text())
    assert docs[0]["scores"]["vuln:CVE-2099-LOW"] == snapshots["low_reach"] and docs[1]["scores"]["vuln:CVE-2099-HIGH"] == snapshots["high_reach"]

    rng = random.Random(2262)
    env_pool = ["AWS_ACCESS_KEY_ID", "AWS_SECRET_ACCESS_KEY", "GITHUB_TOKEN", "NPM_TOKEN", "DATABASE_URL", "OPENAI_API_KEY", "STRIPE_SECRET_KEY", "SLACK_BOT_TOKEN",
                "INTERNAL_API_KEY", "SERVICE_PASSWORD", "SIGNING_SECRET", "HOME", "PATH", "EDITOR", "MY_SETTING", "DD_API_KEY", "REDIS_URL", "AUTH_TOKEN"]
    tool_pool = [("run_shell", "Execute arbitrary shell commands", ["execute"]), ("list_files", "List files in a directory", ["read"]),
                 ("http_get", "Fetch a URL", ["network"]), ("write_file", "Write a file to disk", ["write"]), ("delete_rows", "Delete rows from a table", ["delete"]),
                 ("grant_role", "Grant an IAM role", ["admin"]), ("login", "Authenticate a user", ["auth"]), ("search_docs", "Search indexed documents", ["read"]),
                 ("noop", "Does nothing in particular", []), ("multi", "Read then write then run", ["read", "write", "execute"])]
    server_pool = [f"srv-{i:02d}" for i in range(14)]
    fleet = []
    for a in range(40):
        servers = []
        for sname in rng.sample(server_pool, rng.randint(1, 4)):
            env = {k: "x" for k in rng.sample(env_pool, rng.randint(0, 5))}
            tools = [{"name": t[0], "description": t[1], "capabilities": list(t[2])} for t in rng.sample(tool_pool, rng.randint(0, 4))]
            servers.append({"name": sname, "command": "node x.js", "transport": "stdio", "env": env, "tools": tools, "packages": [{"name": "left-pad", "version": "1.3.0"}]})
        fleet.append({"name": f"agent-{a:02d}", "type": "custom", "status": "configured", "mcp_servers": servers})
    blast = []
    for v in range(120):
        aff_agents = [f"agent-{i:02d}" for i in rng.sample(range(40), rng.randint(1, 6))]
        blast.append({"vulnerability_id": f"CVE-2031-{v:04d}", "package": "left-pad", "severity": rng.choice(["critical", "high", "medium", "low"]),
                      "cvss_score": rng.choice([None, 0, 3.1, 5.5, 6.5, 7.8, 9.8, 10.0, 11.5]), "epss_score": rng.choice([None, 0.0, 0.013, 0.2, 0.57, 0.92, 1.4]),
                      "is_kev": rng.random() < 0.2, "affected_agents": aff_agents, "affected_servers": rng.sample(server_pool, rng.randint(1, 3))})
    g = build_context_graph(copy.deepcopy(fleet), copy.deepcopy(blast))
    docs.append(_ctx_doc("fleet_40", g, annotate_graph(g)))

    # hand-wired corner cases on the reference's own container
    g = ContextGraph()
    for nid, kind, label, meta in (
            ("agent:a", NodeKind.AGENT, "a", {}), ("agent:b", NodeKind.AGENT, "b", {}), ("agent:c", NodeKind.AGENT, "c", {}),
            ("server:a:s", NodeKind.SERVER, "s", {"agent": "a"}), ("server:b:s", NodeKind.SERVER, "s", {"agent": "b"}), ("server:x", NodeKind.SERVER, "lonely", {}),
            ("tool:1", NodeKind.TOOL, "t-exec", {"capabilities": ["read", "execute"]}), ("tool:2", NodeKind.TOOL, "t-none", {"capabilities": []}),
            ("tool:3", NodeKind.TOOL, "t-unknown", {"capabilities": ["teleport"]}), ("tool:4", NodeKind.TOOL, "t-exec", {"capabilities": ["admin"]}),
            ("cred:1", NodeKind.CREDENTIAL, "AWS_KEY", {}), ("cred:2", NodeKind.CREDENTIAL, "", {}), ("cred:3", NodeKind.CREDENTIAL, "path", {}),
            ("cred:4", NodeKind.CREDENTIAL, " github_token ", {}),
            ("vuln:1", NodeKind.VULNERABILITY, "V1", {"cvss_score": 7.5, "epss_score": 0.3, "is_kev": False}),
            ("vuln:2", NodeKind.VULNERABILITY, "V2", {"cvss_score": "9.1", "epss_score": None, "is_kev": 1}),
            ("vuln:3", NodeKind.VULNERABILITY, "V3-unattached", {}), ("vuln:4", NodeKind.VULNERABILITY, "V4-ghost-server", {"cvss_score": 4.0})):
        g.add_node(GraphNode(id=nid, kind=kind, label=label, metadata=meta))
    for s, t, k, meta in (
            ("agent:a", "server:a:s", EdgeKind.USES, {}), ("agent:b", "server:b:s", EdgeKind.USES, {}), ("agent:c", "server:x", EdgeKind.USES, {}),
            ("server:a:s", "tool:1", EdgeKind.PROVIDES, {}), ("server:a:s", "tool:2", EdgeKind.PROVIDES, {}), ("server:b:s", "tool:3", EdgeKind.PROVIDES, {}),
            ("server:x", "tool:4", EdgeKind.PROVIDES, {}), ("server:a:s", "cred:1", EdgeKind.EXPOSES, {}), ("server:a:s", "cred:2", EdgeKind.EXPOSES, {}),
            ("server:b:s", "cred:3", EdgeKind.EXPOSES, {}), ("server:x", "cred:4", EdgeKind.EXPOSES, {}),
            ("server:a:s", "vuln:1", EdgeKind.VULNERABLE_TO, {}), ("server:x", "vuln:1", EdgeKind.VULNERABLE_TO, {}), ("server:b:s", "vuln:2", EdgeKind.VULNERABLE_TO, {}),
            ("server:ghost", "vuln:4", EdgeKind.VULNERABLE_TO, {}), ("agent:a", "agent:b", EdgeKind.SHARES_SERVER, {"server": "s"}),
            ("agent:a", "agent:c", EdgeKind.SHARES_SERVER, {"server": "other"}), ("agent:b", "agent:c", EdgeKind.SHARES_CREDENTIAL, {"credential": "AWS_KEY"}),
            ("tool:1", "server:b:s", EdgeKind.PROVIDES, {})):               # a PROVIDES pointing INTO a server: its mirrored twin sits in the server's adjacency
        g.add_edge(GraphEdge(source=s, target=t, kind=k, metadata=meta))
    g.adjacency["server:x"].append(GraphEdge(source="server:x", target="agent:b", kind=EdgeKind.USES))      # hand-wired, not in graph.edges (:347-352)
    g.adjacency["server:ghost"].append(GraphEdge(source="server:ghost", target="tool:1", kind=EdgeKind.PROVIDES))
    extra = [(nid, compute(g.nodes[nid], g)) for nid in ("server:a:s", "agent:a")]      # non-vulnerability nodes get the degenerate score
    docs.append(_ctx_doc("hand_wired", g, annotate_graph(g), extra))

    path = OUT / "context" / "effective_reach.json.gz"
    path.parent.mkdir(parents=True, exist_ok=True)
    with gzip.GzipFile(path, "wb", mtime=0) as fh:
        fh.write(json.dumps(docs, separators=(",", ":"), sort_keys=True).encode())
    for d in docs:
        print(f"effective_reach {d['name']}: {len(d['nodes'])} nodes {len(d['edges'])} edges {len(d['scores'])} scored")
    print(f"-> {path} {path.stat().st_size / 1024:.0f} KiB")


def lateral_golden():
    """Pin agent_bom_b200.lateral (and oracle/lateral_oracle.py) against the reference's find_lateral_paths on ContextGraphs the
    reference built: its own effective-reach test fixtures, a seeded fleet with shared servers and credentials, hand-wired corner cases."""
    import copy

    from agent_bom.context_graph import ContextGraph, EdgeKind, GraphEdge, GraphNode, NodeKind, build_context_graph, find_lateral_paths

    spec = importlib.util.spec_from_file_location("ref_test_effective_reach2", REF / "tests" / "test_effective_reach.py")
    ref_tests = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_tests)

    def doc_for(name, g, sources, depths):
        keep_node = ("capabilities", "agent", "severity")
        nodes = [[n.id, n.kind.value, n.label, {k: n.metadata[k] for k in keep_node if k in n.metadata}] for n in g.nodes.values()]
        edges = [[e.source, e.target, e.kind.value, {k: e.metadata[k] for k in ("server", "credential") if k in e.metadata}] for e in g.edges]
        adjacency = {nid: [[e.source, e.target, e.kind.value] for e in lst] for nid, lst in g.adjacency.items() if lst}
        cases = []
        for s in sources:
            for d in depths:
                found = find_lateral_paths(g, s, max_depth=d)
                cases.append({"source": s, "max_depth": d, "paths": [
                    {"source": p.source, "target": p.target, "hops": p.hops, "edges": [k.value for k in p.edges], "composite_risk": p.composite_risk,
                     "summary": p.summary, "credential_exposure": p.credential_exposure, "tool_exposure": p.tool_exposure, "vuln_ids": p.vuln_ids} for p in found]})
        print(f"lateral {name}: {len(nodes)} nodes {len(edges)} edges, {len(cases)} searches, {sum(len(c['paths']) for c in cases)} paths")
        return {"name": name, "nodes": nodes, "edges": edges, "adjacency": adjacency, "cases": cases}

    docs = []
    agents, blast = ref_tests._high_reach_fixture()
    g = build_context_graph(agents, blast)
    docs.append(doc_for("high_reach", g, list(g.nodes) + ["agent:nobody"], (1, 2, 4, 6)))

    rng = random.Random(397)
    env_pool = ["AWS_ACCESS_KEY_ID", "GITHUB_TOKEN", "NPM_TOKEN", "DATABASE_URL", "OPENAI_API_KEY", "SLACK_BOT_TOKEN", "INTERNAL_API_KEY", "SERVICE_PASSWORD"]
    tool_pool = [("run_shell", "Execute arbitrary shell commands", ["execute"]), ("list_files", "List files in a directory", ["read"]),
                 ("http_get", "Fetch a URL", ["network"]), ("write_file", "Write a file to disk", ["write"]), ("exec_sql", "Execute SQL", ["execute"])]
    server_pool = [f"srv-{i:02d}" for i in range(10)]
    fleet = []
    for a in range(24):
        servers = []
        for sname in rng.sample(server_pool, rng.randint(1, 3)):
            env = {k: "x" for k in rng.sample(env_pool, rng.randint(0, 3))}
            tools = [{"name": t[0], "description": t[1], "capabilities": list(t[2])} for t in rng.sample(tool_pool, rng.randint(0, 3))]
            servers.append({"name": sname, "command": "node x.js", "transport": "stdio", "env": env, "tools": tools, "packages": []})
        fleet.append({"name": f"agent-{a:02d}", "type": "custom", "status": "configured", "mcp_servers": servers})
    blast = [{"vulnerability_id": f"CVE-2032-{v:03d}", "package": "p", "severity": rng.choice(["critical", "high", "medium", "low"]),
              "affected_agents": [f"agent-{i:02d}" for i in rng.sample(range(24), rng.randint(1, 4))], "affected_servers": rng.sample(server_pool, 2)} for v in range(30)]
    g = build_context_graph(copy.deepcopy(fleet), copy.deepcopy(blast))
    some = [f"agent:agent-{i:02d}" for i in (0, 5, 11, 23)]
    servers = [nid for nid in g.nodes if nid.startswith("server:")][:3]
    tools = [nid for nid in g.nodes if nid.startswith("tool:")][:2]
    docs.append(doc_for("fleet_24", g, some + servers + tools + [next(n for n in g.nodes if n.startswith("cred:"))], (1, 2, 3, 4)))
    # a sparse fleet (few shared names): searches run deep instead of stopping at 100 one-hop sharing edges
    fleet2 = []
    for a in range(16):
        servers = [{"name": f"own-{a}-{k}", "command": "x", "transport": "stdio", "env": {rng.choice(env_pool): "x"},
                    "tools": [{"name": t[0], "description": t[1], "capabilities": list(t[2])} for t in rng.sample(tool_pool, 2)], "packages": []} for k in range(2)]
        if a % 4 == 0:
            servers.append({"name": "hub", "command": "x", "transport": "stdio", "env": {}, "tools": [], "packages": []})
        fleet2.append({"name": f"a{a:02d}", "type": "custom", "status": "configured", "mcp_servers": servers})
    g = build_context_graph(copy.deepcopy(fleet2), [])
    docs.append(doc_for("fleet_sparse", g, [f"agent:a{i:02d}" for i in (0, 1, 4, 15)] + ["server:a00:hub"], (2, 4, 6)))

    # the scenarios of the reference's own TestLateralPaths (tests/test_context_graph.py:187-300), built with its helpers
    spec2 = importlib.util.spec_from_file_location("ref_test_context_graph", REF / "tests" / "test_context_graph.py")
    rt = importlib.util.module_from_spec(spec2)
    spec2.loader.exec_module(rt)
    scenarios = {
        "shared_server": ([rt._agent(name="agent-a", servers=[rt._server(name="shared-srv")]), rt._agent(name="agent-b", servers=[rt._server(name="shared-srv")])], []),
        "no_cycles": ([rt._agent(name="agent-a", servers=[rt._server(name="shared-srv", env={"API_KEY": "x"})]),
                       rt._agent(name="agent-b", servers=[rt._server(name="shared-srv", env={"API_KEY": "y"})])], []),
        "risk_scoring": ([rt._agent(name="agent-a", servers=[rt._server(name="srv", env={"SECRET_KEY": "x"})]), rt._agent(name="agent-b", servers=[rt._server(name="srv")])],
                         [rt._blast(severity="critical", agents=["agent-a", "agent-b"], servers=["srv"])]),
        "credential_along_path": ([rt._agent(name="agent-a", servers=[rt._server(name="srv", env={"TOKEN": "x"})]), rt._agent(name="agent-b", servers=[rt._server(name="srv")])], []),
        "execute_tool": ([rt._agent(name="agent-a", servers=[rt._server(name="srv", tools=[rt._tool("run_shell", "Execute shell commands")])]),
                          rt._agent(name="agent-b", servers=[rt._server(name="srv")])], []),
        "cap_20_agents": ([rt._agent(name=f"agent-{i}", servers=[rt._server(name="shared")]) for i in range(20)], []),
        "dense_15_agents": ([rt._agent(name=f"agent-{i}", servers=[rt._server(name="shared", env={"KEY": "x"}, tools=[rt._tool("exec", "run code")])]) for i in range(15)], []),
    }
    for label, (agents_data, blast_data) in scenarios.items():
        g = build_context_graph(agents_data, blast_data)
        first = "agent:agent-a" if "agent:agent-a" in g.nodes else "agent:agent-0"
        docs.append(doc_for(f"reference_test_{label}", g, [first, "agent:nonexistent"], (0, 4)))

    g = ContextGraph()
    for nid, kind, label, meta in (
            ("agent:a", NodeKind.AGENT, "a", {}), ("agent:b", NodeKind.AGENT, "b", {}), ("agent:a2", NodeKind.AGENT, "a", {}),
            ("server:a:s", NodeKind.SERVER, "s", {"agent": "a"}), ("server:b:s", NodeKind.SERVER, "s", {"agent": "b"}),
            ("tool:a", NodeKind.TOOL, "ta", {"agent": "a", "capabilities": ["execute"]}), ("tool:b", NodeKind.TOOL, "tb", {"agent": "b", "capabilities": ["execute"]}),
            ("tool:none", NodeKind.TOOL, "tn", {"capabilities": ["read"]}), ("cred:shared", NodeKind.CREDENTIAL, "GITHUB_TOKEN", {"servers": []}),
            ("cred:b", NodeKind.CREDENTIAL, "B_SECRET", {"agent": "b"}), ("vuln:1", NodeKind.VULNERABILITY, "CVE-1", {"severity": "high"}),
            ("iam:r", NodeKind.IAM_ROLE, "role", {})):
        g.add_node(GraphNode(id=nid, kind=kind, label=label, metadata=meta))
    for s, t, k, meta in (
            ("agent:a", "server:a:s", EdgeKind.USES, {}), ("agent:b", "server:b:s", EdgeKind.USES, {}), ("agent:a2", "server:a:s", EdgeKind.USES, {}),
            ("server:a:s", "tool:a", EdgeKind.PROVIDES, {}), ("server:b:s", "tool:b", EdgeKind.PROVIDES, {}), ("server:a:s", "tool:none", EdgeKind.PROVIDES, {}),
            ("server:a:s", "cred:shared", EdgeKind.EXPOSES, {}), ("server:b:s", "cred:shared", EdgeKind.EXPOSES, {}), ("server:b:s", "cred:b", EdgeKind.EXPOSES, {}),
            ("server:b:s", "vuln:1", EdgeKind.VULNERABLE_TO, {}), ("agent:a", "agent:b", EdgeKind.SHARES_SERVER, {"server": "s"}),
            ("agent:a", "agent:b", EdgeKind.SHARES_CREDENTIAL, {"credential": "GITHUB_TOKEN"}),       # parallel edge: the same node sequence arrives twice
            ("iam:r", "agent:a", EdgeKind.ATTACHED_TO, {}), ("server:a:s", "ghost:x", EdgeKind.PROVIDES, {}), ("ghost:x", "agent:b", EdgeKind.USES, {})):
        g.add_edge(GraphEdge(source=s, target=t, kind=k, metadata=meta))
    docs.append(doc_for("hand_wired", g, list(g.nodes) + ["ghost:x"], (0, 1, 2, 3, 5, 7)))

    path = OUT / "context" / "lateral.json.gz"
    path.parent.mkdir(parents=True, exist_ok=True)
    with gzip.GzipFile(path, "wb", mtime=0) as fh:
        fh.write(json.dumps(docs, separators=(",", ":"), sort_keys=True).encode())
    print(f"-> {path} {path.stat().st_size / 1024:.0f} KiB")


def centrality_golden():
    """Pin UnifiedGraph.degree_centrality / bottleneck_nodes (graph/container.py:540-567) on the walk-fixture graphs, and the whole
    GraphBackend surface (graph_backend.py:41-155, 245-306) on op sequences replayed against the reference's InMemoryBackend."""
    from agent_bom.graph_backend import InMemoryBackend, from_unified_graph

    def guarded(fn):
        try:
            return {"value": fn()}
        except KeyError as exc:
            return {"key_error": exc.args[0]}

    unified = {}
    for name, g in (("kat_schema", kat_schema()), ("kat_directed", kat_directed()), ("kat_chain", kat_chain()), ("kat_reach_misc", kat_reach_misc()),
                    ("kat_derived", kat_derived()), ("kat_probe", kat_probe()), ("mesh_inventory", mesh_inventory()), ("estate_150", estate(150)),
                    ("estate_dense_40", estate(40, dense=(6, 8, 3)))):
        unified[name] = {"degree": guarded(g.degree_centrality), "bottleneck_5": guarded(g.bottleneck_nodes),
                         "bottleneck_12": guarded(lambda g=g: g.bottleneck_nodes(top_n=12)), "n_nodes": len(g.nodes)}
        print(f"centrality {name}: {len(g.nodes)} nodes -> {str(unified[name]['bottleneck_5'])[:90]}")

    rng = random.Random(548)
    backends = []

    def record(label, ops, sources, pairs):
        b = InMemoryBackend()
        for op in ops:
            if op[0] == "n":
                b.add_node(op[1], op[2], op[3], **op[4])
            else:
                b.add_edge(op[1], op[2], op[3], op[4], directed=op[5], **op[6])
        ids = list(b._nodes) + sorted({t for nb in b._adj.values() for t in nb} - set(b._nodes))
        doc = {"label": label, "ops": ops, "node_count": b.node_count(), "edge_count": b.edge_count(), "to_dict": b.to_dict(),
               "centrality": guarded(b.centrality_scores), "bottleneck_5": guarded(b.bottleneck_nodes), "bottleneck_20": guarded(lambda: b.bottleneck_nodes(top_n=20)),
               "neighbors": {nid: b.neighbors(nid) for nid in ids[:: max(1, len(ids) // 25)]},
               "has_edge": [[s, t, b.has_edge(s, t)] for s, t in pairs[:40]],
               "bfs": [[s, d, b.bfs(s, d)] for s in sources for d in (0, 1, 2, 4, 9)],
               "shortest": [[s, t, b.shortest_path(s, t)] for s, t in pairs]}
        backends.append(doc)
        print(f"backend {label}: {b.node_count()} nodes {b.edge_count()} edges, {len(doc['bfs'])} bfs, {len(pairs)} pairs")

    # seeded op soup: undirected and directed edges, re-added pairs (attributes overwritten, order kept), self loops, endpoints without a record
    for label, n, m in (("soup-small", 14, 30), ("soup-mid", 120, 420), ("soup-sparse", 300, 340)):
        names = [f"n{i:03d}" for i in range(n)]
        ops = [["n", nid, rng.choice(["agent", "server", "tool"]), nid.upper(), {"tier": rng.randint(0, 3)} if rng.random() < 0.3 else {}] for nid in names]
        rng.shuffle(ops)
        pool = names + ["ghost-a", "ghost-b"]
        for _ in range(m):
            s, t = rng.choice(pool), rng.choice(pool)
            ops.append(["e", s, t, rng.choice(["uses", "provides", "shares_server"]), rng.choice([1.0, 2.0, 3.5]), rng.random() < 0.4, {"note": "x"} if rng.random() < 0.2 else {}])
        if label == "soup-small":
            ops.append(["n", "n001", "agent", "re-added", {}])          # a node added twice keeps its place, takes the new attributes
        sources = rng.sample(names, min(8, n)) + ["ghost-a", "nope"]
        pairs = [[rng.choice(pool + ["nope"]), rng.choice(pool + ["nope"])] for _ in range(60)] + [[names[0], names[0]]]
        record(label, ops, sources, pairs)
    # a 70-node chain plus a star: deep trees, more than 50 nodes so the sample is a strict prefix
    ops = [["n", f"c{i:02d}", "server", f"c{i}", {}] for i in range(70)] + [["n", "hub", "agent", "hub", {}]]
    ops += [["e", f"c{i:02d}", f"c{i + 1:02d}", "uses", 1.0, True, {}] for i in range(69)] + [["e", "hub", f"c{i:02d}", "uses", 1.0, False, {}] for i in range(0, 70, 7)]
    record("chain-and-star", ops, ["c00", "c35", "hub"], [["c00", "c69"], ["c69", "c00"], ["hub", "c33"], ["c10", "hub"]])
    record("empty", [], ["x"], [["x", "y"]])
    ug = mesh_inventory()
    ref_b = from_unified_graph(ug, backend="memory")
    bridge = {"n_nodes": ref_b.node_count(), "n_edges": ref_b.edge_count(), "to_dict": ref_b.to_dict(), "centrality": ref_b.centrality_scores(),
              "bottleneck_10": guarded(lambda: ref_b.bottleneck_nodes(top_n=10)),
              "bfs": [[s, 4, ref_b.bfs(s, 4)] for s in list(ug.nodes)[::9]]}
    path = OUT / "context" / "centrality.json.gz"
    path.parent.mkdir(parents=True, exist_ok=True)
    with gzip.GzipFile(path, "wb", mtime=0) as fh:
        fh.write(json.dumps({"unified": unified, "backends": backends, "mesh_bridge": bridge}, separators=(",", ":"), sort_keys=True).encode())
    print(f"-> {path} {path.stat().st_size / 1024:.0f} KiB")


# ── store contract (SURVEY §8 a10 / b): the reference's own stores answer, method by method ─────────────────────────────
def store_contract():
    """Replay the store-level scenarios of the reference's tests (tests/test_graph_api.py:845-1020 — SQLite store BFS, reverse
    impact, persisted attack paths, edge budget — and the ``_RecordingGraphStore`` cases :1133-1456, the reference's model of a
    complete alternative backend) through the reference's OWN stores and record every method-level answer:

    * ``engine``: a store that delegates to the in-memory engine exactly like ``PostgresGraphStore`` (api/postgres_graph.py:864-931)
      and ``_RecordingGraphStore`` (tests/test_graph_api.py:1319-1375) do — the contract ``B200GraphStore`` follows;
    * ``sqlite``: ``SQLiteGraphStore`` on a file it wrote itself (api/graph_store.py:533-790) — recorded next to it so the known
      deltas (edge budget counts only the traversed direction, silent 5 000 / 25 000 caps) stay visible.
    """
    import tempfile

    from agent_bom.api.graph_store import SQLiteGraphStore
    from agent_bom.graph import AttackPath

    def scen_bfs():            # :845-858
        g = UnifiedGraph(scan_id="traversal-scan", tenant_id="default")
        g.add_node(UnifiedNode(id="agent:a", entity_type=AG, label="agent-a"))
        g.add_node(UnifiedNode(id="server:s", entity_type=SRV, label="server-s"))
        g.add_node(UnifiedNode(id="vuln:cve", entity_type=VULN, label="CVE-2026-1"))
        g.add_edge(UnifiedEdge(source="agent:a", target="server:s", relationship=R.USES, traversable=True))
        g.add_edge(UnifiedEdge(source="server:s", target="vuln:cve", relationship=R.VULNERABLE_TO, traversable=True))
        return g

    def scen_impact():         # :909-921
        g = UnifiedGraph(scan_id="impact-scan", tenant_id="default")
        g.add_node(UnifiedNode(id="agent:a", entity_type=AG, label="agent-a"))
        g.add_node(UnifiedNode(id="server:s", entity_type=SRV, label="server-s"))
        g.add_edge(UnifiedEdge(source="agent:a", target="server:s", relationship=R.USES))
        return g

    def scen_attack_paths():   # :923-959
        g = UnifiedGraph(scan_id="attack-path-scan", tenant_id="default")
        g.add_node(UnifiedNode(id="agent:a", entity_type=AG, label="agent-a"))
        g.add_node(UnifiedNode(id="server:s", entity_type=SRV, label="server-s"))
        g.add_node(UnifiedNode(id="vuln:cve", entity_type=VULN, label="CVE-2026-1"))
        g.add_edge(UnifiedEdge(source="agent:a", target="server:s", relationship=R.USES))
        g.add_edge(UnifiedEdge(source="server:s", target="vuln:cve", relationship=R.VULNERABLE_TO))
        g.attack_paths.append(AttackPath(source="agent:a", target="vuln:cve", hops=["agent:a", "server:s", "vuln:cve"], edges=["uses", "vulnerable_to"], composite_risk=9.8))
        return g

    def scen_attack_fields():  # :961-995
        g = UnifiedGraph(scan_id="attack-path-fields", tenant_id="default")
        g.add_node(UnifiedNode(id="agent:a", entity_type=AG, label="agent-a"))
        g.add_node(UnifiedNode(id="tool:shell", entity_type=TOOL, label="run_shell"))
        g.add_node(UnifiedNode(id="vuln:cve", entity_type=VULN, label="CVE-2026-1"))
        g.add_edge(UnifiedEdge(source="agent:a", target="tool:shell", relationship=R.REACHES_TOOL))
        g.add_edge(UnifiedEdge(source="tool:shell", target="vuln:cve", relationship=R.VULNERABLE_TO))
        g.attack_paths.append(AttackPath(source="agent:a", target="vuln:cve", hops=["agent:a", "tool:shell", "vuln:cve"], edges=["reaches_tool", "vulnerable_to"],
                                         composite_risk=9.9, summary="agent-a can reach run_shell before CVE-2026-1", credential_exposure=["AWS_SECRET_ACCESS_KEY"],
                                         tool_exposure=["run_shell"], vuln_ids=["CVE-2026-1"]))
        g.attack_paths.append(AttackPath(source="agent:a", target="tool:shell", hops=["agent:a", "tool:shell"], edges=["reaches_tool"], composite_risk=4.0))
        return g

    def scen_budget():         # :997-1020
        g = UnifiedGraph(scan_id="budget-scan", tenant_id="default")
        g.add_node(UnifiedNode(id="server:s", entity_type=SRV, label="server-s"))
        g.add_node(UnifiedNode(id="tool:t", entity_type=TOOL, label="tool-t"))
        for index in range(3):
            g.add_node(UnifiedNode(id=f"agent:in-{index}", entity_type=AG, label=f"in-{index}"))
            g.add_edge(UnifiedEdge(source=f"agent:in-{index}", target="server:s", relationship=R.USES))
        g.add_edge(UnifiedEdge(source="server:s", target="tool:t", relationship=R.PROVIDES_TOOL))
        return g

    def scen_recording():      # :1133-1138 — a single-node store
        g = UnifiedGraph(scan_id="store-scan", tenant_id="default")
        g.add_node(UnifiedNode(id="agent:a", entity_type=AG, label="agent-a"))
        return g

    def stamp(g, scan):
        g.scan_id, g.tenant_id = scan, "default"
        return g

    scenarios = [
        ("bfs", scen_bfs(), ["agent:a", "server:s", "vuln:cve", "missing:x"]),
        ("impact", scen_impact(), ["server:s", "agent:a", "missing:x"]),
        ("attack_paths", scen_attack_paths(), ["agent:a", "vuln:cve"]),
        ("attack_fields", scen_attack_fields(), ["agent:a", "tool:shell"]),
        ("budget", scen_budget(), ["server:s", "agent:in-1", "tool:t"]),
        ("recording", scen_recording(), ["agent:a", "missing:x"]),
        ("kat_probe", stamp(kat_probe(), "kat-probe"), None),
        ("kat_derived", stamp(kat_derived(), "kat-derived"), None),
        ("estate_dense", stamp(estate(12, dense=(4, 6, 2)), "estate-dense"), None),
    ]

    class EngineStore:
        """PostgresGraphStore / _RecordingGraphStore delegation over one in-memory graph."""

        def __init__(self, graph):
            self.graph = graph

        def bfs_paths(self, *, tenant_id="", scan_id="", source, max_depth=4, traversable_only=True):
            if not self.graph.has_node(source):
                return [], set()
            return (self.graph.bfs(source, max_depth=max_depth, traversable_only=traversable_only),
                    self.graph.reachable_from(source, max_depth=max_depth, traversable_only=traversable_only, include_source=False))

        def impact_of(self, *, tenant_id="", scan_id="", node_id, max_depth=4):
            return self.graph.impact_of(node_id, max_depth=max_depth) if self.graph.has_node(node_id) else None

        def traverse_subgraph(self, *, tenant_id="", scan_id="", roots, **kw):
            return self.graph.traverse_subgraph(roots, **kw)

        def attack_paths_for_sources(self, *, tenant_id="", scan_id="", source_ids):
            return [p for p in self.graph.attack_paths if p.source in source_ids]

        def attack_paths(self, *, tenant_id="", scan_id="", offset=0, limit=100):
            paths = sorted(self.graph.attack_paths, key=lambda p: (-p.composite_risk, p.source, p.target))
            return self.graph.scan_id, self.graph.created_at, paths[offset: offset + limit], len(paths)

    def ap(p):
        return {"source": p.source, "target": p.target, "hops": list(p.hops), "edges": [enum_value(e) for e in p.edges], "composite_risk": p.composite_risk,
                "summary": p.summary, "credential_exposure": list(p.credential_exposure), "tool_exposure": list(p.tool_exposure), "vuln_ids": list(p.vuln_ids)}

    def sub(res):
        g, depth, trunc = res
        return {"nodes": sorted(g.nodes), "edges": sorted([e.source, e.target, enum_value(e.relationship)] for e in g.edges),
                "depth_by_node": dict(sorted(depth.items())), "truncated": bool(trunc)}

    trav_cfgs = [
        dict(direction="forward", max_depth=1, max_edges=1), dict(direction="forward", max_depth=4), dict(direction="reverse", max_depth=4),
        dict(direction="both", max_depth=3, max_nodes=4), dict(direction="both", max_depth=4, traversable_only=True),
        dict(direction="forward", max_depth=3, relationship_types={"uses", "depends_on", "contains", "provides_tool"}),
        dict(direction="both", max_depth=4, static_only=True), dict(direction="reverse", max_depth=2, include_roots=False),
        dict(direction="both", max_depth=10, max_nodes=5000, max_edges=25000),
    ]
    rng = random.Random(77)
    doc = {"what": "method-level answers of the reference's stores (engine-delegating store and SQLiteGraphStore) for the scenarios of "
                   "tests/test_graph_api.py:845-1020,1133-1456 and three larger fixtures", "scenarios": []}
    for name, g, probes in scenarios:
        ids = list(g.nodes)
        if probes is None:
            probes = rng.sample(ids, min(10, len(ids))) + ["missing:x"]
        tmp = Path(tempfile.mkdtemp()) / "graph.db"
        sq = SQLiteGraphStore(tmp)
        sq.save_graph(g)
        en = EngineStore(g)
        scan = g.scan_id
        calls = []
        for nid in probes:
            for depth, trav in ((3, True), (4, False), (1, True)):
                kw = dict(source=nid, max_depth=depth, traversable_only=trav)
                row = {"method": "bfs_paths", "kwargs": kw}
                for label, st in (("engine", en), ("sqlite", sq)):
                    paths, reach = st.bfs_paths(tenant_id="default", scan_id=scan, **kw)
                    row[label] = {"paths": paths, "reachable": sorted(reach)}
                calls.append(row)
            for depth in (3, 4, 0):
                kw = dict(node_id=nid, max_depth=depth)
                row = {"method": "impact_of", "kwargs": kw}
                for label, st in (("engine", en), ("sqlite", sq)):
                    row[label] = st.impact_of(tenant_id="default", scan_id=scan, **kw)
                calls.append(row)
        for cfg in trav_cfgs:
            roots = [probes[0], probes[-2] if len(probes) > 1 else probes[0], "missing:x"]
            kw = dict(cfg)
            if "relationship_types" in kw:
                kw["relationship_types"] = sorted(kw["relationship_types"])
            row = {"method": "traverse_subgraph", "kwargs": dict(kw, roots=roots)}
            for label, st in (("engine", en), ("sqlite", sq)):
                call_kw = dict(cfg)
                row[label] = sub(st.traverse_subgraph(tenant_id="default", scan_id=scan, roots=list(roots), **call_kw))
            calls.append(row)
        for srcs in ([probes[0]], list(probes), []):
            row = {"method": "attack_paths_for_sources", "kwargs": {"source_ids": sorted(srcs)}}
            for label, st in (("engine", en), ("sqlite", sq)):
                row[label] = sorted((ap(p) for p in st.attack_paths_for_sources(tenant_id="default", scan_id=scan, source_ids=set(srcs))), key=lambda d: (d["source"], d["target"]))
            calls.append(row)
        for off, lim in ((0, 10), (1, 1)):
            row = {"method": "attack_paths", "kwargs": {"offset": off, "limit": lim}}
            for label, st in (("engine", en), ("sqlite", sq)):
                sid, _created, paths, total = st.attack_paths(tenant_id="default", scan_id=scan, offset=off, limit=lim)
                row[label] = {"scan_id": sid, "paths": [ap(p) for p in paths], "total": total}
            calls.append(row)
        # unknown snapshot: the None / empty conventions
        miss = {"bfs_paths": list(sq.bfs_paths(tenant_id="default", scan_id="no-such-scan", source=probes[0], max_depth=3)),
                "impact_of": sq.impact_of(tenant_id="default", scan_id="no-such-scan", node_id=probes[0], max_depth=3),
                "attack_paths_for_sources": sq.attack_paths_for_sources(tenant_id="default", scan_id="no-such-scan", source_ids={probes[0]})}
        miss["bfs_paths"] = [miss["bfs_paths"][0], sorted(miss["bfs_paths"][1])]
        doc["scenarios"].append({
            "name": name, "scan_id": scan,
            "nodes": [[n.id, enum_value(n.entity_type), n.label, n.severity, n.risk_score] for n in g.nodes.values()],
            "edges": [[e.source, e.target, enum_value(e.relationship), e.direction, bool(e.traversable)] for e in g.edges],
            "attack_paths": [ap(p) for p in g.attack_paths], "calls": calls, "missing_snapshot": miss,
        })
        print(f"store contract {name}: {len(g.nodes)} nodes, {len(g.edges)} edges, {len(calls)} calls")
    out = OUT / "store"
    out.mkdir(parents=True, exist_ok=True)
    with gzip.open(out / "contract.json.gz", "wb") as fh:
        fh.write(json.dumps(doc, sort_keys=True).encode())


# ── ExposurePath envelopes (SURVEY §8 f2) ───────────────────────────────────────────────────────────────────────────────
def envelope_golden():
    """REST ``_serialize_attack_path`` (api/routes/graph.py:597-670) and MCP ``_exposure_path_payload`` (mcp_tools/graph.py:78-100)
    of the unmodified reference for ranked derived paths and for hand-made materialised paths (missing hops, ghost endpoints,
    pairs without an edge, bidirectional pairs)."""
    from agent_bom.api.routes.graph import _serialize_attack_path
    from agent_bom.graph import AttackPath
    from agent_bom.mcp_tools.graph import _exposure_path_payload

    def node_rec(n):
        return {"id": n.id, "entity_type": enum_value(n.entity_type), "label": n.label, "severity": n.severity, "risk_score": n.risk_score, "attributes": dict(n.attributes)}

    def edge_rec(e):
        return {"source": e.source, "target": e.target, "relationship": enum_value(e.relationship), "direction": e.direction, "traversable": bool(e.traversable)}

    def ap(p):
        d = p.to_dict()
        d["edges"] = [enum_value(x) for x in d["edges"]]
        return d

    cases = []
    probe = kat_probe()
    manual = [
        AttackPath(source="a", target="d", hops=["a", "d"], edges=["shares_cred"], composite_risk=55.0, summary="bidirectional pair", vuln_ids=[" CVE-X ", "CVE-X"]),
        AttackPath(source="", target="", hops=["s", "b", "c"], edges=[], composite_risk=8.5, summary=""),
        AttackPath(source="s", target="nowhere", hops=["s", "nowhere", "c"], edges=["uses"], composite_risk=3.0, tool_exposure=["t1"], credential_exposure=["K"]),
        AttackPath(source="c", target="d", hops=["c", "d"], edges=["depends_on", "extra"], composite_risk=95.0),
    ]
    graphs = [("kat_derived", kat_derived(), None), ("kat_probe", probe, manual), ("estate_dense", estate(12, dense=(4, 6, 2)), None), ("mesh", mesh_inventory(), None)]
    for name, g, paths in graphs:
        g.scan_id = f"{name}-scan"
        ranked = paths if paths is not None else _derived_attack_paths(g)
        sample = ranked[:120] + ranked[-20:] if len(ranked) > 140 else ranked
        offs = list(range(len(ranked)))[:120] + list(range(len(ranked)))[-20:] if len(ranked) > 140 else list(range(len(ranked)))
        rest = [_serialize_attack_path(p, g.edges, nodes_by_id=g.nodes, rank=r + 1, scan_id=g.scan_id) for p, r in zip(sample, offs)]
        rest_plain = [_serialize_attack_path(p, g.edges) for p in sample[:5]]
        mcp = [_exposure_path_payload(p, nodes_by_id=g.nodes, edges=g.edges, rank=r + 1, scan_id=g.scan_id) for p, r in zip(sample, offs)]
        cases.append({"name": name, "scan_id": g.scan_id, "nodes": [node_rec(n) for n in g.nodes.values()], "edges": [edge_rec(e) for e in g.edges],
                      "paths": [ap(p) for p in sample], "ranks": [r + 1 for r in offs], "rest": rest, "rest_without_nodes": rest_plain, "mcp": mcp})
        print(f"envelope {name}: {len(sample)} of {len(ranked)} paths")
    out = OUT / "envelope"
    out.mkdir(parents=True, exist_ok=True)
    with gzip.open(out / "envelopes.json.gz", "wb") as fh:
        fh.write(json.dumps({"cases": cases}, sort_keys=True).encode())


# ── random estates (tests/test_oracle_vs_reference_live.py) ─────────────────────────────────────────────────────────────
LIVE_SEEDS = list(range(11, 27))


def random_estate(seed: int) -> UnifiedGraph:
    """A typed multigraph through the reference's own add_node / add_edge: an estate-shaped core (agents → servers → packages →
    vulnerabilities, credentials, tools) plus noise edges of every relationship type, bidirectional and non-traversable edges,
    duplicates, self loops and ghost endpoints."""
    rng = random.Random(seed)
    ET = EntityType
    n_agents, n_servers, n_pkgs = rng.randint(2, 6), rng.randint(3, 9), rng.randint(4, 12)
    n_vulns, n_creds, n_tools = rng.randint(3, 14), rng.randint(1, 6), rng.randint(1, 6)
    sev = ["", "low", "medium", "high", "critical"]
    nodes, edges = [], []

    def add(prefix, count, et, with_risk=False):
        ids = []
        for i in range(count):
            nid = f"{prefix}:{seed}:{rng.randrange(10**6):06d}:{i}"
            ids.append(nid)
            if with_risk:
                nodes.append((nid, et, rng.choice(sev), rng.choice([0.0, 0.0, 3.5, 7.5, 9.8]), f"{prefix.upper()}-{i}"))
            else:
                nodes.append((nid, et))
        return ids

    agents, servers, pkgs = add("agent", n_agents, ET.AGENT), add("server", n_servers, ET.SERVER), add("pkg", n_pkgs, ET.PACKAGE)
    vulns = add("vuln", n_vulns, ET.VULNERABILITY, True) + add("mis", rng.randint(0, 3), ET.MISCONFIGURATION, True)
    creds, tools = add("cred", n_creds, ET.CREDENTIAL), add("tool", n_tools, ET.TOOL)
    extra = add("user", rng.randint(0, 2), ET.USER) + add("model", rng.randint(0, 2), ET.MODEL) + add("prov", rng.randint(0, 1), ET.PROVIDER)
    rng.shuffle(nodes)                       # insertion order is what discovery order hangs on
    for a in agents:
        for s in rng.sample(servers, rng.randint(1, min(3, len(servers)))):
            edges.append((a, s, R.USES))
    for s in servers:
        for p in rng.sample(pkgs, rng.randint(0, min(4, len(pkgs)))):
            edges.append((s, p, R.DEPENDS_ON))
        for c in rng.sample(creds, rng.randint(0, min(3, len(creds)))):
            edges.append((s, c, R.EXPOSES_CRED))
        for t in rng.sample(tools, rng.randint(0, min(3, len(tools)))):
            edges.append((s, t, R.PROVIDES_TOOL))
        if rng.random() < 0.3:
            edges.append((s, rng.choice(vulns), R.VULNERABLE_TO))
    for p in pkgs:
        for v in rng.sample(vulns, rng.randint(0, min(3, len(vulns)))):
            edges.append((p, v, R.VULNERABLE_TO))
        if rng.random() < 0.3:
            edges.append((p, rng.choice(pkgs), R.DEPENDS_ON))          # transitive dependency (possibly a self loop)
    for v in rng.sample(vulns, min(3, len(vulns))):
        edges.append((v, rng.choice(pkgs), R.AFFECTS))
    everything = agents + servers + pkgs + vulns + creds + tools + extra
    rels = list(R)
    for _ in range(rng.randint(8, 30)):                                  # noise: any relationship, direction, traversability
        a, b = rng.choice(everything), rng.choice(everything)
        edges.append((a, b, rng.choice(rels), rng.choice(["directed", "directed", "bidirectional"]), rng.random() > 0.2))
    for _ in range(rng.randint(0, 3)):                                   # ghost endpoints
        edges.append((rng.choice(everything), f"ghost:{seed}:{rng.randrange(1000)}", rng.choice(rels)))
        edges.append((f"ghost:{seed}:{rng.randrange(1000)}", rng.choice(everything), rng.choice(rels)))
    edges += rng.sample(edges, min(5, len(edges)))                       # exact duplicates: add_edge keeps the first
    rng.shuffle(edges)
    return mk(nodes, edges)


def live_golden():
    """tests/golden/live/estates.json.xz: the list of small-battery fixtures, one random estate per seed, in one xz stream
    (per-file gzip would be half as large again)."""
    docs = [battery_doc(f"live_{seed}", random_estate(seed), random.Random(seed), small=True) for seed in LIVE_SEEDS]
    path = OUT / "live" / "estates.json.xz"
    path.parent.mkdir(parents=True, exist_ok=True)
    path.write_bytes(lzma.compress(json.dumps(docs, separators=(",", ":"), sort_keys=True).encode(), preset=9 | lzma.PRESET_EXTREME))
    print(f"live estates: {len(docs)} seeds -> {path.name} {path.stat().st_size / 1024:.0f} KiB")


def main():
    if "--live-only" in sys.argv:
        live_golden()
        return
    if "--envelope-only" in sys.argv:
        envelope_golden()
        return
    if "--store-only" in sys.argv:
        store_contract()
        return
    if "--lateral-only" in sys.argv:
        lateral_golden()
        return
    if "--centrality-only" in sys.argv:
        centrality_golden()
        return
    if "--effective-reach-only" in sys.argv:
        effective_reach_golden()
        return
    if "--snapshot-only" in sys.argv:
        snapshot_identity()
        return
    if "--identity-only" in sys.argv:
        estate_identity()
        builder_identity()
        snapshot_identity()
        return
    store_contract()
    envelope_golden()
    estate_identity()
    builder_identity()
    snapshot_identity()
    effective_reach_golden()
    centrality_golden()
    lateral_golden()
    live_golden()
    rng = random.Random(20260921)
    run_battery("kat_schema", kat_schema(), rng, small=True)
    run_battery("kat_directed", kat_directed(), rng, small=True)
    run_battery("kat_chain", kat_chain(), rng, small=True)
    run_battery("kat_reach_misc", kat_reach_misc(), rng, small=True)
    run_battery("kat_derived", kat_derived(), rng, small=True)
    run_battery("kat_probe", kat_probe(), rng, small=True)
    run_battery("mesh_inventory", mesh_inventory(), rng, small=False)
    run_battery("estate_150", estate(150), rng, small=False)
    run_battery("estate_dense_40", estate(40, dense=(6, 8, 3)), rng, small=False)


if __name__ == "__main__":
    main()
