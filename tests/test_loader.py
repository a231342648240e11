"""Loader (SURVEY.md §8 row f-1): Jaeger JSON -> SoA problems.

1. Against the goldens: the hotel_reservation fixtures were minted from the reference's own loader
   (executor.py) on the shipped trace directories; `load_jaeger_dir` on the same directories must
   hand the engine the same arrays, the same invocation graph and the same ground truth.  The raw
   traces are the original project's data/ directory (25 MB per trace directory, not committed): set
   TW_REFERENCE_DATA to it to run this part; without it this part is skipped.
2. Self-contained: synthetic services are written out as Jaeger JSON files (one trace per request,
   server span -> client spans -> callee server spans) and read back; the loader must reproduce the
   generator's arrays, DAG and ground truth.
"""
import glob
import json
import os

import numpy as np
import pytest

from golden_util import Golden

HERE = os.path.dirname(os.path.abspath(__file__))
REF_ROOT = os.environ.get("TW_REFERENCE_DATA", "")
REF_DATA = os.path.join(REF_ROOT, "hotel_reservation") if REF_ROOT else ""
GOLDENS = sorted(glob.glob(os.path.join(HERE, "golden", "hotel_load*__*.npz")) +
                 glob.glob(os.path.join(HERE, "golden", "media_load*__*.npz")) +
                 glob.glob(os.path.join(HERE, "golden", "node_load*__*.npz")))
ALIBABA = sorted(glob.glob(os.path.join(HERE, "golden", "alibaba_synth__*.npz")))
_cache = {}


def _services(dataset):
    from traceweaver_b200.loader import load_jaeger_dir
    if dataset not in _cache:
        layout = dataset.split("_")[0]
        sub = {"hotel": "hotel_reservation", "media": "media_microservices", "node": "nodejs_microservices"}[layout]
        _cache[dataset] = {s.name: s for s in load_jaeger_dir(os.path.join(REF_ROOT, sub, dataset), layout=layout)}
    return _cache[dataset]


def _loopless(name):
    """The reference names a self-loop service with a random id ("<16 random characters>-loop",
    executor.py:396-398), the loader with "<callee>-<n>-loop": compare them as one token."""
    return "<loop>" if name.endswith("-loop") else name


@pytest.mark.parametrize("path", ALIBABA, ids=[os.path.basename(p)[:-4] for p in ALIBABA])
def test_alibaba_layout_matches_reference_loader(path):
    """`--fix 5` (executor.py:377-470) on the committed synthetic traces of the Alibaba ETL's layout
    (tests/golden/make_alibaba_traces.py; fixtures minted by the reference run with --fix 5)."""
    from traceweaver_b200.loader import load_jaeger_dir
    if "alibaba" not in _cache:
        _cache["alibaba"] = {_loopless(s.name): s for s in
                             load_jaeger_dir(os.path.join(HERE, "golden", "alibaba_synth"), layout="alibaba")}
    g = Golden(path)
    z, m = g.z, g.meta
    svc = _cache["alibaba"][_loopless(m["process"])]
    assert _loopless(svc.in_ep) == _loopless(m["in_ep"])
    assert [_loopless(e) for e in svc.out_eps_given] == [_loopless(e) for e in m["out_eps_given"]]
    assert [_loopless(e) for e in svc.out_eps] == [_loopless(e) for e in m["out_eps_topo"]]
    assert [[_loopless(a), _loopless(b)] for a, b in svc.graph_edges] == [[_loopless(a), _loopless(b)] for a, b in m["graph_edges"]]
    want, got = g.problem(), svc.problem
    assert np.array_equal(got.in_start, want.in_start) and np.array_equal(got.in_end, want.in_end)
    assert got.preds == want.preds
    for e in range(g.E):
        assert np.array_equal(got.out_start[e], want.out_start[e]) and np.array_equal(got.out_end[e], want.out_end[e])
    assert [t for t, _ in svc.in_ids] == list(z["in_trace"]) and [s for _, s in svc.in_ids] == list(z["in_sid"])
    for e, gidx in enumerate(g.pos_given):
        assert [s for _, s in svc.out_ids[e]] == list(z[f"out{gidx}_sid"])
    assert np.array_equal(svc.truth, z["truth"])


@pytest.mark.skipif(not os.path.isdir(REF_DATA), reason="TW_REFERENCE_DATA (the original project's data/ directory) is not set")
@pytest.mark.parametrize("path", GOLDENS, ids=[os.path.basename(p)[:-4] for p in GOLDENS])
def test_loader_matches_reference_loader(path):
    g = Golden(path)
    z, m = g.z, g.meta
    svc = _services(m["dataset"])[m["process"]]
    assert svc.in_ep == m["in_ep"]
    assert svc.out_eps_given == m["out_eps_given"]
    assert svc.out_eps == m["out_eps_topo"]
    assert [list(e) for e in svc.graph_edges] == m["graph_edges"]
    want = g.problem()
    got = svc.problem
    assert np.array_equal(got.in_start, want.in_start) and np.array_equal(got.in_end, want.in_end)
    assert got.preds == want.preds
    for e in range(g.E):
        assert np.array_equal(got.out_start[e], want.out_start[e]), e
        assert np.array_equal(got.out_end[e], want.out_end[e]), e
    assert [t for t, _ in svc.in_ids] == list(z["in_trace"]) and [s for _, s in svc.in_ids] == list(z["in_sid"])
    for e, gidx in enumerate(g.pos_given):
        assert [t for t, _ in svc.out_ids[e]] == list(z[f"out{gidx}_trace"])
        assert [s for _, s in svc.out_ids[e]] == list(z[f"out{gidx}_sid"])
    assert np.array_equal(svc.truth, z["truth"])


def _write_traces(block, s, directory, callee_names, root_op="HTTP GET /hotels"):
    """Service `s` of a synthetic block as one Jaeger trace file per request."""
    E = len(block.out_start)
    n = block.in_start.shape[1]
    kind = lambda v: [{"key": "span.kind", "type": "string", "value": v}]
    procs = {"p0": {"serviceName": "front", "tags": []}}
    for e in range(E):
        procs[f"p{e + 1}"] = {"serviceName": callee_names[e], "tags": []}
    for i in range(n):
        tid = f"{i:016x}"
        ref = lambda sid: [{"refType": "CHILD_OF", "traceID": tid, "spanID": sid}]
        spans = []
        for e in reversed(range(E)):                    # JSON order is not the call order
            j = int(block.truth[e, s, i])
            st, en = int(block.out_start[e][s, j]), int(block.out_end[e][s, j])
            spans.append({"traceID": tid, "spanID": f"s{e}", "operationName": f"/callee{e}", "references": ref(f"c{e}"),
                          "startTime": st + 1, "duration": max(en - st - 2, 0), "tags": kind("server"),
                          "processID": f"p{e + 1}"})
            spans.append({"traceID": tid, "spanID": f"c{e}", "operationName": f"/callee{e}", "references": ref("root"),
                          "startTime": st, "duration": en - st, "tags": kind("client"), "processID": "p0"})
        spans.append({"traceID": tid, "spanID": "root", "operationName": root_op, "references": [],
                      "startTime": int(block.in_start[s, i]), "duration": int(block.in_end[s, i] - block.in_start[s, i]),
                      "tags": kind("server"), "processID": "p0"})
        with open(os.path.join(directory, f"{(n - i):05d}.json"), "w") as fh:     # file names in reverse time order
            json.dump({"data": [{"traceID": tid, "spans": spans, "processes": procs}]}, fh)


@pytest.mark.parametrize("shape,load", [("hotel_frontend", 150.0), ("hotel_search", 100.0), ("media_nginx", 120.0)])
def test_loader_roundtrip_on_synthetic_traces(tmp_path, shape, load):
    from traceweaver_b200 import synth
    from traceweaver_b200.loader import load_jaeger_dir, to_host_batch, accuracy
    blk = synth.make_block(shape, 2, 120, load, seed=3)
    E = len(blk.out_start)
    names = [f"svc{e}" for e in range(E)]
    _write_traces(blk, 1, str(tmp_path), names)
    services = load_jaeger_dir(str(tmp_path))
    assert [s.name for s in services] == ["front"]                 # the callees make no calls of their own
    svc = services[0]
    want = blk.problem(1)
    # the generator's ep order is a topological order of its DAG; the loader derives the DAG from the
    # traces (an edge survives iff it is never violated), which contains the generator's edges
    order = [names.index(ep) for ep in svc.out_eps]
    assert np.array_equal(svc.problem.in_start, want.in_start) and np.array_equal(svc.problem.in_end, want.in_end)
    for e, g in enumerate(order):
        assert np.array_equal(svc.problem.out_start[e], want.out_start[g])
        assert np.array_equal(svc.problem.out_end[e], want.out_end[g])
        assert np.array_equal(svc.truth[e], blk.truth[g, 1])
        for b in want.preds[g]:
            assert order.index(b) in svc.problem.preds[e]
    hb = to_host_batch(services)
    assert hb.n_problems == 1 and hb.no_skip()
    assert accuracy(svc, svc.truth) == 1.0


def test_loader_rejects_what_the_reference_rejects(tmp_path):
    from traceweaver_b200 import synth
    from traceweaver_b200.loader import load_jaeger_dir
    blk = synth.make_block("hotel_search", 1, 5, 100.0, seed=1)
    _write_traces(blk, 0, str(tmp_path), ["a", "b"], root_op="HTTP GET /other")
    assert load_jaeger_dir(str(tmp_path)) == []                    # first-span filter, executor.py:838
    f = sorted(glob.glob(str(tmp_path / "*.json")))[0]
    d = json.load(open(f))
    d["data"][0]["spans"][0]["tags"] = []
    json.dump(d, open(f, "w"))
    with pytest.raises(ValueError):
        load_jaeger_dir(str(tmp_path), first_span="HTTP GET /other")
