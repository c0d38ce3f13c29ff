"""CPU: host-side logic and the C-ABI surface (no compute calls — there is no GPU here)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from oracle import fitgnn_oracle as fo
from tests import golden_io as gio

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_header_symbol():
    import fitgnn_b200
    hdr = open(os.path.join(ROOT, "include", "fitgnn.h")).read()
    declared = set(re.findall(r"\b(fitgnn_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(fitgnn_b200._lib.SIGNATURES), declared ^ set(fitgnn_b200._lib.SIGNATURES)
    handle = ctypes.CDLL(fitgnn_b200._lib.LIB_PATH)
    for name in declared:
        assert hasattr(handle, name), name
    assert handle.fitgnn_abi_version() == 1


def test_struct_layouts_match_header():
    import fitgnn_b200
    assert ctypes.sizeof(fitgnn_b200._lib.PackStruct) == 5 * 8 + 8 * 8
    assert ctypes.sizeof(fitgnn_b200._lib.PlanStruct) == (6 + 27) * 8


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "fitgnn_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert "fitgnn_oracle" not in src, f


def test_cpu_tensors_are_rejected():
    import fitgnn_b200
    with pytest.raises(fitgnn_b200._lib.FitgnnError):
        fitgnn_b200.ops.gemm_bias_act(torch.zeros(2, 4), torch.zeros(4, 4))
    conv = fitgnn_b200.GCNConv(4, 8)
    with pytest.raises(RuntimeError):
        conv(torch.zeros(3, 4), torch.zeros(2, 0, dtype=torch.long))


def test_state_dict_keys_match_reference():
    import argparse
    import fitgnn_b200
    args = argparse.Namespace(num_layers1=2, num_features=12, hidden=32, num_classes=4, layer_name="GCNConv")
    sd = gio.state_dict(gio.load("node_small"))
    for cls in (fitgnn_b200.Classify_node, fitgnn_b200.Classify_graph_gc, fitgnn_b200.Classify_graph_gs):
        m = cls(args)
        assert set(m.state_dict().keys()) == set(sd.keys())
        m.load_state_dict(sd)
    assert fitgnn_b200.Regress_node(args).lt1.out_features == 1
    with pytest.raises(NotImplementedError):
        fitgnn_b200.Classify_node(argparse.Namespace(num_layers1=2, num_features=4, hidden=8, num_classes=2,
                                                     layer_name="GATConv"))


@pytest.mark.parametrize("mode", ["none", "extra", "cluster"])
def test_partition_from_components_matches_reference_order(mode):
    import fitgnn_b200
    d = gio.load("node_small")
    comps = gio.components(d, mode)
    cos = gio.coarsenings_for_oracle(d, mode, comps)
    p = fitgnn_b200.coarsen.partition_from_components(comps, [c["C"] if c else None for c in cos], int(d["n"]))
    ref = gio.subgraphs(d, mode + "_sub")
    assert p.k == len(ref)
    # every node's subgraph is the one whose map_dict / core set holds it
    subs = fo.build_subgraphs(d["edge_index"], d["x"], d["y"], comps, cos, mode)
    assert np.array_equal(p.part, fo.partition_vector(subs, int(d["n"])))


def test_synth_generators_are_seeded():
    import fitgnn_b200
    a = fitgnn_b200.synth.powerlaw_graph(500, 1200, seed=1)
    b = fitgnn_b200.synth.powerlaw_graph(500, 1200, seed=1)
    assert np.array_equal(a, b)
    pa, comps, C_list = fitgnn_b200.synth.neighborhood_partition(a, 500, 0.3, seed=1)
    pb, _, _ = fitgnn_b200.synth.neighborhood_partition(a, 500, 0.3, seed=1)
    assert np.array_equal(pa.part, pb.part)
    # ratio is honoured per component: k_c == ceil(ratio * n_c) unless neighbourhoods run out
    for comp, C in zip(comps, C_list):
        if C is not None:
            assert C.shape[0] >= int(np.ceil(0.3 * len(comp)))
            assert np.all(np.diff(C.tocsc().indptr) == 1)
    ei, part, cw, k = fitgnn_b200.synth.planted_partition(3000, 20000, 0.5, seed=2, device="cpu")
    ei2, part2, _, _ = fitgnn_b200.synth.planted_partition(3000, 20000, 0.5, seed=2, device="cpu")
    assert torch.equal(ei, ei2) and torch.equal(part, part2)
    assert int(part.max()) + 1 == k and ei.shape[0] == 2
    sizes = torch.bincount(part.long())
    assert torch.allclose(cw, 1.0 / torch.sqrt(sizes[part.long()].double()))


def test_oracle_aligned_layout_invariants():
    """The layout checker itself: in-order greedy placement, no subgraph straddles a multiple of 32, padding only at
    group tails, nothing moves when everything already fits."""
    import numpy as np
    from oracle import fitgnn_oracle as fo
    rng = np.random.default_rng(0)
    sizes = rng.integers(1, 14, 5000)
    sub_ptr = np.concatenate([[0], np.cumsum(sizes)])
    new_start, n_al = fo.aligned_layout(sub_ptr, 32)
    assert (np.diff(new_start[:-1]) >= sizes[:-1]).all() and n_al == new_start[-2] + sizes[-1]
    first, last = new_start[:-1], new_start[:-1] + sizes - 1
    assert (first // 32 == last // 32).all()
    pad = np.diff(new_start) - sizes  # padding rows after each subgraph
    nxt = new_start[1:-1]
    assert ((pad[:-1] == 0) | (nxt % 32 == 0)).all() and pad[-1] == 0
    assert 1.0 <= n_al / sub_ptr[-1] < 1.25
    assert fo.aligned_layout([0, 33], 32) is None
    s2, n2 = fo.aligned_layout([0, 32, 64, 96], 32)
    assert list(s2) == [0, 32, 64, 96] and n2 == 96
    # known answer (sizes 3,7,20,3,7,24,6)
    s3, n3 = fo.aligned_layout([0, 3, 10, 30, 33, 40, 64, 70], 32)
    assert list(s3) == [0, 3, 10, 32, 35, 64, 88, 94] and n3 == 94
    # degree policy: (max row degree desc, size desc, index asc) with gap filling from the end of that order.
    # sizes 3,1,1,30 with chain graphs inside (row degree incl. self loop: 2,3,2 | 1 | 1 | 2,3,...,3,2)
    sub_ptr = np.array([0, 3, 4, 5, 35])
    deg = np.concatenate([[2, 3, 2], [1], [1], [2] + [3] * 28 + [2]])
    rowptr = np.concatenate([[0], np.cumsum(deg)])
    s4, n4 = fo.aligned_layout(sub_ptr, 32, "degree", rowptr)
    # order: sub 3 (deg 2, size 30), sub 0 (deg 2, size 3), sub 1, sub 2 (deg 0).  sub 3 -> 0..29; sub 0 does not fit the
    # 2 remaining rows -> the tail fills them: sub 2 at 30, sub 1 at 31; then sub 0 at 32
    assert list(s4) == [32, 31, 30, 0, 35] and n4 == 35
    s5, n5 = fo.aligned_layout(sub_ptr, 32, "order", rowptr)
    assert list(s5) == [0, 3, 4, 32, 62] and n5 == 62


def test_bench_reference_arm_contract_on_cpu():
    """`bench.py --impl reference` (the oracle port of node_infer_Gs_GD timed on the host cores) prints ONE JSON line with
    the keys the driver reads; run here on the small workload (no GPU involved)."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload",
                          "products-small", "--steps", "1", "--warmup", "0", "--cpu-seconds", "1"],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "subgraph-inference nodes/sec" and d["unit"] == "nodes/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": "nodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "subgraphs" in cb["sample"]
    assert set(d["config"]) >= {"workload", "subgraphs", "mode", "l2", "features"} and "model" not in d["config"]
    # ranks other than 0 print nothing and exit 0 (torchrun launches every rank)
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=root, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.parametrize("flags", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "d"],
                                   ["--gpus", "2", "--dump-outputs", "d"], ["--only-modes", "--dump-outputs", "d"]])
def test_bench_refuses_arguments_it_cannot_honour(tmp_path, flags):
    """No timed step, or a dump of a run whose timed path is not the single-GPU headline: a usage error before any work."""
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + flags, capture_output=True, text=True, timeout=120,
                         cwd=tmp_path)
    assert out.returncode == 2 and "error:" in out.stderr and out.stdout == ""
    assert os.listdir(tmp_path) == []


@pytest.mark.parametrize("mode,flags", [("none", {}), ("extra", dict(extra_node=True)), ("cluster", dict(extra_node=True, cluster_node=True))])
def test_reference_cache_layout_roundtrip(tmp_path, mode, flags):
    """The reference's preprocessing cache (main.py:131-172 `save()`, read at main.py:270-275 / inference.py:543-548): file
    names, node_type / graph_type rules, un-pickling behind stand-ins for torch_geometric / pygsp, and the partition derived
    from candidate + C_list == the one derived from the fixture's components (the device builders' input)."""
    from oracle import ref_shims
    ref_shims.install()
    import fitgnn_b200 as fg
    from fitgnn_b200 import cache as fc
    d = gio.load("node_small")
    comps = gio.components(d, mode)
    cos = gio.coarsenings_for_oracle(d, mode, comps)
    subs = [ref_shims.Data(x=torch.tensor(s["x"]), edge_index=torch.tensor(s["edge_index"]), y=torch.tensor(s["y"]),
                           mask=torch.tensor(s["mask"]), orig_idx=torch.tensor(s["orig_idx"])) for s in gio.subgraphs(d, mode + "_sub")]
    cand = []
    for comp in comps:
        g = ref_shims.Graph(np.zeros((len(comp), len(comp))))
        g.info = {"orig_idx": np.asarray(comp)}
        cand.append(g)
    C_list = [c["C"] for c in cos if c is not None]       # only components with > 1 node have a C (utils.py:164-166)
    Gc_list = [ref_shims.Graph(c["W"]) for c in cos if c is not None]
    paths = fc.save_reference_cache(str(tmp_path), "cora", "variation_neighborhoods", 0.3, "node_cls", subs, cand, C_list, Gc_list,
                                    **flags)
    tag = {"none": "d", "extra": "e", "cluster": "c"}[mode]  # cluster_node wins over extra_node (main.py:117-121)
    assert paths["subgraph_list"].endswith(f"dataset/cora/saved/variation_neighborhoods/0.3_{tag}_full_subgraph_list.pt")
    assert sorted(os.listdir(os.path.dirname(paths["subgraph_list"]))) == sorted(
        f"0.3_{tag}_full_{f}" for f in ("subgraph_list.pt", "candidate.pkl", "C_list.pkl", "Gc_list.pkl"))
    got = fc.load_reference_cache(str(tmp_path), "cora", "variation_neighborhoods", 0.3, **flags)
    assert not got.graph_level and len(got.subgraph_list) == len(subs) and got.saved_graph_list is None
    assert all(torch.equal(a.edge_index, b.edge_index) and torch.equal(a.x, b.x) for a, b in zip(got.subgraph_list, subs))
    partition, comps2, C2 = fc.partition_from_cache(got, int(d["n"]))
    want = fg.coarsen.partition_from_components(comps, [c["C"] if c is not None else None for c in cos], int(d["n"]))
    assert np.array_equal(partition.part, want.part) and np.array_equal(partition.cweight, want.cweight) and partition.k == want.k
    assert fc.cache_paths("r", "x", "m", 0.5, use_community_detection=True)["Gc_list"].endswith("0.5_d_community_Gc_list.pkl")
    with pytest.raises(FileNotFoundError):
        fc.load_reference_cache(str(tmp_path), "cora", "variation_neighborhoods", 0.7)
    # graph-task layout: list of lists + Gc_list + saved_graph_list, no candidate / C_list (main.py:154-171)
    gpaths = fc.save_reference_cache(str(tmp_path), "zinc", "variation_neighborhoods", 0.3, "graph_reg", [subs[:2], subs[2:5]],
                                     Gc_list=subs[:2], saved_graph_list=[0, 3])
    gg = fc.load_reference_cache(str(tmp_path), "zinc", "variation_neighborhoods", 0.3)
    assert gg.graph_level and gg.saved_graph_list == [0, 3] and gg.candidate is None and len(gg.Gc_list) == 2
    assert not os.path.exists(gpaths["candidate"])


def test_tuning_switches_are_known_to_the_library():
    """fitgnn_tuning_get / _set are host-only: every switch include/fitgnn.h documents exists, unknown names are refused,
    a set value reads back (no GPU involved)."""
    import ctypes as C
    from fitgnn_b200._lib import FitgnnError, lib, set_tuning
    names = ["gemm_ws", "head_bulk", "agg_wide", "gemm_wide", "gemm_pair", "gemm_pair_ws", "gemm_prefetch", "sm_reserve",
             "gemm_debug"]
    header = open(os.path.join(ROOT, "include", "fitgnn.h")).read().lower()
    for name in names:
        v = C.c_int32(-12345)
        assert lib().fitgnn_tuning_get(name.encode(), C.byref(v)) == 0 and v.value != -12345, name
        assert name in header, f"{name} is not documented in include/fitgnn.h"
        old = set_tuning(name, v.value + 1)
        assert old == v.value
        w = C.c_int32(0)
        lib().fitgnn_tuning_get(name.encode(), C.byref(w))
        assert w.value == v.value + 1
        set_tuning(name, old)
    assert lib().fitgnn_tuning_get(b"gemm_debug", C.byref(v)) == 0 and v.value == 0  # never on by default
    with pytest.raises(FitgnnError):
        set_tuning("no_such_switch", 1)
