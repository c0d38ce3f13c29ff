#!/usr/bin/env python
"""Benchmark of the hot path on BASELINE.json's headline workload.

  python bench.py [--gpus N] [--steps K] [--warmup W]              (torchrun launches N>1, one rank per GPU)
  python bench.py --impl reference [...]                            (the restated reference CPU path)

Workload (config.workload = "products"): ogbn-products-shaped synthetic graph — 2,449,029 nodes, 61,859,140
undirected edges, 100 features, 47 classes, planted partition at coarsening ratio 0.5 — all subgraphs Gs
through a 2-layer GCN (hidden 512) + lt1 + log_softmax.  One step = one forward of EVERY subgraph, i.e. logits
for every node.  metric = subgraph-inference nodes/sec.  Prints one JSON line (rank 0).
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
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PROFILER_RANGE = False  # --profiler-range together with --only-modes: cudaProfilerStart/Stop around the blocks' timed steps
METRIC = "subgraph-inference nodes/sec"
UNIT = "nodes/s"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--workload", default="products", choices=["products", "products-small"])
    p.add_argument("--mode", default="none", choices=["none", "extra", "cluster"])
    p.add_argument("--ratio", type=float, default=0.5)
    p.add_argument("--precision", default="auto", choices=["auto", "fp32", "bf16x3", "fp16x2", "fp16"],
                   help="arithmetic of the dense transforms: bf16x3 = bf16 hi/lo planes for both operands, 3 MMAs (fp32-grade: parity "
                        "~5e-7); fp16x2 = bf16x3 first layer, then the hidden state as ONE fp16 plane, 2 MMAs (parity ~1.5e-5 of the "
                        "1e-3 bound; the verdict's '2 instead of 3 MMAs for the K = 512 layer'); fp16 = fp16x2 with ONE fp16 weight plane in "
                        "the 512 x 512 transform (1 MMA, W-stationary CTA pairs; parity ~1.8e-5); fp32 = CUDA-core GEMM; auto = fp16")
    p.add_argument("--hidden", type=int, default=512)
    p.add_argument("--cpu-seconds", type=float, default=15.0, help="CPU work budget of the cpu_baseline sample")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--profiler-range", action="store_true",
                   help="cudaProfilerStart/Stop around the timed steps (for `ncu --profile-from-start off`)")
    p.add_argument("--no-projection", action="store_true", help="skip the Gc projection kernels (Xc = C·X, Ac = P·A·P^T)")
    p.add_argument("--align-policy", default="degree", choices=["degree", "order"],
                   help="placement of the subgraphs in the group-aligned pack (see include/fitgnn.h)")
    p.add_argument("--no-fuse-aggregate", action="store_true",
                   help="classic schedule: stand-alone SpMM per layer instead of the aggregation fused into the transform")
    p.add_argument("--features", default="auto", choices=["auto", "packed", "table"],
                   help="layout of the input features: 'packed' = one row per pack row in pack order (what the reference's "
                        "collated batch.x holds, built once with the pack); 'table' = node-ordered [N, F] table gathered "
                        "through gid every step; auto = packed in mode none with one chunk per rank, else table")
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--collective", default="auto", choices=["auto", "none", "push", "p2p", "ce", "nccl"],
                   help="N>1: what happens to the logits after the head.  none = they stay sharded by rank (subgraphs are "
                        "independent: the path has no exchange step; the reference's metrics need an all-reduce of three scalars).  "
                        "push = head into the local slot, then ONE small kernel bulk-stores the slot to all "
                        "peers on a side stream, overlapping the next step's compute (measured slower: it takes SMs from the "
                        "persistent GEMMs); "
                        "p2p = head kernel stores into every rank's gather buffer over NVLink "
                        "(+ a one-element all-reduce as barrier); ce = head into the local slot, copy-engine pushes to the "
                        "peers on a side stream overlapping the next step's compute; nccl = local slot, then all_gather; "
                        "auto = p2p at 2 GPUs, push (with as many SMs left free by the GEMM grids) above (measured, "
                        "profiles/r2_multi_gpu.md); the variant not chosen (sharded / gathered) is timed "
                        "after the headline and reported in multi_gpu.sharded / multi_gpu.gathered")
    p.add_argument("--ce-peers", type=int, default=-1,
                   help="--collective push: peers (by rank distance) served by the copy engines instead of the push kernel; "
                        "-1 = measured default (0 up to 4 GPUs)")
    p.add_argument("--push-ctas", type=int, default=-1,
                   help="CTAs of the peer-push kernel (--collective push); -1 = 16 up to 4 GPUs, 24 at 8 (measured)")
    p.add_argument("--sm-reserve", type=int, default=-1,
                   help="SMs the persistent GEMM grids leave free (tuning 'sm_reserve'); -1 = the push kernel's CTA count with "
                        "--collective push, else 0")
    p.add_argument("--agg-wide", type=int, default=None, help="tuning 'agg_wide' (A/B of the fused-aggregation tile)")
    p.add_argument("--chunks", type=int, default=1, help="N>1: chunks per rank; chunk c's all-gather overlaps chunk c+1")
    p.add_argument("--modes", default="none_heavy_tail,cluster,train,per_query,alt_precision,coarsen",
                   help="N=1: extra blocks measured after the headline (comma separated, '' = none): none_heavy_tail = same "
                        "graph shape with power-law subgraph sizes (hybrid fused + classic schedule); cluster = the headline "
                        "graph with cluster_node augmentation (sharded pack, streamed forward); train = one GD training step "
                        "(forward + backward + Adam) on the headline pack; per_query = the reference's per-sample latency loop; "
                        "alt_precision = the headline configuration in the other arithmetics (bf16x3 and fp16x2 beside an fp16 headline); "
                        "coarsen = the coarsening algorithm itself on Cora- / PubMed-shaped graphs (device costs + host contraction) "
                        "with the oracle's CPU path and a partition-equality check beside it")
    p.add_argument("--only-modes", action="store_true", help="skip the headline measurement (profiling the --modes blocks)")
    p.add_argument("--mode-steps", type=int, default=0, help="timed steps of the --modes blocks (0 = min(--steps, 5))")
    p.add_argument("--max-rows", type=int, default=1 << 22, help="rows per shard of the streamed forward (--modes blocks)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write the last step's logits for a fixed sample of the nodes to DIR/logits.npy "
                        "(float32 [rows, C], node order) and their node ids to DIR/node_ids.npy (float64), for comparing builds")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "ours" or a.gpus != 1 or a.only_modes):
        p.error("--dump-outputs takes the headline of a single-GPU --impl ours run")
    return a


def workload_shape(name):
    if name == "products":
        return 2449029, 61859140, 100, 47
    return 200000, 5000000, 100, 47  # products-small: same generator, for quick checks


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled every 50 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.proc = index, [], False, None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()

    def mark(self):
        """index of the next sample (call at the start / end of the timed region)"""
        return len(self.rows)

    def summary(self, lo=0, hi=None):
        """samples [lo, hi) widened by one on each side (the 50 ms poll may straddle a short timed region)"""
        sm, smax, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        hi = len(self.rows) if hi is None else hi
        for r in self.rows[max(0, lo - 1): hi + 1]:
            try:
                sm.append(float(r[0])); smax = max(smax, float(r[1]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, "fallback"


DUMP_ROWS = 1 << 18  # nodes in --dump-outputs: 262,144 x (47 fp32 logits + an fp64 id) = 51 MB, under the 64 MB a dump may take


def dump_outputs(out_dir, logits, core_gid, n):
    """--dump-outputs: rows of `logits` ([n_core, C], pack order, core_gid[i] = node of row i) for a seeded sample of the n
    nodes (all of them when n <= DUMP_ROWS), in ascending node order.  Keyed by node id, so a build that orders the pack
    differently still compares row for row."""
    ids = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    row_of_node = torch.empty(n, dtype=torch.long, device=logits.device)
    row_of_node[core_gid.long()] = torch.arange(core_gid.numel(), device=logits.device)
    sample = logits[row_of_node[torch.from_numpy(ids).to(logits.device)]].float().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "logits.npy"), sample)
    np.save(os.path.join(out_dir, "node_ids.npy"), ids.astype(np.float64))


def generate(args, device):
    import fitgnn_b200 as fg
    n, e_und, F, C = workload_shape(args.workload)
    ei, part, cw, k = fg.synth.planted_partition(n, e_und, args.ratio, seed=args.seed, device=device)
    part = fg.synth.relabel_partition_reference_order(part)
    X = fg.synth.features(n, F, seed=args.seed, device=device)
    sd = fg.synth.init_state_dict(F, args.hidden, C, seed=args.seed)
    return n, F, C, ei, part, cw, k, X, sd


# ------------------------------------------------------------------------------------------------- CPU arm
def cpu_reference(args, ei, part, X, sd, k, seconds, steps=1, warmup=0):
    """The reference's batched CPU inference (node_infer_Gs_GD run.py:49-115: 128-subgraph block-diagonal batches,
    gcn_norm + F.linear + index_select/index_add per layer, lt1, log_softmax; timer around model() only) restated
    in oracle/fitgnn_oracle.py, on all host cores, over a bounded sample of consecutive subgraphs."""
    from oracle import fitgnn_oracle as fo
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ei_c, part_c, X_c = ei.cpu().numpy(), part.cpu().numpy(), X.cpu().numpy()
    sd_c = {k_: v.cpu() for k_, v in sd.items()}
    # calibrate on 8 batches, then size the sample for ~`seconds` of CPU work per step
    def prep(sub_ids):
        subs = fo.subgraphs_from_partition(ei_c, X_c, part_c, sub_ids)
        batches = [fo.collate(subs[b:b + 128]) for b in range(0, len(subs), 128)]
        return batches, sum(s["x"].shape[0] for s in subs)

    keep = {}

    def run(batches):
        t = 0.0
        outs = []
        with torch.no_grad():
            for x, e in batches:
                t0 = time.perf_counter()
                o = fo.classify_node(sd_c, x, e)
                t += time.perf_counter() - t0
                outs.append(o)
        keep["logits"] = outs
        return t

    cal, cal_nodes = prep(np.arange(0, min(k, 8 * 128)))
    run(cal[:2])
    t_cal = run(cal)
    n_batches = int(max(8, min(k // 128, seconds / max(t_cal / len(cal), 1e-6))))
    batches, nodes = prep(np.arange(0, min(k, n_batches * 128)))
    for _ in range(warmup):
        run(batches)
    times = [run(batches) for _ in range(max(1, steps))]
    t = float(np.median(times))
    base = dict(value=nodes / t, unit=UNIT, cores=cores, kind="port",
                sample=f"first {len(batches)} batches x 128 subgraphs ({nodes} nodes) of the same graph, "
                       f"torch {torch.__version__} CPU fp32 no_grad, median of {len(times)}")
    base["_logits"] = torch.cat(keep["logits"], 0)  # rows = the first `nodes` rows of the pack order (popped by the caller)
    return base, t, nodes


PARITY_RTOL = 1e-3  # north_star: logits within 1e-3 relative of the reference path


def parity_block(got, want, what):
    """GPU logits vs the CPU arm's logits of the same rows: max |diff| relative to max(1, max |want|) (the measure the
    parity tests use) and the element-wise bound |diff| <= rtol*|want| + 1e-2*rtol*max|want|.  Fails the run beyond 1e-3."""
    got = got.detach().double().cpu()
    want = want.detach().double().cpu()
    assert got.shape == want.shape, (tuple(got.shape), tuple(want.shape))
    scale = max(1.0, float(want.abs().max())) if want.numel() else 1.0
    err = (got - want).abs()
    ok = bool((err <= PARITY_RTOL * want.abs() + 1e-2 * PARITY_RTOL * scale).all())
    blk = {"against": what, "rows": int(want.shape[0]), "max_abs_err": float(err.max()) if want.numel() else 0.0,
           "max_rel_err": (float(err.max()) / scale) if want.numel() else 0.0, "rtol": PARITY_RTOL, "ok": ok}
    if not ok or blk["max_rel_err"] > PARITY_RTOL:
        raise SystemExit(f"bench: PARITY FAILURE {json.dumps(blk)}")
    return blk


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    device = "cuda" if torch.cuda.is_available() else "cpu"  # generation only; nothing timed runs on the GPU
    n, F, C, ei, part, cw, k, X, sd = generate(args, device)
    base, t, nodes = cpu_reference(args, ei, part, X, sd, k, args.cpu_seconds, steps=args.steps, warmup=min(args.warmup, 1))
    base.pop("_logits", None)
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_of(args, n, F, C, k), "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def config_of(args, n, F, C, k):
    return {"workload": f"{args.workload}: ogbn-products-shaped synthetic, {n} nodes, "
                        f"{workload_shape(args.workload)[1]} undirected edges, F={F}, C={C}, planted partition "
                        f"ratio {args.ratio} (k={k}), mode={args.mode}, 2-layer GCN hidden={args.hidden} + lt1 + log_softmax",
            "subgraphs": k, "mode": args.mode, "l2": "inputs larger than L2 (activations are GBs per layer)",
            "features": "pack-ordered rows" if features_packed(args) else "node-ordered table + gid"}


def features_packed(args, n_chunks=None):
    """Input layout of the timed forward (see --features): the reference's own layout (one x row per subgraph row, collated
    in subgraph order) unless asked otherwise / not applicable."""
    if n_chunks is None:
        n_chunks = 1 if args.gpus == 1 else args.chunks
    return args.features == "packed" or (args.features == "auto" and args.mode == "none" and n_chunks == 1)


# ------------------------------------------------------------------------------------------------- GPU arm
def _time_cuda(fn, reps=3, warm=1):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), r


def projection_bench(fg, ei, part, cw, k, X, n, F):
    """The coarsened-graph projection on the same graph (SURVEY §8 a9-a11): group nodes by cluster, Xc = C·X
    (fp64 accumulate), Ac = P·A·P^T pattern + counts.  Algorithmic bytes per SURVEY §8d."""
    hbm_peak, _, _ = measured_peaks()
    E = ei.shape[1]
    t_grp, (members, member_ptr) = _time_cuda(lambda: fg.ops.group_by_part(part, k))
    t_xc, Xc = _time_cuda(lambda: fg.ops.project_features(members, member_ptr, cw, X))
    b_xc = 4 * n * F + 4 * k * F + 12 * n + 4 * (k + 1)
    del Xc
    t_ac, (row, col, cnt, rowptr) = _time_cuda(lambda: fg.ops.project_adj(ei, part, k), reps=2)
    nnz_ac = int(row.numel())
    b_ac = 16 * E + 4 * n + 20 * nnz_ac
    del row, col, cnt, rowptr
    return {"group_by_part_ms": t_grp,
            "xc": {"kernel": "project_features_kernel", "ms": t_xc, "algo_GB": b_xc / 1e9, "GBps": b_xc / t_xc / 1e6,
                   "frac": b_xc / t_xc / 1e6 / hbm_peak, "bound": "hbm"},
            "ac": {"kernel": "adj_keys + radix sort + run-length (plan + fill, incl. 3 host syncs)", "ms": t_ac,
                   "algo_GB": b_ac / 1e9, "GBps": b_ac / t_ac / 1e6, "frac": b_ac / t_ac / 1e6 / hbm_peak,
                   "nnz_ac": nnz_ac, "directed_edges": E, "bound": "hbm (sort passes are not algorithmic bytes)"}}


def spmm_standalone_bench(fg, pack, H, traffic=None):
    """The H-wide segmented SpMM as its own launch on the same pack (the default schedule fuses this aggregation into
    the previous transform's epilogue, so it is timed here on its own): fp32 in, bf16 hi/lo planes out."""
    hbm_peak, _, _ = measured_peaks()
    Hm = torch.rand(pack.n_rows, H, device=pack.device)
    hubs = fg.ops.find_hubs(pack.rowptr, None, pack.n_rows)
    out = (torch.empty(pack.n_rows, H, dtype=torch.bfloat16, device=pack.device),
           torch.empty(pack.n_rows, H, dtype=torch.bfloat16, device=pack.device))
    t, _ = _time_cuda(lambda: fg.ops.spmm_symnorm(pack.rowptr, pack.col, pack.dinv, Hm, H, None, None, 0, None, out=out,
                                                  split=True, hubs=hubs), reps=5, warm=2)
    R = pack.n_rows
    b = 4 * (R + 1) + 4 * pack.nnz + 4 * R + 4 * R * H + 4 * R * H
    return {"kernel": "spmm_512_standalone", "bound": "hbm", "achieved": b / t / 1e6, "peak": hbm_peak, "unit": "GB/s",
            "frac": b / t / 1e6 / hbm_peak, "frac_of_nominal_8000": b / t / 1e6 / 8000.0, "traffic": traffic,
            "algorithmic_bytes": int(b), "ms": t, "peak_source": "measured (hbm_gbs)",
            "note": "stand-alone launch on the same pack; the default schedule fuses this aggregation into gemm0's epilogue"}


def _time_forward(fwd, Xp, out, steps, warmup, sampler):
    """W untimed + K timed forwards on the current stream (CUDA events), per-kernel events inside."""
    for _ in range(max(warmup, 3)):
        fwd(Xp, out=out)
    torch.cuda.synchronize()
    fwd.enable_profile(True)
    l0 = fwd.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    m0 = sampler.mark() if sampler else 0
    if PROFILER_RANGE:
        torch.cuda.cudart().cudaProfilerStart()
    e0.record()
    for _ in range(steps):
        fwd(Xp, out=out)
    e1.record()
    torch.cuda.synchronize()
    if PROFILER_RANGE:
        torch.cuda.cudart().cudaProfilerStop()
    m1 = sampler.mark() if sampler else 0
    ms = e0.elapsed_time(e1) / steps
    prof = fwd.profile_summary()
    fwd.enable_profile(False)
    return ms, prof, fwd.launches - l0, (sampler.summary(m0, m1) if sampler else None)


def _kernel_table(prof, steps):
    """per-step kernel times: profile_summary() holds the mean launch duration per part; a streamed forward launches every
    op once per part and step, so ms is already 'per step' after summing over the parts."""
    hbm_peak, _, _ = measured_peaks()
    tot = max(1e-9, sum(r["ms"] for r in prof.values()))
    out = {}
    for name, r in prof.items():
        out[name] = {"ms": r["ms"], "algo_GB": r["bytes"] / 1e9, "GBps": r["bytes"] / (r["ms"] * 1e-3) / 1e9,
                     "TFLOPs": (r["flops"] / (r["ms"] * 1e-3) / 1e12) if r["flops"] else 0.0, "share": r["ms"] / tot,
                     "launches_per_step": r["launches"] // max(1, steps)}
    return out


def _spmm_roofline(kernels, prefer=None):
    """The SpMM with the largest algorithmic traffic of a mode block (the one the block's time hinges on)."""
    hbm_peak, _, _ = measured_peaks()
    names = [k_ for k_ in kernels if "spmm" in k_]
    if not names:
        return None
    nm = prefer if prefer in kernels else max(names, key=lambda k_: kernels[k_]["algo_GB"])
    r = kernels[nm]
    return {"kernel": nm, "bound": "hbm", "achieved": r["GBps"], "peak": hbm_peak, "unit": "GB/s", "frac": r["GBps"] / hbm_peak,
            "frac_of_nominal_8000": r["GBps"] / 8000.0, "algorithmic_bytes": int(r["algo_GB"] * 1e9), "ms": r["ms"],
            "traffic": None, "peak_source": "measured (hbm_gbs)"}


def mode_none_heavy_tail(args, fg, device, n, e_und, F, C, sd, precision, steps, sampler):
    """Mode 'none' on the same graph shape with heavy-tailed subgraph sizes (power law, max 500: what real coarsenings look
    like, SURVEY §7): subgraphs <= 32 rows run the fused group-aligned schedule, the rest the classic SpMM + GEMM one."""
    from oracle import fitgnn_oracle as fo
    ei, part, cw, k = fg.synth.planted_partition(n, e_und, args.ratio, seed=args.seed + 1, device=device, sizes="powerlaw")
    part = fg.synth.relabel_partition_reference_order(part)
    X = fg.synth.features(n, F, seed=args.seed + 1, device=device)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    pack = fg.build_pack(ei, part, k, "none")
    torch.cuda.synchronize(); build_ms = (time.perf_counter() - t0) * 1e3
    sizes = torch.bincount(part.long(), minlength=k).float()
    fwd = fg.StreamedForward(pack, sd, precision=precision)
    Xp = fwd.table_features(X)
    out = torch.empty(fwd.n_out, (C + 3) // 4 * 4, device=device)
    ms, prof, launches, clocks = _time_forward(fwd, Xp, out, steps, args.warmup, sampler)
    kernels = _kernel_table(prof, steps)
    # parity: the first 64 x 128 subgraphs through the reference's batched CPU path
    n_sub = min(k, 64 * 128)
    subs = fo.subgraphs_from_partition(ei.cpu().numpy(), X.cpu().numpy(), part.cpu().numpy(), np.arange(n_sub))
    sel = [np.ones(s_["x"].shape[0], dtype=bool) for s_ in subs]
    want = fo.node_infer_batched({k_: v.cpu() for k_, v in sd.items()}, subs, sel, "node_cls", 128)
    blk = {"workload": f"products shape ({n} nodes, {e_und} undirected edges), power-law subgraph sizes (alpha 1.8, max 500), mode none",
           "ms_per_step": ms, "value": n / (ms * 1e-3), "unit": UNIT, "steps": steps, "subgraphs": k,
           "subgraph_rows": {"mean": float(sizes.mean()), "p99": float(torch.quantile(sizes[: 1 << 24], 0.99)), "max": int(sizes.max()),
                             "rows_in_subgraphs_over_32": float(sizes[sizes > 32].sum() / sizes.sum())},
           "schedule": {kind: int(sum(f.pack.n_rows for f, k_ in zip(fwd.parts, fwd.kinds) if k_ == kind)) for kind in set(fwd.kinds)},
           "pack": {"rows": pack.n_rows, "nnz": pack.nnz, "build_ms": build_ms},
           "hub_rows": int(sum(f.hubs_all[1] for f in fwd.parts)), "gpu_launches": launches, "kernels": kernels,
           "roofline_spmm": _spmm_roofline(kernels, "c_spmm1"), "clocks": clocks,
           "parity": parity_block(out[: want.shape[0], :C], want, f"oracle CPU path, first {n_sub} subgraphs")}
    return blk


def mode_cluster(args, fg, device, n, F, C, ei, part, cw, k, X, sd, precision, steps, sampler):
    """cluster_node augmentation (utils.py:190-233; the only ogbn-products row the reference ran, memory_usage.csv:42) on the
    headline graph: N + nnz(Ac) pack rows, built as shards of --max-rows rows and streamed through the classic schedule."""
    import scipy.sparse as sp_
    from oracle import fitgnn_oracle as fo
    torch.cuda.synchronize(); t0 = time.perf_counter()
    row, col, cnt, ac_rowptr = fg.ops.project_adj(ei, part, k)
    del cnt
    ac_col = col.to(torch.int32)
    members, member_ptr = fg.ops.group_by_part(part, k)
    Xc = fg.ops.project_features(members, member_ptr, cw, X)
    Xtab = torch.cat([X, Xc], 0)  # de-duplicated feature table: every node once + one C·X row per cluster
    del members, member_ptr
    torch.cuda.synchronize(); proj_ms = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter()
    stream = fg.build_pack_stream(ei, part, k, "cluster", max_rows=args.max_rows, ac_rowptr=ac_rowptr, ac_col=ac_col)
    torch.cuda.synchronize(); build_ms = (time.perf_counter() - t0) * 1e3
    fwd = fg.StreamedForward(stream, sd, precision=precision)
    Xp = fwd.table_features(Xtab)
    out = torch.empty(fwd.n_out, (C + 3) // 4 * 4, device=device)
    ms, prof, launches, clocks = _time_forward(fwd, Xp, out, steps, args.warmup, sampler)
    kernels = _kernel_table(prof, steps)
    # parity on the first 256 subgraphs: the oracle's subgraph builder needs the out-edges of their core nodes and the
    # rows of Ac of their adjacent clusters only, so it is handed exactly those (same subgraphs, seconds instead of minutes)
    n_sub = min(k, 256)
    part_l = part.long()
    src_in = part_l[ei[0]] < n_sub
    ei_s = ei[:, src_in].cpu().numpy()
    nb = torch.unique(part_l[ei[1][src_in]])
    in_nb = torch.zeros(k, dtype=torch.bool, device=device)
    in_nb[nb] = True
    keep = in_nb[row] & in_nb[col]
    adj = sp_.csr_matrix((np.ones(int(keep.sum()), dtype=bool), (row[keep].cpu().numpy(), col[keep].cpu().numpy())), shape=(k, k))
    co = dict(part=part_l.cpu().numpy(), CX=Xc.cpu().numpy(), adj=adj)
    subs = fo.build_subgraphs(ei_s, X.cpu().numpy(), np.zeros(n, dtype=np.int64), [np.arange(n)], [co], "cluster",
                              only=set(range(n_sub)))[:n_sub]
    sel = []
    for s_ in subs:
        m = np.zeros(s_["x"].shape[0], dtype=bool)
        m[: len(s_["core"])] = True
        sel.append(m)
    want = fo.node_infer_batched({k_: v.cpu() for k_, v in sd.items()}, subs, sel, "node_cls", 128)
    rows_per_sub = stream.n_rows / k
    blk = {"workload": f"headline graph, cluster_node augmentation (utils.py:190-233), {len(stream.packs)} shards of <= {args.max_rows} rows",
           "ms_per_step": ms, "value": n / (ms * 1e-3), "unit": UNIT, "steps": steps, "subgraphs": k,
           "pack": {"rows": stream.n_rows, "nnz": stream.nnz, "shards": len(stream.packs), "rows_per_subgraph": rows_per_sub,
                    "bytes": stream.nbytes(), "build_ms": build_ms, "projection_ms": proj_ms, "nnz_ac": int(row.numel())},
           "hub_rows": int(sum(f.hubs_all[1] for f in fwd.parts)), "gpu_launches": launches, "kernels": kernels,
           "roofline_spmm": _spmm_roofline(kernels), "roofline_spmm_last_layer": _spmm_roofline(kernels, "spmm1"), "clocks": clocks,
           "parity": parity_block(out[: want.shape[0], :C], want, f"oracle CPU path (reference subgraph builder), first {n_sub} subgraphs")}
    return blk


def mode_train(args, fg, device, n, F, C, ei, part, k, X, precision, steps, sampler):
    """One optimiser step of node_train_Gs_GD (run.py:177-215) on the headline pack: forward over ALL subgraphs in train mode
    (conv -> ELU -> Philox dropout fused), one loss over the train rows, backward on the tensor cores (dW = Gᵀ·A through
    fitgnn_gemm_tn, dX through the NT kernel, Âᵀ through the reversed CSR), one fused Adam kernel over the flat parameters."""
    import types
    pack = fg.build_pack(ei, part, k, "none")
    margs = types.SimpleNamespace(num_layers1=2, num_features=F, hidden=args.hidden, num_classes=C, layer_name="GCNConv")
    torch.manual_seed(args.seed)
    model = fg.Classify_node(margs).to(device)
    opt = fg.train.FusedAdam(model.parameters(), lr=0.01, weight_decay=0.0005)  # main.py:193-194 defaults
    g = torch.Generator(device=device).manual_seed(args.seed)
    y = torch.randint(0, C, (n,), generator=g, device=device)
    train_mask = torch.rand(n, generator=g, device=device) < 0.1
    csr = fg.train.pack_csr(pack)
    csr.transposed()
    losses = [fg.train.train_step_Gs(model, pack, X, y, train_mask, opt, csr=csr) for _ in range(2)]
    torch.cuda.synchronize()
    m0 = sampler.mark() if sampler else 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        losses.append(fg.train.train_step_Gs(model, pack, X, y, train_mask, opt, csr=csr))
    e1.record()
    torch.cuda.synchronize()
    m1 = sampler.mark() if sampler else 0
    ms = e0.elapsed_time(e1) / steps
    # the weight-gradient GEMM of the hidden layer on its own: dW[512, 512] = Gᵀ·A over all rows
    G = torch.randn(n, args.hidden, device=device)
    A = torch.randn(n, args.hidden, device=device)
    t_tn, _ = _time_cuda(lambda: fg.ops.gemm_tn(G, A), reps=3, warm=1)
    flops = 2.0 * n * args.hidden * args.hidden
    _, tc_peak, _ = measured_peaks()
    del G, A
    return {"workload": "headline pack, one GD training step (forward in train mode + loss over 10% train rows + backward + Adam)",
            "ms_per_step": ms, "value": n / (ms * 1e-3), "unit": "nodes/s per optimiser step", "steps": steps,
            "loss_first_last": [losses[0], losses[-1]], "precision": precision,
            "gemm_tn": {"shape": [n, args.hidden, args.hidden], "ms": t_tn, "logical_TFLOPs": flops / t_tn / 1e9,
                        "bf16_mma_TFLOPs": 3 * flops / t_tn / 1e9, "frac_of_bf16_peak": 3 * flops / t_tn / 1e9 / tc_peak,
                        "includes": "transposing bf16 hi/lo split of both operands + batched split-K tcgen05 GEMM + reduction"},
            "clocks": sampler.summary(m0, m1) if sampler else None}


def dtype_of(fwd):
    if not getattr(fwd, "f16_hidden", False):
        return "bf16x3(f32 accumulate)"
    if getattr(fwd, "f16_layer0", False):
        return ("fp16 planes for every operand of the two wide transforms (aggregated features, hidden state, weights: 1 MMA per "
                "product), fp16 hidden state x fp16 hi/lo weights (2 MMAs) in the head; f32 accumulate")
    if getattr(fwd, "w_single", False):
        return ("bf16x3 first layer; fp16 hidden state x ONE fp16 weight plane (1 MMA) in the 512 x 512 transforms, x fp16 hi/lo "
                "weights (2 MMAs) in the head; f32 accumulate")
    return "bf16x3 first layer; fp16 A x fp16 hi/lo W, 2 MMAs, f32 accumulate for the 512-wide layers"


def mode_precisions(args, fg, device, n, F, C, ei, part, k, X, sd, steps, sampler, precision):
    """alt_precision block: every other tensor-core arithmetic than the headline's, same configuration, same box."""
    others = [p_ for p_ in ("bf16x3", "fp16x2", "fp16") if p_ != precision]
    if precision == "fp32":
        others = ["bf16x3"]
    res = {}
    for which in others:
        res[which] = mode_precision(args, fg, device, n, F, C, ei, part, k, X, sd, steps, sampler, which)
        torch.cuda.empty_cache()
    first = res[others[0]]
    return {**first, "others": {w_: r_ for w_, r_ in res.items() if w_ != others[0]}}


def mode_precision(args, fg, device, n, F, C, ei, part, k, X, sd, steps, sampler, which):
    """The headline configuration in the OTHER arithmetic than the headline's: 'bf16x3' = bf16 hi/lo planes for both operands of
    every transform (3 MMAs per product, fp32-grade agreement with the reference path) or 'fp16x2' = bf16x3 first layer, then the
    hidden state as ONE fp16 plane (half its bytes, 2 MMAs per product, activations rounded to 11 bits) — what the choice buys
    and what it costs (parity), side by side with the headline."""
    from oracle import fitgnn_oracle as fo
    pack = fg.build_pack(ei, part, k, "none")
    fwd = fg.PackedForward(pack, sd, head="log_softmax", rows="core", precision=which, align_policy=args.align_policy)
    Xp = fwd.pack_features(X)
    out = torch.empty(fwd.n_out, (C + 3) // 4 * 4, device=device)
    for _ in range(max(args.warmup, 3)):
        fwd(Xp, out=out, packed=True)
    torch.cuda.synchronize()
    fwd.enable_profile(True)
    l0 = fwd.launches
    m0 = sampler.mark() if sampler else 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fwd(Xp, out=out, packed=True)
    e1.record()
    torch.cuda.synchronize()
    m1 = sampler.mark() if sampler else 0
    ms = e0.elapsed_time(e1) / steps
    kernels = _kernel_table(fwd.profile_summary(), steps)
    n_sub = min(k, 64 * 128)
    subs = fo.subgraphs_from_partition(ei.cpu().numpy(), X.cpu().numpy(), part.cpu().numpy(), np.arange(n_sub))
    sel = [np.ones(s_["x"].shape[0], dtype=bool) for s_ in subs]
    want = fo.node_infer_batched({k_: v.cpu() for k_, v in sd.items()}, subs, sel, "node_cls", 128)
    return {"workload": f"headline configuration with precision='{which}'",
            "ms_per_step": ms, "value": n / (ms * 1e-3), "unit": UNIT, "steps": steps, "gpu_launches": fwd.launches - l0,
            "dtype": dtype_of(fwd),
            "kernels": kernels, "clocks": sampler.summary(m0, m1) if sampler else None,
            "parity": parity_block(out[: want.shape[0], :C], want, f"oracle CPU path, first {n_sub} subgraphs")}


def mode_coarsen(args, fg, device):
    """The coarsening algorithm itself (SURVEY §8f rank 4; coarsening_utils.py:18-182, variation_neighborhoods) on Cora- and
    PubMed-shaped power-law graphs (BASELINE.json configs[0], [1]): spectral basis + batched candidate costs + level projections
    on the device, the sequential contraction on the host.  CPU arm and parity on the Cora-shaped graph: the oracle's
    restatement of the reference algorithm, fed the SAME spectral basis, must return the same partition.  Never raises: a
    failure is reported in the block instead of costing the bench line."""
    try:
        from fitgnn_b200 import coarsen_algo as ca
        out = {}
        for name, n, e_und, r in (("cora_shaped", 2708, 5278, 0.7), ("pubmed_shaped", 19717, 44324, 0.5)):
            ei = torch.tensor(fg.synth.powerlaw_graph(n, e_und, seed=0), device=device)
            lab = ca.connected_components(ei, n)
            roots, inv, sizes = torch.unique(lab, return_inverse=True, return_counts=True)
            big = int(torch.argmax(sizes))  # the giant component (the reference coarsens component by component)
            nodes = torch.nonzero(inv == big).view(-1)
            local = torch.full((n,), -1, dtype=torch.int64, device=device)
            local[nodes] = torch.arange(nodes.numel(), device=device)
            sel = inv[ei[0]] == big
            eic = torch.stack([local[ei[0][sel]], local[ei[1][sel]]])
            nc = int(nodes.numel())
            core = ca.variation_neighborhoods if device.type == "cuda" else ca._coarsen
            sync = torch.cuda.synchronize if device.type == "cuda" else (lambda: None)
            row, col, w, _ = ca._coalesce(eic[0], eic[1], torch.ones(eic.shape[1], dtype=torch.float64, device=device), nc)
            sync(); t0 = time.perf_counter()
            lk, Uk = ca.laplacian_subspace(row, col, w, nc, 10)
            sync(); t_basis = time.perf_counter() - t0
            core(eic, nc, r, 10, Uk, lk)  # warm-up
            sync(); t0 = time.perf_counter()
            res = core(eic, nc, r, 10, Uk, lk)
            sync(); t_algo = time.perf_counter() - t0
            blk = {"nodes": nc, "directed_edges": int(eic.shape[1]), "r": r, "supernodes": res.k, "levels": res.levels,
                   "basis_ms": t_basis * 1e3, "contraction_levels_ms": t_algo * 1e3,
                   "what": "basis = smallest-10 Laplacian eigenpairs on the device; contraction_levels = batched candidate costs + "
                           "level projections on the device and the sequential contraction on the host, all levels"}
            if name == "cora_shaped":
                from oracle import coarsen_oracle as co
                import scipy.sparse as sp
                W = sp.coo_matrix((np.ones(eic.shape[1]), (eic[0].cpu().numpy(), eic[1].cpu().numpy())), shape=(nc, nc)).tocsr()
                W.data[:] = 1.0
                t0 = time.perf_counter()
                Cm, _, lv = co.coarsen(W, Uk.cpu().numpy(), lk.cpu().numpy(), K=10, r=r)
                t_cpu = time.perf_counter() - t0
                blk["cpu_baseline"] = {"ms": t_cpu * 1e3, "kind": "port", "cores": 1,
                                       "what": "oracle restatement of coarsening_utils.coarsen (numpy, per-set dense costs), same basis"}
                blk["parity"] = {"partition_equal": bool(np.array_equal(Cm.indices, res.part.cpu().numpy())),
                                 "cweight_equal": bool(np.array_equal(Cm.data, res.cweight.cpu().numpy())), "levels_equal": lv == res.levels,
                                 "against": "oracle CPU path (pinned bit-exactly to the reference on tests/golden/coarsen_algo.npz), same (Uk, lk)"}
            if name == "pubmed_shaped":  # the edge family: closed-form costs of all edges + the greedy matching in parallel rounds
                core_e = ca.coarsen if device.type == "cuda" else ca._coarsen
                core_e(eic, nc, r, 10, Uk, lk, method="variation_edges")
                sync(); t0 = time.perf_counter()
                res_e = core_e(eic, nc, r, 10, Uk, lk, method="variation_edges")
                sync()
                blk["variation_edges"] = {"ms": (time.perf_counter() - t0) * 1e3, "supernodes": res_e.k, "levels": res_e.levels}
            out[name] = blk
        return out
    except Exception as e:  # noqa: BLE001 — this block must not cost the bench line
        return {"error": f"{type(e).__name__}: {e}"}


def mode_per_query(args, fg, device, n, F, C, ei, part, k, X, sd, precision, sampler):
    """The reference's own inference-time measurement (inference.py:672-688): ONE subgraph forward per queried node, timer
    around `model(x, edge_index)` only (the subgraph and its features are on the device before the timer starts), first sample
    dropped, mean of the rest.  Here: the queried node's subgraph as a one-subgraph pack prepared up front (as `graphs[i]` is),
    timed = the forward's launches — eagerly, and as a CUDA-graph replay — with a device synchronisation per query (the
    reference's timer has none, SURVEY §0.8); the CPU arm runs the oracle's per-query forward on the same queries."""
    from oracle import fitgnn_oracle as fo
    n_q = 64
    g = torch.Generator(device="cpu").manual_seed(args.seed)
    q_nodes = torch.randint(0, n, (n_q,), generator=g)
    pack = fg.build_pack(ei, part, k, "none")
    subs = part.long()[q_nodes.to(device)]
    fwds, xs, rows_of = [], [], []
    for s_ in subs.tolist():
        sp = fg.infer.select_subgraphs(pack, torch.tensor([s_], device=device))
        f = fg.PackedForward(sp, sd, head="log_softmax", rows="core", precision=precision, fuse_aggregate=False)
        fwds.append(f)
        xs.append(f.pad_features(X[sp.gid.long()].contiguous()))  # the subgraph's own x rows (graphs[i].x)
        rows_of.append(sp)
        # the one-subgraph pack reads its features directly: gid := identity
        import dataclasses
        f.pack = dataclasses.replace(sp, gid=torch.arange(sp.n_rows, dtype=torch.int32, device=device), n_src=sp.n_rows)
    def run(i):
        return fwds[i](xs[i])
    for i in range(n_q):
        run(i)
    torch.cuda.synchronize()
    t_eager = []
    for i in range(n_q):
        t0 = time.perf_counter(); out = run(i); torch.cuda.synchronize(); t_eager.append(time.perf_counter() - t0)
    graphs = [fwds[i].capture(xs[i]) for i in range(n_q)]
    torch.cuda.synchronize()
    t_graph = []
    for i in range(n_q):
        t0 = time.perf_counter(); graphs[i].graph.replay(); torch.cuda.synchronize(); t_graph.append(time.perf_counter() - t0)
    # CPU arm + parity on the same queries
    ei_c, part_c, X_c = ei.cpu().numpy(), part.cpu().numpy(), X.cpu().numpy()
    sub_list = fo.subgraphs_from_partition(ei_c, X_c, part_c, subs.cpu().numpy())
    sd_c = {k_: v.cpu() for k_, v in sd.items()}
    t_cpu, worst = [], 0.0
    torch.set_num_threads(os.cpu_count() or 1)
    for i, sg in enumerate(sub_list):
        x_, e_ = torch.as_tensor(sg["x"]), torch.as_tensor(sg["edge_index"])
        t0 = time.perf_counter()
        with torch.no_grad():
            want = fo.classify_node(sd_c, x_, e_)
        t_cpu.append(time.perf_counter() - t0)
        got = graphs[i].static_out[:, :C].cpu()
        worst = max(worst, float((got - want).abs().max() / max(1.0, float(want.abs().max()))))
    if worst > PARITY_RTOL:
        raise SystemExit(f"bench: PARITY FAILURE per_query max_rel_err {worst}")
    rows = [int(p_.n_rows) for p_ in rows_of]
    return {"workload": f"{n_q} random query nodes, one subgraph forward each (inference.py:672-688), mode none",
            "queries": n_q, "subgraph_rows_mean": float(np.mean(rows)), "subgraph_rows_max": int(max(rows)),
            "latency_us_eager_mean": float(np.mean(t_eager[1:]) * 1e6), "latency_us_graph_replay_mean": float(np.mean(t_graph[1:]) * 1e6),
            "launches_per_query": 5, "cpu_latency_us_mean": float(np.mean(t_cpu[1:]) * 1e6), "cpu_cores": os.cpu_count(),
            "timer": "perf_counter around the forward incl. a device synchronise; first query dropped (inference.py:688)",
            "parity": {"max_rel_err": worst, "rtol": PARITY_RTOL, "ok": True, "against": "oracle per-query forward, same queries"}}


def main_ours(args):
    import torch.distributed as dist

    import fitgnn_b200 as fg
    from fitgnn_b200.dist import ShardedPack

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    from fitgnn_b200._lib import set_tuning
    if args.push_ctas <= 0:
        args.push_ctas = 16 if world <= 4 else 24
    if args.ce_peers < 0:
        args.ce_peers = 0
    args.ce_peers = min(args.ce_peers, max(0, world - 2))
    uses_push = world > 1 and (args.collective == "push" or (args.collective in ("auto", "none") and world > 2))
    sm_reserve = args.sm_reserve if args.sm_reserve >= 0 else (args.push_ctas if uses_push else 0)

    def apply_reserve(coll):
        """the persistent GEMM grids leave SMs free only while the push kernel runs beside them"""
        set_tuning("sm_reserve", sm_reserve if (coll == "push" or args.sm_reserve >= 0) else 0)
    if args.agg_wide is not None:
        set_tuning("agg_wide", args.agg_wide)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    n, F, C, ei, part, cw, k, X, sd = generate(args, device)
    if args.only_modes:  # profiling entry: just the --modes blocks, printed as the JSON line
        assert world == 1, "--only-modes is a single-GPU run"
        precision = args.precision if args.precision != "auto" else os.environ.get("FITGNN_PRECISION", "fp16")
        k_steps = args.mode_steps or min(args.steps, 5)
        res = {}
        for m in [m_ for m_ in args.modes.split(",") if m_]:
            if m == "none_heavy_tail":
                res[m] = mode_none_heavy_tail(args, fg, device, n, workload_shape(args.workload)[1], F, C, sd, precision, k_steps, None)
            elif m == "train":
                res[m] = mode_train(args, fg, device, n, F, C, ei, part, k, X, precision, k_steps, None)
            elif m == "per_query":
                res[m] = mode_per_query(args, fg, device, n, F, C, ei, part, k, X, sd, precision, None)
            elif m == "alt_precision":
                res[m] = mode_precisions(args, fg, device, n, F, C, ei, part, k, X, sd, k_steps, None, precision)
            elif m == "coarsen":
                res[m] = mode_coarsen(args, fg, device)
            else:
                res[m] = mode_cluster(args, fg, device, n, F, C, ei, part, cw, k, X, sd, precision, k_steps, None)
            torch.cuda.empty_cache()
        print(json.dumps({"modes": res}))
        return
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pack = fg.build_pack(ei, part, k, args.mode)
    torch.cuda.synchronize()
    pack_build_first_ms = (time.perf_counter() - t0) * 1e3  # incl. first-use kernel loading + workspace cudaMallocs
    del pack
    t0 = time.perf_counter()
    pack = fg.build_pack(ei, part, k, args.mode)
    torch.cuda.synchronize()
    pack_build_ms = (time.perf_counter() - t0) * 1e3
    ei_keep = ei if (rank == 0 and world == 1 and not (args.no_cpu_baseline and args.no_projection and not args.modes)) else None
    del ei
    if args.mode == "cluster":
        raise SystemExit("bench: the headline is mode none/extra; cluster_node runs as a block: --modes cluster [--only-modes]")
    n_chunks = 1 if world == 1 else args.chunks
    shard = ShardedPack(pack, world, rank, args.hidden, F, n_chunks=n_chunks, local_table=world > 1)
    precision = args.precision
    if precision == "auto":
        precision = os.environ.get("FITGNN_PRECISION", "fp16")
    fwds = [fg.PackedForward(lp, sd, head="log_softmax", rows="core", precision=precision,
                             fuse_aggregate=False if args.no_fuse_aggregate else "auto", align_policy=args.align_policy)
            for lp in shard.locals]
    fwd = fwds[0]
    align_ms = None
    if fwd.apack is not None and world == 1:  # the group alignment the fused schedule needs (done once per pack, timed on its own)
        torch.cuda.synchronize(); t0 = time.perf_counter()
        _ap = pack.aligned(32, args.align_policy)
        torch.cuda.synchronize(); align_ms = (time.perf_counter() - t0) * 1e3
        del _ap
    # the group-aligned schedule takes the feature table un-padded ([n, 100]); the classic one wants the K-padded pitch
    Xd = X if (fwd.apack is not None and F % 4 == 0) else fwd.pad_features(X)
    X_full = Xd
    if shard.table_ids is not None:  # N > 1: this rank's rows of the feature table only (its own nodes in mode none)
        Xd = Xd[shard.table_ids].contiguous()

    # pack-ordered features: the reference's models receive one copy of x per subgraph row, collated in subgraph order
    # (utils.py:248, run.py:336); the layout is produced once, with the pack (mode none: N rows either way, the same bytes)
    packed = features_packed(args, len(fwds))
    if packed and len(fwds) != 1:
        raise SystemExit("bench: --features packed needs --chunks 1")
    X_table = Xd
    if packed:
        Xd = fwd.pack_features(X_table)
    Cp = (C + 3) // 4 * 4  # logits row pitch padded to 16 bytes (aligned stores in the head kernel); columns >= C unused
    gbuf = shard.gather_buffer(Cp, device) if world > 1 else None

    # fused output exchange (see dist.PeerGather): needs the group-aligned schedule (row-mapped head stores)
    pg, coll_gather = None, "nccl" if world > 1 else "none"
    want_coll = args.collective
    gather_pref = args.collective if args.collective not in ("auto", "none") else ("p2p" if world <= 2 else "push")
    if world > 1 and gather_pref != "nccl" and all(f.apack is not None for f in fwds):
        try:
            from fitgnn_b200.dist import PeerGather
            pg = PeerGather(shard, Cp, device, n_buffers=2, backend="ipc")
            # measured (profiles/r1_multi_gpu.md, profiles/r2_multi_gpu.md): the fused peer stores win at 2 GPUs; from 4 on the head
            # becomes NVLink-egress-bound and an exchange overlapped with the next step is ahead: copy engines reach ~310 GB/s
            # in the all-to-all pattern, the SM-driven push kernel ~45 GB/s per CTA up to ~490 GB/s — provided the persistent GEMM
            # grids leave its SMs free (tuning sm_reserve), otherwise every CTA it occupies delays one GEMM CTA by the whole push;
            # the multicast store does not help an all-gather (every rank still has to RECEIVE all the other slots)
            coll_gather = gather_pref
        except Exception as e:  # IPC not permitted in this container, ...
            if args.collective == "p2p":
                raise
            print(f"bench: peer buffers unavailable ({e}); using the NCCL all-gather", file=sys.stderr)
    if world > 1:  # every rank must take the same path
        ok = torch.tensor([1 if pg is not None else 0], device=device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            pg, coll_gather = None, "nccl"
    # the headline ends every step with ALL logits on every rank (north_star: "the final logit all-gather");
    # --collective none leaves them sharded.  The other variant is timed after the headline and reported beside it.
    collective = "none" if (world == 1 or want_coll == "none") else coll_gather
    apply_reserve(collective)

    def run_local(Xin, buf):
        """outputs stay sharded: every chunk's head writes this rank's slot of `buf` (same layout as the gathered variants)"""
        for c, f in enumerate(fwds):
            f(Xin, out=shard.slot(buf, c), packed=packed)
        return buf

    def run_p2p(Xin, b, coll):
        if coll in ("ce", "push"):
            pg.acquire(b)
            for c, f in enumerate(fwds):
                f(Xin, out=shard.slot(pg.tensors[b], c), packed=packed)
            # completes behind the next step; the timed region ends with pg.wait on both buffers
            pg.exchange_async(b, engine=coll, push_ctas=args.push_ctas, ce_peers=args.ce_peers if coll == "push" else 0)
            return pg.tensors[b]
        for c, f in enumerate(fwds):
            f(Xin, peer_ptrs=pg.slot_ptrs(b, c), packed=packed)
        pg.barrier()
        return pg.tensors[b]

    def drain(coll=None):
        coll = collective if coll is None else coll
        if pg is not None and coll in ("ce", "push"):
            for b in range(2):
                pg.wait(b)

    step_no = [0]

    def run_chunks(Xin, buf):
        """forward of every local chunk; chunk c's all-gather is enqueued asynchronously (NCCL stream) right after its
        head kernel, so it overlaps the compute of chunk c+1; the current stream then waits for all of them."""
        works = []
        for c, f in enumerate(fwds):
            f(Xin, out=shard.slot(buf, c), packed=packed)  # the head kernel writes straight into this rank's slot
            works.append(shard.all_gather_(buf, c, async_op=True))
        for w in works:
            w.wait()
        return buf

    def step(coll=None):
        coll = collective if coll is None else coll
        if world == 1:
            return fwd(Xd, packed=packed)
        if coll == "none":
            return run_local(Xd, gbuf)
        if pg is not None and coll != "nccl":
            step_no[0] += 1
            return run_p2p(Xd, step_no[0] % 2, coll)
        return run_chunks(Xd, gbuf)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # nvidia-smi takes a few hundred ms to initialise NVML and can stall kernel launches while it does: start it before
    # the warm-up and wait for its first sample, so that only its steady 200 ms polling overlaps the timed region
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        out = step()  # same allocation pattern as the timed loop (the previous step's output stays alive)
    barrier()
    if rank == 0:
        t_wait = time.time()
        while not sampler.rows and time.time() - t_wait < 10.0:
            time.sleep(0.05)
    for f in fwds:
        f.enable_profile(True)
    launches0 = sum(f.launches for f in fwds)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if args.profiler_range:
        torch.cuda.cudart().cudaProfilerStart()
    mark0 = sampler.mark()
    ev0.record()
    dbg = os.environ.get("FITGNN_BENCH_DEBUG") == "1"
    step_ev, step_cpu = [], []
    for _ in range(args.steps):
        if dbg:
            step_cpu.append(time.perf_counter())
        out = step()
        if dbg:
            e_ = torch.cuda.Event(enable_timing=True)
            e_.record()
            step_ev.append(e_)
    drain()  # pipelined exchange: every step's outputs are complete on every rank before the clock stops
    ev1.record()
    barrier()
    mark1 = sampler.mark()
    if args.profiler_range:
        torch.cuda.cudart().cudaProfilerStop()
    ms = ev0.elapsed_time(ev1) / args.steps
    if dbg and rank == 0:
        ends = [ev0.elapsed_time(e_) for e_ in step_ev]
        print("debug: step end times on the GPU (ms since start):", [round(x, 2) for x in ends], file=sys.stderr)
        print("debug: step enqueue start times on the CPU (ms):", [round((c - step_cpu[0]) * 1e3, 2) for c in step_cpu],
              file=sys.stderr)
    gpu_launches = sum(f.launches for f in fwds) - launches0
    prof = {}
    for f in fwds:  # per-kernel time summed over this rank's chunks (ms per step)
        for name, r in f.profile_summary().items():
            agg = prof.setdefault(name, dict(ms=0.0, launches=0, bytes=0, flops=0))
            agg["ms"] += r["ms"]; agg["launches"] += r["launches"]; agg["bytes"] += r["bytes"]; agg["flops"] += r["flops"]
        f.enable_profile(False)
    rank_kernel_ms = None
    if world > 1:
        fwd_ms = torch.tensor([sum(v["ms"] for v in prof.values())], device=device, dtype=torch.float64)
        all_fwd = [torch.zeros_like(fwd_ms) for _ in range(world)]
        dist.all_gather(all_fwd, fwd_ms)
        rank_kernel_ms = [float(x.item()) for x in all_fwd]
    t = torch.tensor([ms], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    if args.dump_outputs:  # single GPU (parse): `out` is the last timed step's [n, C] logits in pack order
        dump_outputs(args.dump_outputs, out, pack.core_gid, n)

    # ---- N > 1: the result equals a single-GPU forward of the whole pack on EVERY rank (outside the timing).  Sharded
    # outputs are all-gathered once here for the check; the gathered variants are checked as they come out of a step.
    verify, other_info = None, None
    if world > 1:
        ref_rows = fg.PackedForward(pack, sd, head="log_softmax", rows="core", precision=precision,
                                    fuse_aggregate=False if args.no_fuse_aggregate else "auto",
                                    align_policy=args.align_policy)(X_full)
        full = torch.empty(n, C, device=device)
        full[pack.core_gid.long()] = ref_rows[:, :C]
        del ref_rows

        def check(res):
            gathered = res.view(-1, Cp)[shard.node_index(device)][:, :C]
            err = (gathered - full).abs().max().reshape(1)
            dist.all_reduce(err, op=dist.ReduceOp.MAX)
            return float(err.item())

        res = step()
        drain()
        barrier()
        if collective == "none":
            for c in range(n_chunks):
                shard.all_gather_(res, c, async_op=False)
            barrier()
        verify = check(res)
        del res
        # the other variant (headline gathered -> sharded outputs, headline sharded -> all-gathered), same steps / warm-up / clock
        other = coll_gather if collective == "none" else "none"
        apply_reserve(other)
        for _ in range(max(args.warmup, 3)):
            out = step(other)
        drain(other)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(args.steps):
            out = step(other)
        drain(other)
        g1.record()
        barrier()
        tg = torch.tensor([g0.elapsed_time(g1) / args.steps], device=device, dtype=torch.float64)
        dist.all_reduce(tg, op=dist.ReduceOp.MAX)
        if other == "none":
            for c in range(n_chunks):
                shard.all_gather_(out, c, async_op=False)
            barrier()
        g_err = check(out)
        other_info = {"collective": other, "ms_per_step": float(tg.item()), "value": n / (float(tg.item()) * 1e-3),
                      "unit": UNIT, "all_gather_bytes": int(n * Cp * 4) if other != "none" else 0,
                      "vs_single_gpu_max_abs_err_all_ranks": g_err}
        del full
        apply_reserve(collective)
        barrier()

    # ---- N = 1: the pack-ordered input gives the same logits, bit for bit, as the node-ordered table gathered through gid
    packed_check = None
    if world == 1 and packed:
        a_ = fwd(Xd, packed=True).clone()
        b_ = fwd(X_table)
        t_tab, _ = _time_cuda(lambda: fwd(X_table), reps=3, warm=1)
        packed_check = {"packed_vs_table_max_abs_err": float((a_ - b_).abs().max().item()),
                        "forward_ms_table_features": t_tab}
        del a_, b_

    # ---- end to end through the public API with HOST buffers: every step copies X from pinned host memory to the
    # device, runs the forward (+ all-gather) and copies this rank's logits back to pinned host memory.  Steps are
    # software-pipelined over three streams with double buffers (H2D of step i+1 and D2H of step i-1 overlap the
    # compute of step i); the timed region covers all copies of all K steps.
    e2e = None
    o_dev = None
    if not args.no_e2e:
        # one contiguous DMA per step.  N > 1: every rank copies only the feature rows its own subgraphs reference
        # (ShardedPack(local_table=True)): nothing about X is exchanged between the ranks.
        Fp = Xd.shape[1]
        X_host = Xd.cpu().pin_memory()  # N > 1: the rank's own rows of the feature table (shard.table_ids)
        n_loc = sum(f.n_out for f in fwds)
        NB = 2
        X_in = [torch.zeros_like(Xd) for _ in range(NB)]
        o_dev = None
        if pg is not None:
            o_dev = pg.tensors
        else:
            o_dev = [shard.gather_buffer(Cp, device) if world > 1 else torch.empty(n_loc, Cp, device=device) for _ in range(NB)]
        o_host = [torch.empty(n_loc, Cp, dtype=torch.float32).pin_memory() for _ in range(NB)]
        s_in, s_cmp, s_out = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
        ev_in = [torch.cuda.Event() for _ in range(NB)]
        ev_cmp = [torch.cuda.Event() for _ in range(NB)]
        ev_out = [torch.cuda.Event() for _ in range(NB)]

        def e2e_run(k_steps):
            for i in range(k_steps):
                b = i % NB
                with torch.cuda.stream(s_in):
                    s_in.wait_event(ev_cmp[b])  # the compute that last read X_in[b] is done
                    X_in[b].copy_(X_host, non_blocking=True)
                    ev_in[b].record(s_in)
                with torch.cuda.stream(s_cmp):
                    s_cmp.wait_event(ev_in[b])
                    s_cmp.wait_event(ev_out[b])  # the D2H that last read o_dev[b] is done
                    if world > 1 and collective == "none":
                        run_local(X_in[b], o_dev[b])
                    elif pg is not None and collective != "nccl":
                        run_p2p(X_in[b], b, collective)
                    elif world > 1:
                        run_chunks(X_in[b], o_dev[b])
                    else:
                        fwd(X_in[b], out=o_dev[b], packed=packed)
                    ev_cmp[b].record(s_cmp)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_cmp[b])
                    if world > 1:  # this rank's own slice of the logits, chunk by chunk
                        off = 0
                        for c in range(n_chunks):
                            sl = shard.slot(o_dev[b], c)
                            o_host[b][off: off + sl.shape[0]].copy_(sl, non_blocking=True)
                            off += sl.shape[0]
                    else:
                        o_host[b].copy_(o_dev[b], non_blocking=True)
                    ev_out[b].record(s_out)

        e2e_run(2)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s_in)
        e2e_run(args.steps)
        s_out.wait_stream(s_cmp)
        s_out.wait_stream(s_in)
        with torch.cuda.stream(s_out):
            drain()
        e1.record(s_out)
        barrier()
        t2 = torch.tensor([e0.elapsed_time(e1) / args.steps], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        h2d = torch.tensor([X_host.numel() * 4], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(h2d)
        # the host -> device link alone, every rank copying at once (no compute, no D2H): what the e2e step is bound by.  At N = 1
        # this is the PCIe link (~55 GB/s); at N > 1 the ranks share the host's memory system and PCIe switches, and the
        # per-rank figure shows how far below its own link each of them falls
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(s_in):
            c0.record(s_in)
            for _ in range(4):
                X_in[0].copy_(X_host, non_blocking=True)
            c1.record(s_in)
        barrier()
        t_copy = torch.tensor([c0.elapsed_time(c1) / 4], device=device, dtype=torch.float64)
        my_bytes = float(X_host.numel() * 4)
        copy_gbps = torch.tensor([my_bytes / (float(t_copy.item()) * 1e-3) / 1e9], device=device, dtype=torch.float64)
        copy_min = copy_gbps.clone()
        if world > 1:
            dist.all_reduce(t_copy, op=dist.ReduceOp.MAX)
            dist.all_reduce(copy_gbps)  # sum = aggregate
            dist.all_reduce(copy_min, op=dist.ReduceOp.MIN)
        e2e = {"value": n / (float(t2.item()) * 1e-3), "unit": UNIT, "ms_per_step": float(t2.item()),
               "h2d_bytes_per_step": int(h2d.item()), "d2h_bytes_per_step": int(n * Cp * 4),
               "h2d_GBps_per_rank_in_step": float(h2d.item()) / world / (float(t2.item()) * 1e-3) / 1e9,
               "h2d_alone": {"ms": float(t_copy.item()), "GBps_aggregate": float(copy_gbps.item()),
                             "GBps_slowest_rank": float(copy_min.item()),
                             "note": "the H2D copy of the step's features alone, all ranks at once (pinned memory, one DMA per rank): "
                                     "the floor of the e2e step"},
               "pipelining": "3 streams, double-buffered; every rank copies in the feature rows its own subgraphs reference "
                             "(the whole table at N = 1) over its own PCIe link and copies its own slice of the logits out"}
    if rank == 0:
        sampler.stop()

    if pg is not None:  # nobody may still be writing into a buffer that is about to be unmapped / freed
        barrier()
        o_dev = out = None
        pg.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    hbm_peak, tc_peak, peak_src = measured_peaks()
    kernels = {}
    for name, r in prof.items():
        gbs = r["bytes"] / (r["ms"] * 1e-3) / 1e9
        tfs = r["flops"] / (r["ms"] * 1e-3) / 1e12 if r["flops"] else 0.0
        kernels[name] = {"ms": r["ms"], "algo_GB": r["bytes"] / 1e9, "GBps": gbs, "TFLOPs": tfs,
                         "share": r["ms"] / max(1e-9, sum(x["ms"] for x in prof.values()))}

    dom = max(kernels, key=lambda k_: kernels[k_]["ms"])

    traffic = {}
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath) and world == 1 and args.workload == "products" and args.mode == "none":
        traffic = json.load(open(tpath))
        if getattr(fwd, "f16_hidden", False):  # per-launch DRAM bytes from the committed ncu capture of this same command
            traffic = traffic.get("_fp16" if getattr(fwd, "w_single", False) else "_fp16x2", {})

    f16_hidden = bool(getattr(fwd, "f16_hidden", False))

    def roofline_of(name):
        r = kernels[name]
        # MMAs per logical product: bf16x3 = 3 (hi*hi + lo*hi + hi*lo); fp16 hidden state = 2 (A*W_hi + A*W_lo) for every
        # transform whose A operand is the fp16 plane (all but the first)
        mmas = 2 if (f16_hidden and name not in ("gemm0_agg", "gemm0")) else 3
        if f16_hidden and getattr(fwd, "w_single", False) and name.startswith(("gemm", "conv")) and name not in ("gemm0_agg", "gemm0"):
            mmas = 1  # precision 'fp16': ONE fp16 weight plane in the hidden -> hidden transforms
        if getattr(fwd, "f16_layer0", False) and name in ("gemm0_agg", "gemm0"):
            mmas = 1  # the first transform on fp16 planes as well
        tensor_bound = (name.startswith(("gemm", "conv")) or name == "head") and precision != "fp32" and \
            mmas * r["TFLOPs"] / tc_peak > r["GBps"] / hbm_peak
        if tensor_bound:
            ach = mmas * r["TFLOPs"]
            return {"kernel": name, "bound": "tensor", "achieved": ach, "peak": tc_peak, "unit": "TFLOP/s",
                    "frac": ach / tc_peak, "traffic": traffic.get(name), "algorithmic_bytes": int(r["algo_GB"] * 1e9),
                    "peak_source": peak_src + f" (bf16_tflops_sustained; {mmas} 16-bit MMAs per logical product)"}
        return {"kernel": name, "bound": "hbm", "achieved": r["GBps"], "peak": hbm_peak, "unit": "GB/s",
                "frac": r["GBps"] / hbm_peak, "frac_of_nominal_8000": r["GBps"] / 8000.0, "traffic": traffic.get(name),
                "algorithmic_bytes": int(r["algo_GB"] * 1e9), "peak_source": peak_src + " (hbm_gbs)"}

    spmm_names = [k_ for k_ in kernels if k_.startswith("spmm")]
    spmm_main = max(spmm_names, key=lambda k_: kernels[k_]["algo_GB"]) if spmm_names else dom
    fused = fwd.apack is not None
    # one-time Gc projection kernels on the same graph, timed after (and outside of) the hot-path measurement
    projection = projection_bench(fg, ei_keep, part, cw, k, X, n, F) if (world == 1 and not args.no_projection) else None
    spmm_roof = spmm_standalone_bench(fg, shard.locals[0], args.hidden, traffic.get("spmm_512_standalone")) \
        if (fused and world == 1) else roofline_of(spmm_main)
    line = {"metric": METRIC, "value": n / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None,
            "dtype": "f32" if precision == "fp32" else dtype_of(fwd), "data": "synthetic",
            "config": config_of(args, n, F, C, k), "roofline": roofline_of(dom), "roofline_spmm": spmm_roof,
            "schedule": (("spmm0 -> transform -> [GCNConv in one kernel: transform + aggregation on the accumulators + bias + ELU] -> "
                          "head" if getattr(fwd, "conv_fused", False) else
                          "spmm0 -> [transform + next layer's aggregation in the epilogue] -> transform -> head") +
                         f" (group-aligned pack, {fwd.apack.n_rows} rows incl. padding)") if fused else "spmm + transform per layer -> head",
            "kernels": kernels, "gpu_launches": gpu_launches, "clocks": sampler.summary(mark0, mark1),
            "pack": {"rows": pack.n_rows, "nnz": pack.nnz, "subgraphs": pack.n_sub, "build_ms": pack_build_ms, "build_first_call_ms": pack_build_first_ms, "align_ms": align_ms,
                     "bytes": pack.nbytes(), "rank_loads": shard.loads},
            "multi_gpu": {"chunks_per_rank": n_chunks, "collective": collective, "sm_reserve": sm_reserve,
                          "push_ctas": args.push_ctas if "push" in (collective, coll_gather) else None,
                          "ce_peers": args.ce_peers if "push" in (collective, coll_gather) else None,
                          "outputs": ("sharded by rank (independent subgraphs: no exchange on the path); multi_gpu.gathered times "
                                      "the all-gathered variant") if (world > 1 and collective == "none") else
                                     ("all-gathered on every rank every step; multi_gpu.sharded times the same steps with the "
                                      "logits left on the rank that computed them" if world > 1 else "single GPU"),
                          "gathered_vs_single_gpu_max_abs_err_all_ranks": verify, "rank_kernel_ms": rank_kernel_ms,
                          "all_gather_bytes": int(n * Cp * 4) if (world > 1 and collective != "none") else 0,
                          "exposed_ms": (ms - max(rank_kernel_ms)) if rank_kernel_ms else 0.0,
                          ("gathered" if collective == "none" else "sharded"): other_info}}
    if packed_check:
        line["features_check"] = packed_check
    if projection:
        line["projection"] = projection
    if e2e:
        line["e2e"] = e2e
    if world == 1 and not args.no_cpu_baseline:
        base, _, _ = cpu_reference(args, ei_keep, part, X, sd, k, args.cpu_seconds)
        want = base.pop("_logits")
        line["cpu_baseline"] = base
        # the headline run against the reference path: GPU logits of the rows the CPU arm computed (pack order = batch order)
        got = fwd(Xd, packed=packed)
        line["parity"] = parity_block(got[: want.shape[0], :C], want, "cpu_baseline logits (oracle port of run.py:49-115), same rows")
        del got, want
    modes = [m for m in args.modes.split(",") if m] if world == 1 else []
    if modes:
        # free the headline's buffers first: the cluster_node pack alone is ~15 GB, its activations ~10 GB per shard
        fwds = fwd = shard = Xd = X_table = X_full = out = o_dev = gbuf = None
        if e2e:
            del X_in, X_host, o_host
        pack = None
        torch.cuda.empty_cache()
        k_steps = args.mode_steps or min(args.steps, 5)
        sampler2 = ClockSampler(local_rank)
        sampler2.start()
        t_wait = time.time()
        while not sampler2.rows and time.time() - t_wait < 10.0:
            time.sleep(0.05)
        line["modes"] = {}
        for m in modes:
            if m == "none_heavy_tail":
                line["modes"][m] = mode_none_heavy_tail(args, fg, device, n, workload_shape(args.workload)[1], F, C, sd, precision,
                                                        k_steps, sampler2)
            elif m == "cluster":
                line["modes"][m] = mode_cluster(args, fg, device, n, F, C, ei_keep, part, cw, k, X, sd, precision, k_steps, sampler2)
            elif m == "train":
                line["modes"][m] = mode_train(args, fg, device, n, F, C, ei_keep, part, k, X, precision, k_steps, sampler2)
            elif m == "per_query":
                line["modes"][m] = mode_per_query(args, fg, device, n, F, C, ei_keep, part, k, X, sd, precision, sampler2)
            elif m == "alt_precision":
                line["modes"][m] = mode_precisions(args, fg, device, n, F, C, ei_keep, part, k, X, sd, k_steps, sampler2, precision)
            elif m == "coarsen":
                line["modes"][m] = mode_coarsen(args, fg, device)
            else:
                raise SystemExit(f"bench: unknown --modes entry {m!r}")
            torch.cuda.empty_cache()
        sampler2.stop()
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    PROFILER_RANGE = a.profiler_range and a.only_modes
    if a.impl == "reference":
        main_reference(a)
    else:
        main_ours(a)
