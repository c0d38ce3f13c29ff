"""SAGEConv on the products-shaped workload of bench.py: ogbn-products-shaped synthetic graph (planted partition, ratio 0.5,
mode 'none'), F = 100, hidden 512, C = 47, a 2-layer SAGE model (seeded weights with PyG's keys) + lt1 + log_softmax,
run over the whole pack by PackedForward.  Prints one JSON line:

  * step_ms: forward time per step (CUDA events around `--steps` forwards after `--warmup` untimed ones);
  * kernels: per launch CUDA-event time, algorithmic bytes / FLOPs, and the share of the least time the hardware could
    take — max(bytes / 7.7 TB/s, tensor work / 2,250 TFLOP/s), the HGX B200 data-sheet figures per GPU — naming which of
    the two bounds it.  bf16x3 issues three bf16 MMAs per product, so its tensor work is 3x the algorithmic FLOPs;
  * parity: logits of a seeded sample of subgraphs against the torch-CPU SAGE restatement (tests/sage_oracle.py) on those
    subgraphs alone; the run aborts above 1e-3 relative;
  * gpu: card name, power limit and max SM clock, read in the same run.

Usage: python scripts/bench_sage.py [--steps 10] [--warmup 3] [--workload products|products-small] [--json-out PATH]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_TBS = 7.7          # HGX B200 data sheet, one GPU
BF16_TFLOPS = 2250.0   # dense BF16, one GPU
PARITY_RTOL = 1e-3
SHAPES = {"products": (2449029, 61859140), "products-small": (200000, 5000000)}


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30)
        name, power, clk = [c.strip() for c in r.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:  # the card name from the driver is still worth reporting
        return {"name": torch.cuda.get_device_name(0), "power_limit": None, "error": repr(e)}


def kernel_table(prof):
    out = {}
    for name, r in prof.items():
        s = r["ms"] * 1e-3
        tensor = 3 * r["flops"] if name.startswith("gemm") or name == "head" else 0
        t_mem, t_tc = r["bytes"] / (HBM_TBS * 1e12), tensor / (BF16_TFLOPS * 1e12)
        out[name] = {"ms": r["ms"], "launches": r["launches"], "algo_GB": r["bytes"] / 1e9,
                     "algo_TFLOP": r["flops"] / 1e12, "GBps": r["bytes"] / s / 1e9, "TFLOPs": r["flops"] / s / 1e12,
                     "bound": "hbm" if t_mem >= t_tc else "tensor (bf16x3: 3 MMAs per product)",
                     "share_of_peak": max(t_mem, t_tc) / s}
    return out


def parity(fg, so, fo, ei, part, X, sd, logits, core_gid, n_sub, k):
    rng = np.random.default_rng(0)
    sub_ids = np.sort(rng.choice(k, size=min(k, n_sub), replace=False))
    subs = fo.subgraphs_from_partition(ei.cpu().numpy(), X.cpu().numpy(), part.cpu().numpy(), sub_ids)
    row_of = torch.full((int(core_gid.max()) + 1,), -1, dtype=torch.long, device=core_gid.device)
    row_of[core_gid.long()] = torch.arange(core_gid.numel(), device=core_gid.device)
    sd_c = {k_: v.cpu() for k_, v in sd.items()}
    got, want = [], []
    with torch.no_grad():
        for b in range(0, len(subs), 128):
            x, e = fo.collate(subs[b:b + 128])
            want.append(so.classify_node(sd_c, x, e))
            nodes = torch.from_numpy(np.concatenate([s["orig_idx"] for s in subs[b:b + 128]])).to(core_gid.device)
            got.append(logits[row_of[nodes]].cpu())
    got, want = torch.cat(got).double(), torch.cat(want).double()
    scale = max(1.0, float(want.abs().max()))
    err = float((got - want).abs().max())
    blk = {"subgraphs": len(subs), "rows": int(want.shape[0]), "max_abs_err": err, "max_rel_err": err / scale,
           "rtol": PARITY_RTOL, "against": "tests/sage_oracle.py (torch CPU fp32) on the sampled subgraphs"}
    if not err / scale <= PARITY_RTOL:
        raise SystemExit(f"bench_sage: PARITY FAILURE {json.dumps(blk)}")
    return blk


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--workload", default="products", choices=sorted(SHAPES))
    p.add_argument("--parity-subgraphs", type=int, default=512)
    p.add_argument("--json-out", default=None)
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sage: needs a CUDA device (there is no CPU measurement)")
    import fitgnn_b200 as fg
    from oracle import fitgnn_oracle as fo
    from tests import sage_oracle as so

    dev = torch.device("cuda:0")
    n, e_und = SHAPES[a.workload]
    F, H, C = 100, 512, 47
    ei, part, _, k = fg.synth.planted_partition(n, e_und, 0.5, seed=0, device=dev)
    part = fg.synth.relabel_partition_reference_order(part)
    X = fg.synth.features(n, F, seed=0, device=dev)
    sd = {k_: v.to(dev) for k_, v in so.init_state_dict(F, H, C, seed=0).items()}
    pack = fg.build_pack(ei, part, k, "none")
    fwd = fg.PackedForward(pack, sd, head="log_softmax", rows="core", precision="bf16x3")
    for _ in range(max(1, a.warmup)):
        out = fwd(X)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        out = fwd(X)
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / a.steps
    fwd.enable_profile(True)  # per-kernel events in separate passes: the event records stay out of the step time
    for _ in range(a.steps):
        fwd(X)
    torch.cuda.synchronize()
    kernels = kernel_table(fwd.profile_summary())
    fwd.enable_profile(False)
    line = {"bench": "sage_products", "workload": f"{a.workload}: {n} nodes, {e_und} undirected edges, planted partition "
                                                  f"ratio 0.5 (k={k}), mode none, F={F}, 2-layer SAGEConv hidden={H}, C={C}",
            "precision": "bf16x3", "steps": a.steps, "warmup": a.warmup, "step_ms": step_ms,
            "nodes_per_s": n / (step_ms * 1e-3), "kernels": kernels, "sum_kernel_ms": sum(r["ms"] for r in kernels.values()),
            "pack": {"rows": pack.n_rows, "nnz": pack.nnz, "subgraphs": pack.n_sub},
            "parity": parity(fg, so, fo, ei, part, X, sd, out, pack.core_gid, a.parity_subgraphs, k),
            "gpu": gpu_info(), "peaks": {"hbm_TBps": HBM_TBS, "bf16_dense_TFLOPs": BF16_TFLOPS, "source": "data sheet"}}
    s = json.dumps(line)
    print(s)
    if a.json_out:
        os.makedirs(os.path.dirname(os.path.abspath(a.json_out)), exist_ok=True)
        with open(a.json_out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
