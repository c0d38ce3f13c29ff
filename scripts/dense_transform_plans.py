"""Which kernel instantiation and plan every dispatch case of tests/test_gpu_dense_transform.py reaches.

One torch.profiler pass per case (CUDA activities only), then the kernels of that pass from the exported trace: the template
name (tile width, epilogue warps, CTA pair), the grid and the dynamic shared memory.  Whether a launch keeps its weights
resident (W-stationary) is a run-time argument of the same instantiation and can have the same grid and shared memory as the
streaming plan; the condition table in the test file states which cases take it.

    python scripts/dense_transform_plans.py [--out DIR]     (needs cuda:0; writes DIR/plans.txt and nothing else)
"""
import argparse
import json
import os
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for plans.txt (default: print only)")
    args = ap.parse_args()
    import fitgnn_b200 as fg
    from tests import test_gpu_dense_transform as t

    lines = [f"device: {torch.cuda.get_device_name(0)}"]
    with tempfile.TemporaryDirectory() as tmp:
        for case in t.DISPATCH_CASES:
            M, K, N, bias_kind, act, switches = case.values
            A, _ = t.planes(fg, M, K, 1)
            W, _ = t.planes(fg, N, K, 2)
            bias = t.make_bias(bias_kind, N, 3)
            with t.tuning(fg, **switches):
                fg.ops.gemm_bias_act(A, W, bias, act, K=K, N=N, precision=fg.ops.GEMM_BF16X3)  # warm-up (smem attribute)
                torch.cuda.synchronize()
                with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                    fg.ops.gemm_bias_act(A, W, bias, act, K=K, N=N, precision=fg.ops.GEMM_BF16X3)
                    torch.cuda.synchronize()
            path = os.path.join(tmp, "trace.json")
            prof.export_chrome_trace(path)
            with open(path) as f:
                events = json.load(f)["traceEvents"]
            for e in events:
                if e.get("cat") == "kernel" and "gemm_bf16x3_kernel" in e.get("name", ""):
                    a = e.get("args", {})
                    name = e["name"].split("gemm_bf16x3_kernel")[1].split(">")[0] + ">"
                    lines.append(f"{case.id:32s} gemm_bf16x3_kernel{name:28s} grid {a.get('grid')} "
                                 f"smem {a.get('shared memory')}")
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "plans.txt"), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
