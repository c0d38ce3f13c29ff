"""Whole-pack GCN forward: the schedule that runs every subgraph of a pack through the conv stack + head in
a handful of kernel launches (replaces the per-batch Python loops run.py:59-77 / inference.py:672-688 and
the per-subgraph loops network.py:118-135, :189-204).

Schedule (SURVEY §7 ideas 2-4; all preserve the reference's arithmetic up to fp32 re-association):
  * layer 0, F > hidden  : transform-first on the DE-DUPLICATED feature rows (X holds each node once;
                           the SpMM gathers Z[gid[col]]), because (X W^T)[row] depends on the global row only
  * layer 0, F <= hidden : aggregate-first (gather F-wide rows), then GEMM with fused bias + ELU
  * layers >= 1          : aggregate-first; the LAST layer aggregates only the rows the caller reads
                           (core rows for node tasks, M.mask rows for graph tasks)
  * head                 : lt1 (+ log_softmax / softmax) on those rows only
  * fused aggregation    : when every row is an output row and every subgraph has <= 32 rows (the many-tiny-subgraphs
                           regime of high coarsening ratios, e.g. the products workload) the pack is group-aligned once
                           and layers >= 1 get their propagate from the PREVIOUS transform's epilogue
                           (fitgnn_gcn_transform_aggregate): no SpMM launch and no fp32 round trip of the hidden state

SAGEConv state_dicts (conv.{i}.lin_l.weight / lin_l.bias / lin_r.weight) run the classic schedule with the mean
aggregation of spmm.cu: layer 0 aggregate-first on the operand [mean x | x] (one GEMM against [W_l | W_r]) or, F > hidden,
transform-first Z = X·[W_l ; W_r]^T on the de-duplicated rows followed by mean + root + bias + ELU through gid; later layers
aggregate-first; the last one on the output rows only; then the head.  The pack's CSR is used as is and its one self entry
per row is the root, not a neighbour (skip_self).  A pack collapses the self-loop edges of its input into that single entry,
so on a graph with self-loop edges the pack result differs from PyG's SAGEConv, which counts such an edge as a neighbour;
the subgraphs the reference builds have none.  bf16x3 or fp32 only (the fp16 precisions run bf16x3, as for packs that are
not eligible for the fused schedule); the fused aggregation is not built for SAGE.
"""
from __future__ import annotations

import torch

from . import ops
from .pack import Pack

_HEADS = {"identity": ops.HEAD_IDENTITY, "log_softmax": ops.HEAD_LOG_SOFTMAX, "softmax": ops.HEAD_SOFTMAX}


def conv_layers(sd):
    return len({k.split(".")[1] for k in sd if k.startswith("conv.")})


def is_sage(sd):
    """A SAGEConv state_dict (PyG SAGEConv keys lin_l / lin_r) rather than a GCNConv one."""
    return "conv.0.lin_l.weight" in sd


class PackedForward:
    """Prepared forward over one pack.  `state_dict` uses the reference's keys (conv.{i}.lin.weight,
    conv.{i}.bias, lt1.weight, lt1.bias — network.py:11-22).  `rows` selects the output rows:
    'core' (node tasks), 'mask' (graph tasks: x[mask], network.py:129) or 'all'."""

    def __init__(self, pack: Pack, state_dict, head="log_softmax", rows="core", precision="bf16x3",
                 with_head=True, fuse_layer0=False, fuse_aggregate="auto", align_policy="degree", out_map=None,
                 blocked_spmm="auto", dense_spmm="lds", conv_fused=False):
        """precision: 'bf16x3' (default: tcgen05 tensor cores on a bf16 hi/lo split of both operands, fp32 accumulate,
        ~2^-17 relative operand error) or 'fp32' (exact-fp32 CUDA-core GEMM: the numerics anchor, explicit opt-in).
        out_map (int32 [n_out]): output row i is written to row out_map[i] of the `out` tensor passed to __call__
        (which then is required) — how StreamedForward lets several forwards fill one result in subgraph_list order."""
        if precision not in ("bf16x3", "fp32", "fp16x2", "fp16"):
            raise ValueError(f"precision={precision!r}")
        self.pack = pack
        dev = pack.device
        # 'fp16x2' (opt-in): bf16x3 for the first layer, then the HIDDEN STATE travels as one fp16 plane (half the bytes, two MMAs
        # per product instead of three; 2^-11 per element — include/fitgnn.h FITGNN_GEMM_FP16X2).  Fused schedule only: a pack
        # that is not eligible for it runs plain bf16x3.
        # 'fp16' (opt-in): fp16x2 whose hidden -> hidden transforms (layers >= 1) take their weights as ONE fp16 plane as well:
        # one MMA per product, and a CTA pair's half of the 256 x 512 weight block stays resident in shared memory (the
        # W-stationary pair plan of gemm_tcgen05.cu).  The head keeps its hi/lo weights (it is HBM-bound; they are free).
        self.f16_hidden = precision in ("fp16x2", "fp16")
        self.w_single = precision == "fp16"
        self.precision = ops.GEMM_FP32 if precision == "fp32" else ops.GEMM_BF16X3
        self.kalign = 8 if self.precision == ops.GEMM_BF16X3 else 4
        self.L = conv_layers(state_dict)
        assert self.L >= 1
        self.head = _HEADS[head]
        self.with_head = with_head
        f32 = dict(dtype=torch.float32, device=dev)
        self.sage = is_sage(state_dict)
        if self.sage:
            self._init_sage(state_dict, rows, fuse_aggregate, out_map, f32)
            return
        self.W, self.b = [], []
        for i in range(self.L):
            w = state_dict[f"conv.{i}.lin.weight"].detach().to(**f32)
            self.W.append(self._prep_weight(w))
            self.b.append(state_dict[f"conv.{i}.bias"].detach().to(**f32).contiguous())
        self.F = state_dict["conv.0.lin.weight"].shape[1]
        self.H = state_dict["conv.0.lin.weight"].shape[0]
        assert self.H % 4 == 0, "hidden width must be a multiple of 4"
        if with_head:
            self.Wl = self._prep_weight(state_dict["lt1.weight"].detach().to(**f32))
            self.bl = state_dict["lt1.bias"].detach().to(**f32).contiguous()
            self.C = state_dict["lt1.weight"].shape[0]
        self._select_rows(rows)
        self.Fp = self._kpad(self.F)
        self.transform_first = self.F > self.H
        # high-degree rows are split across a CTA (found once; the pack is immutable)
        self.hubs_all = ops.find_hubs(pack.rowptr, None, pack.n_rows)
        self.hubs_out = self.hubs_all if self.out_rows is None else ops.find_hubs(pack.rowptr, self.out_rows, self.n_out)
        self.launches = 0
        # block-staged SpMM (spmm.cu spmm_block_kernel) for the all-rows aggregations of packs whose rows have several
        # entries each: the sources of a block of whole subgraphs are staged in shared memory once instead of being fetched
        # through L2 once per entry.  'auto': from 8 entries per row on average — cluster_node packs (measured r2c/r2d: with
        # 2-4 entries per row the pipelined gather kernel is faster, its source rows are re-hit in L1/L2 anyway).
        self._blk = None
        import os
        min_deg = float(os.environ.get("FITGNN_BLOCKED_MIN", "8"))  # env: A/B runs of bench.py
        if blocked_spmm is True or (blocked_spmm == "auto" and pack.n_rows > 0 and pack.nnz >= min_deg * pack.n_rows):
            if bool((pack.sub_ptr[1:] >= pack.sub_ptr[:-1]).all()):
                self._blk = ops.row_blocks(pack.sub_ptr, pack.n_rows, window=16, compact=True)
                self._blk_order = ops.block_row_order(pack.rowptr, self._blk)
        # how the dense (blocked) aggregations run: 'lds' = shared-memory gathers (spmm_block_kernel; default: bit-identical to
        # the generic kernel and, measured r2k, a little faster: 76.6 vs 81.3 ms on the products cluster pack), 'mma' = per
        # 128 x 128 piece of the block's 0/1 adjacency one tensor-core product (spmm_mma.cu)
        import os
        self._dense_spmm = os.environ.get("FITGNN_DENSE_SPMM", dense_spmm)  # env: A/B runs of bench.py
        # fitgnn_gcn_layer_fused for layer 0 (gather warps inside the GEMM).  Correct but measured SLOWER than
        # SpMM + GEMM on B200 (5.1 ms vs 2.1 ms on the products workload: 4 gather warps per SM cannot hide the gather
        # latency that the stand-alone SpMM hides with 24 warps per SM), hence opt-in.
        self.fused_layer0 = None if fuse_layer0 else False
        self.prof = None  # set to {} by enable_profile(): op name -> dict(events, bytes, flops)
        self._nnz_cache = {}
        # group-aligned pack + aggregation fused into the transform epilogues (see module docstring)
        self.apack = None
        self._planes0 = None
        eligible = (self.precision == ops.GEMM_BF16X3 and self.L >= 2 and not self.transform_first and with_head
                    and self.out_rows is None and self.H > 128 and self.H % 8 == 0 and pack.n_rows > 0)
        if fuse_aggregate and eligible:
            ap = pack.aligned(32, align_policy)
            if ap is not None and ap.agg_ok:
                self.apack = ap
                self.hubs_aligned = ops.find_hubs(ap.rowptr, None, ap.n_rows)
                import os
                tricks = os.environ.get("FITGNN_ENGINE_TRICKS", "1") != "0"
                self.grouped_spmm = os.environ.get("FITGNN_SPMM_GROUPED", "1") != "0"
                self.defer_scale = tricks
                self.fold_bias = tricks and self.Fp > ops.pad4(self.F)
                if self.fold_bias:  # layer-0 weights with the bias in the spare K column (see _forward_aligned)
                    w0 = state_dict["conv.0.lin.weight"].detach().to(**f32)
                    w0 = torch.nn.functional.pad(w0, (0, ops.pad4(self.F) - self.F))
                    self.W0_fold = self._prep_weight(torch.cat([w0, self.b[0][:, None]], 1))
        if fuse_aggregate is True and self.apack is None:
            raise ValueError("fuse_aggregate=True but the pack / model is not eligible for the fused aggregation")
        # classic schedule with the fp16 hidden state: first layer aggregate-first on bf16 planes, its transform writes the
        # fp16 plane, later layers aggregate fp16 -> fp16 (ops.spmm_symnorm_f16) and transform fp16 -> fp16, head on fp16
        self.f16_classic = (self.f16_hidden and self.apack is None and self.precision == ops.GEMM_BF16X3 and self.L >= 2
                            and not self.transform_first and with_head and self.H % 8 == 0 and self.H >= 32)
        if self.f16_hidden and self.apack is None and not self.f16_classic:
            self.f16_hidden = False
        # precision 'fp16' on the fused schedule with the group-local layer-1 aggregation: the FIRST transform runs on fp16 planes
        # too (aggregated features as one fp16 plane straight out of the aggregation kernel, W0 as one fp16 plane).  Emulated
        # logit error 1.9e-5 against 1.8e-5 (profiles/r2_precision_study.md: the hidden state's rounding dominates); what it
        # buys is shared memory — the resident W0 block shrinks from 128 to 64 KB and an A stage from 32 to 16 KB, so the
        # epilogue-bound fused transform gets 8 operand stages instead of 2 (its main loop alone was load-latency-bound at
        # 2.6 us per tile with ONE tile in flight) — and half the bytes between the two kernels.
        self.f16_layer0 = bool(self.f16_hidden and self.w_single and self.apack is not None
                               and getattr(self, "grouped_spmm", False) and ops.pad4(self.F) <= 128
                               and os.environ.get("FITGNN_F16_LAYER0", "1") != "0")
        if self.f16_layer0:
            w0 = state_dict["conv.0.lin.weight"].detach().to(**f32)
            if self.fold_bias:
                w0 = torch.cat([torch.nn.functional.pad(w0, (0, ops.pad4(self.F) - self.F)), self.b[0][:, None]], 1)
            self.W0_f16 = ops.split_f16(w0.contiguous(), ldo=self._kpad(w0.shape[1]), lo=False)
        if self.f16_hidden:  # layers >= 1 and the head take fp16 hi/lo weights (the first layer's A operand stays bf16 hi/lo)
            for i in range(1, self.L):
                self.W[i] = ops.split_f16(state_dict[f"conv.{i}.lin.weight"].detach().to(**f32).contiguous(), ldo=self._kpad(self.H),
                                          lo=not self.w_single)
            # (FITGNN_HEAD_W1=1, A/B: the head's weights as one plane too — 49 KB less resident smem = 3 more A stages)
            self.Wl = ops.split_f16(state_dict["lt1.weight"].detach().to(**f32).contiguous(), ldo=self._kpad(self.H),
                                    lo=not (self.w_single and os.environ.get("FITGNN_HEAD_W1", "0") == "1"))
        # fused schedule on the fp16 plane, second form (conv_fused): spmm0 -> plain first transform -> every later layer as ONE
        # kernel act(Â·(h·W^T) + b) (ops.gcn_conv_aligned_f16: the aggregation on the raw accumulators in the epilogue of the
        # tensor-bound hidden -> hidden transform) -> head, instead of hanging layer i+1's aggregation on layer i's transform.
        # Same launches, same bytes; the exchange-heavy epilogue moves from the K = 100 transform (which it made epilogue-bound
        # with idle tensor cores) under the K = 512 main loop.  MEASURED SLOWER on the products workload (r2ak: plain transform
        # 0.85 ms + conv 1.58 ms against 1.16 + 1.19 ms): the exchange epilogue does not hide behind the MMAs, it stretches
        # them.  Opt-in.
        import os
        cf = os.environ.get("FITGNN_CONV_FUSED", "")  # env: A/B runs of bench.py
        conv_fused = {"0": False, "1": True}.get(cf, conv_fused)
        self.conv_fused = bool(conv_fused) and self.f16_hidden and self.apack is not None and self.H > 128
        self.out_map = None
        if out_map is not None:
            assert with_head, "out_map needs the head"
            self.out_map = out_map.to(device=dev, dtype=torch.int32).contiguous()
            assert self.out_map.numel() == self.n_out
        # row map of the group-aligned head: aligned row -> output row (padding rows dropped)
        self._head_map = None
        if self.apack is not None:
            self._head_map = self.apack.orig_row
            if self.out_map is not None:
                o = self.apack.orig_row.long()
                self._head_map = torch.where(o >= 0, self.out_map.long()[o.clamp(min=0)], o).to(torch.int32).contiguous()

    def _select_rows(self, rows):
        pack, dev = self.pack, self.pack.device
        if rows == "core":
            self.out_rows = pack.core_rows
        elif rows == "mask":
            self.out_rows = pack.mask_rows()
        elif rows == "all":
            self.out_rows = None
        else:
            self.out_rows = rows.to(device=dev, dtype=torch.int32).contiguous()
        if self.out_rows is not None and self.out_rows.numel() == pack.n_rows and bool(
                (self.out_rows.long() == torch.arange(pack.n_rows, device=dev)).all()):
            self.out_rows = None  # identity selection (e.g. mode 'none'): skip the row indirection in the kernels
        self.n_out = pack.n_rows if self.out_rows is None else self.out_rows.numel()

    def _init_sage(self, sd, rows, fuse_aggregate, out_map, f32):
        """SAGEConv weights for the classic schedule (module docstring)."""
        from .autograd import sage_weight_cat
        if fuse_aggregate is True:
            raise ValueError("fuse_aggregate=True: the fused aggregation is not built for SAGEConv models")
        self.f16_hidden = self.w_single = self.f16_classic = self.f16_layer0 = self.conv_fused = False
        self.apack, self._blk, self._head_map = None, None, None
        self.fused_layer0 = False
        self.prof, self.launches, self._nnz_cache = None, 0, {}
        w0 = sd["conv.0.lin_l.weight"]
        self.F, self.H = w0.shape[1], w0.shape[0]
        assert self.H % 4 == 0, "hidden width must be a multiple of 4"
        self.Fp, self.Hp = self._kpad(self.F), self._kpad(self.H)
        self.transform_first = self.F > self.H
        self.W, self.b = [], []
        for i in range(self.L):
            wl = sd[f"conv.{i}.lin_l.weight"].detach().to(**f32)
            wr = sd[f"conv.{i}.lin_r.weight"].detach().to(**f32)
            if i == 0 and self.transform_first:
                w = torch.cat([wl, wr], 0)  # [2H, F]: Z = X·[W_l ; W_r]^T
            else:
                w = sage_weight_cat(wl, wr, self.Fp if i == 0 else self.Hp)  # [H, 2 half]: [mean x | x]·[W_l | W_r]^T
            self.W.append(self._prep_weight(w))
            self.b.append(sd[f"conv.{i}.lin_l.bias"].detach().to(**f32).contiguous())
        if self.with_head:
            self.Wl = self._prep_weight(sd["lt1.weight"].detach().to(**f32))
            self.bl = sd["lt1.bias"].detach().to(**f32).contiguous()
            self.C = sd["lt1.weight"].shape[0]
        self._select_rows(rows)
        self.out_map = None
        if out_map is not None:
            assert self.with_head, "out_map needs the head"
            self.out_map = out_map.to(device=self.pack.device, dtype=torch.int32).contiguous()
            assert self.out_map.numel() == self.n_out

    def _mean(self, name, fn, width, in_cols, out_cols, src_index, last, n_src_rows, out_elem):
        """One mean-aggregation launch; bytes: rowptr + col, every distinct source row once (in_cols wide: the root form
        reads both halves of Z), the output rows, gid and the row selection."""
        p = self.pack
        key = ("nnz", last)
        if key not in self._nnz_cache:
            r = self.out_rows.long() if (last and self.out_rows is not None) else None
            self._nnz_cache[key] = p.nnz if r is None else int((p.rowptr.long()[r + 1] - p.rowptr.long()[r]).sum())
        r_out = self.n_out if last else p.n_rows
        nb = 4 * (r_out + 1) + 4 * self._nnz_cache[key] + 4 * n_src_rows * in_cols + out_elem * r_out * out_cols
        nb += 4 * p.n_rows if src_index is not None else 0
        nb += 4 * r_out if (last and self.out_rows is not None) else 0
        self.launches += 1
        return self._timed(name, fn, nbytes=nb, flops=self._nnz_cache[key] * width)

    def _forward_sage(self, X, out, packed):
        p = self.pack
        bf = self.precision == ops.GEMM_BF16X3
        X = self.pad_features(X)
        gid0 = None if packed else p.gid
        H, Fp, Hp = self.H, self.Fp, self.Hp
        h = None
        for i in range(self.L):
            last = i == self.L - 1
            rows = self.out_rows if last else None
            if i == 0 and self.transform_first:
                A = ops.split_bf16(X) if bf else X
                if bf:
                    self.launches += 1
                Z = self._gemm(A, self.W[0], None, ops.ACT_NONE, N=2 * H, K=Fp, name="gemm0_unique_rows")
                h = self._mean("mean0", lambda: ops.spmm_mean_root(p.rowptr, p.col, Z, H, H, gid0, None, True, self.b[0],
                                                                     ops.ACT_ELU, rows),
                               H, 2 * H, H, gid0, last, Z.shape[0], 4)
                continue
            src, width, half, idx = (X, Fp, Fp, gid0) if i == 0 else (h, H, Hp, None)
            n_src = src.shape[0] if idx is not None else p.n_rows
            A = self._mean(f"mean{i}", lambda: ops.spmm_mean_concat(p.rowptr, p.col, src, width, half, idx, None, True, rows,
                                                                    split=bf),
                           width, width, 2 * half, idx, last, n_src, 4)
            to_head = bf and last and self.with_head and H % 8 == 0
            h = self._gemm(A, self.W[i], self.b[i], ops.ACT_ELU, N=H, K=2 * half, name=f"gemm{i}", split_out=to_head)
        return self._finish(h, out, X.device)

    # -- per-kernel timing for the roofline report (CUDA events on the launching stream) ---------
    def enable_profile(self, on=True):
        self.prof = {} if on else None

    def _timed(self, name, fn, nbytes=0, flops=0):
        if self.prof is None:
            return fn()
        st = torch.cuda.current_stream()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        out = fn()
        b.record(st)
        rec = self.prof.setdefault(name, dict(events=[], bytes=nbytes, flops=flops))
        rec["events"].append((a, b))
        return out

    def profile_summary(self):
        """{op: dict(ms=mean launch duration, launches, bytes, flops)} — call after a synchronize."""
        out = {}
        for name, rec in (self.prof or {}).items():
            ms = [a.elapsed_time(b) for a, b in rec["events"]]
            out[name] = dict(ms=sum(ms) / len(ms), launches=len(ms), bytes=rec["bytes"], flops=rec["flops"])
        return out

    def _spmm_bytes(self, width, src_index, last, n_src_rows, out_elem=4, in_elem=4):
        """Algorithmic bytes of one SpMM launch (SURVEY §8d): CSR rowptr + col, dinv of the sources, the
        optional gid read, every distinct source row once, every output row once, bias."""
        p = self.pack
        key = ("nnz", last)
        if key not in self._nnz_cache:
            if last and self.out_rows is not None:
                r = self.out_rows.long()
                rp = p.rowptr.long()
                nnz = int((rp[r + 1] - rp[r]).sum())
            else:
                nnz = p.nnz
            self._nnz_cache[key] = nnz
        nnz = self._nnz_cache[key]
        r_out = self.n_out if last else p.n_rows
        b = 4 * (r_out + 1) + 4 * nnz + in_elem * n_src_rows * width + out_elem * r_out * width + 4 * width + 4 * n_src_rows
        if src_index is not None:
            b += 4 * p.n_rows
        if last and self.out_rows is not None:
            b += 4 * r_out
        return b

    def _spmm_bytes_aligned(self, width, src_index, n_src_rows):
        """Algorithmic bytes of the layer-0 aggregation on the group-aligned pack (same formula as _spmm_bytes)."""
        ap = self.apack
        b = 4 * (ap.n_rows + 1) + 4 * ap.nnz + 4 * ap.n_rows + 4 * (n_src_rows if src_index is not None else ap.n_rows) * width \
            + 4 * ap.n_rows * width
        return b + (4 * ap.n_rows if src_index is not None else 0)

    # -- helpers -------------------------------------------------------------------------------
    def _kpad(self, k):
        return (k + self.kalign - 1) // self.kalign * self.kalign

    def _prep_weight(self, w):
        """[out, in] fp32 -> K padded with zero columns; bf16 hi/lo planes for the tensor-core path."""
        kp = self._kpad(w.shape[1])
        if self.precision == ops.GEMM_BF16X3:
            return ops.split_bf16(w.contiguous(), ldo=kp)
        if kp != w.shape[1]:
            w = torch.nn.functional.pad(w, (0, kp - w.shape[1]))
        return w.contiguous()

    def _gemm(self, A, W, bias, act, head=ops.HEAD_IDENTITY, N=None, K=None, name="gemm", out=None, split_out=False,
              row_scale=None):
        self.launches += 1 + (1 if (head != ops.HEAD_IDENTITY and self.precision == ops.GEMM_FP32) else 0)
        M = (A[0] if isinstance(A, tuple) else A).shape[0]
        return self._timed(name, lambda: ops.gemm_bias_act(A, W, bias, act, head, precision=self.precision, N=N, K=K,
                                                           out=out, split_out=split_out, row_scale=row_scale),
                           nbytes=4 * (M * K + K * N + M * N), flops=2 * M * K * N)

    def _spmm(self, X, width, src_index, bias, act, last, split, name="spmm", pack=None, out=None):
        p = self.pack if pack is None else pack
        rows = self.out_rows if last else None
        hubs = self.hubs_out if last else self.hubs_all
        if pack is not None:
            hubs = self.hubs_aligned
        n_src_rows = X.shape[0] if src_index is not None else p.n_rows
        if rows is None and pack is None and self._blk is not None and self._dense_spmm == "mma":
            self.launches += 1
            return self._timed(name, lambda: ops.spmm_symnorm_mma(p.rowptr, p.col, p.dinv, X, self._blk, width, src_index, bias,
                                                                  act, out=out, split=split),
                               nbytes=self._spmm_bytes(width, src_index, last, n_src_rows))
        if rows is None and pack is None and self._blk is not None:
            self.launches += 1
            return self._timed(name, lambda: ops.spmm_symnorm_blocked(p.rowptr, p.col, p.dinv, X, self._blk, width, src_index,
                                                                      bias, act, out=out, split=split,
                                                                      row_order=self._blk_order),
                               nbytes=self._spmm_bytes(width, src_index, last, n_src_rows))
        self.launches += 1 + (1 if hubs[1] > 0 else 0)
        return self._timed(name, lambda: ops.spmm_symnorm(p.rowptr, p.col, p.dinv, X, width, src_index, bias, act, rows,
                                                          split=split, hubs=hubs, out=out),
                           nbytes=self._spmm_bytes(width, src_index, last, n_src_rows))

    def _fused_layer0(self, X, last):
        """Layer 0 as ONE kernel: gather warps build Â·X[gid] tiles in shared memory for the tensor-core transform."""
        from ._lib import FitgnnError
        p = self.pack
        rows = self.out_rows if last else None
        n_rows = self.n_out if last else p.n_rows
        to_head = last and self.with_head and self.H % 8 == 0
        nbytes = self._spmm_bytes(self.Fp, p.gid, last, X.shape[0], out_elem=0) + 4 * n_rows * self.H
        flops = 2 * n_rows * self.Fp * self.H
        try:
            out = self._timed("layer0_fused", lambda: ops.gcn_layer_fused(
                p.rowptr, p.col, p.dinv, X, self.Fp, self.W[0], self.b[0], ops.ACT_ELU, src_index=p.gid, out_rows=rows,
                N=self.H, split_out=to_head), nbytes=nbytes, flops=flops)
        except FitgnnError as e:
            if "EUNSUP" not in str(e):
                raise
            self.fused_layer0 = False
            if self.prof is not None:
                self.prof.pop("layer0_fused", None)
            return None
        self.fused_layer0 = True
        self.launches += 1
        return out

    def pad_features(self, X):
        """Rows of the de-duplicated feature table, K-padded (a view when no padding is needed)."""
        if X.shape[1] == self.Fp and X.is_contiguous():
            return X
        Xp = torch.zeros(X.shape[0], self.Fp, dtype=torch.float32, device=X.device)
        Xp[:, : X.shape[1]].copy_(X)
        return Xp

    def pack_features(self, X):
        """Node-ordered feature table [n_src, F] -> one row per pack row, in the row order of the pack this forward
        runs on (the group-aligned pack when the fused schedule is active).  This is the layout the reference feeds its
        models: every subgraph carries its own copy of x (utils.py:248, :266) and the loader collates them in subgraph
        order (run.py:336).  Done once per graph, like the pack itself; `__call__(Xp, packed=True)` then streams the
        rows instead of gathering them through gid.  Padding rows (never read) get row 0."""
        ap = self.apack if self.apack is not None else self.pack
        if X.shape[1] % 4 != 0:
            X = torch.nn.functional.pad(X, (0, ops.pad4(X.shape[1]) - X.shape[1]))
        return X[ap.gid.long().clamp_(min=0)].contiguous()

    def _forward_aligned(self, X, out, peer_ptrs=None, packed=False):
        """spmm0 -> [transform + next layer's aggregation]* -> last transform -> head with the padding rows dropped."""
        ap = self.apack
        M = ap.n_rows
        # X may come un-padded ([n, F]) or with the K-padded pitch: the SpMM reads F columns either way; the planes keep
        # the 8-element pitch the TMA maps need and the TMA unit zero-fills whatever lies beyond K.
        # Bias fold: when the pitch leaves a spare column (Fp > F) the planes carry a constant 1 there and the weight planes
        # carry the bias, so the layer-0 epilogue has no bias add (K = F + 1).  The planes are allocated once (the SpMM never
        # touches columns >= F), so a PackedForward must be driven from one stream at a time.
        Wd = ops.pad4(self.F)  # columns the SpMM reads / writes (X has at least that many: see __call__)
        fold = self.fold_bias
        src = None if packed else ap.gid
        if self.f16_layer0:
            if self._planes0 is None or self._planes0.device != X.device:
                self._planes0 = torch.zeros(M, self.Fp, dtype=torch.float16, device=X.device)
                if fold:
                    self._planes0[:, Wd] = 1.0
            self.launches += 1
            b4 = self._spmm_bytes_aligned(Wd, src, X.shape[0])
            A = self._timed("spmm0", lambda: ops.spmm_symnorm_grouped_f16(ap.rowptr, ap.col, ap.dinv, X, Wd, src, out=self._planes0,
                                                                          pad_value=(1.0 if fold else 0.0)),
                            nbytes=b4 - 2 * ap.n_rows * Wd)  # the output is 2 bytes per element
        elif self._planes0 is None or self._planes0[0].device != X.device:
            hi = torch.zeros(M, self.Fp, dtype=torch.bfloat16, device=X.device)
            lo = torch.zeros(M, self.Fp, dtype=torch.bfloat16, device=X.device)
            if fold:
                hi[:, Wd] = 1.0
            self._planes0 = (hi, lo)
        if self.f16_layer0:
            pass
        elif self.grouped_spmm and Wd <= 128:
            # group-local aggregation: the group's 32 source rows are staged in shared memory once (spmm.cu)
            self.launches += 1
            # the pad columns of the planes (constant 1 of the bias fold / zeros) are re-written with the same values:
            # whole-sector stores instead of a DRAM read-modify-write per row
            A = self._timed("spmm0", lambda: ops.spmm_symnorm_grouped(ap.rowptr, ap.col, ap.dinv, X, Wd, src, split=True,
                                                                      out=self._planes0,
                                                                      pad_value=(1.0 if fold else 0.0)),
                            nbytes=self._spmm_bytes_aligned(Wd, src, X.shape[0]))
        else:
            A = self._spmm(X, Wd, src, None, ops.ACT_NONE, False, split=True, name="spmm0", pack=ap, out=self._planes0)
        K = Wd + 1 if fold else Wd
        if self.conv_fused:
            return self._tail_conv_fused(A, K, M, X, out, peer_ptrs)
        for i in range(self.L - 1):
            Ai, Ki = A, K
            Wi, bi = (self.W0_fold, None) if (i == 0 and fold) else (self.W[i], self.b[i])
            if i == 0 and self.f16_layer0:
                Wi = self.W0_f16
            # the leading dinv[r] of the aggregation moves into the next transform's epilogue (one FFMA with its bias) when
            # that consumer is the plain last transform
            defer = self.defer_scale and i == self.L - 2
            self.launches += 1
            if self.f16_hidden:
                a_b = 2 if not isinstance(Ai, tuple) else 4  # bytes per element of the A operand
                A = self._timed(f"gemm{i}_agg", lambda: ops.gcn_transform_aggregate_f16(
                    Ai, Wi, bi, ops.ACT_ELU, ap.agg_desc, ap.dinv, K=Ki, N=self.H, defer_row_scale=defer),
                    nbytes=a_b * M * Ki + 4 * Ki * self.H + 2 * M * self.H + 12 * M, flops=2 * M * Ki * self.H)
            else:
                A = self._timed(f"gemm{i}_agg", lambda: ops.gcn_transform_aggregate(
                    Ai, Wi, bi, ops.ACT_ELU, ap.agg_desc, ap.dinv, K=Ki, N=self.H, defer_row_scale=defer),
                    nbytes=4 * (M * Ki + Ki * self.H + M * self.H) + 12 * M, flops=2 * M * Ki * self.H)
            K = self.H
        i = self.L - 1
        if self.f16_hidden:
            self.launches += 2
            h = self._timed(f"gemm{i}", lambda: ops.gemm_f16(A, self.W[i], self.b[i], ops.ACT_ELU, row_scale=ap.dinv if self.defer_scale else None,
                                                              out_f16=True, K=K, N=self.H),
                            nbytes=2 * M * K + 4 * K * self.H + 2 * M * self.H, flops=2 * M * K * self.H)
            nb16 = 2 * M * self.H + 4 * self.H * self.C + 4 * self.n_out * self.C + 4 * M
            if peer_ptrs is not None:  # rows go straight into this rank's slot of every rank's gather buffer
                self._timed("head", lambda: ops.gemm_f16_head_rows_peers(h, self.Wl, self.bl, ops.ACT_NONE, self.head, self._head_map,
                                                                         peer_ptrs, ops.pad4(self.C), K=self.H, N=self.C),
                            nbytes=nb16 + 4 * (len(peer_ptrs) - 1) * self.n_out * self.C, flops=2 * M * self.H * self.C)
                return None
            view = None
            if out is None:
                out = torch.empty(self.n_out, ops.pad4(self.C), dtype=torch.float32, device=X.device)
                view = out[:, : self.C]
            self._timed("head", lambda: ops.gemm_f16(h, self.Wl, self.bl, ops.ACT_NONE, self.head, row_map=self._head_map, out=out,
                                                     K=self.H, N=self.C),
                        nbytes=nb16, flops=2 * M * self.H * self.C)
            return out if view is None else view
        h = self._gemm(A, self.W[i], self.b[i], ops.ACT_ELU, N=self.H, K=K, name=f"gemm{i}", split_out=True,
                       row_scale=ap.dinv if self.defer_scale else None)
        view = None
        self.launches += 1
        nb = 4 * (M * self.H + self.H * self.C + self.n_out * self.C) + 4 * M
        if peer_ptrs is not None:  # rows go straight into this rank's slot of every rank's gather buffer
            self._timed("head", lambda: ops.gemm_head_rows_peers(h, self.Wl, self.bl, ops.ACT_NONE, self.head, self._head_map,
                                                                 peer_ptrs, ops.pad4(self.C), K=self.H, N=self.C),
                        nbytes=nb + 4 * (len(peer_ptrs) - 1) * self.n_out * self.C, flops=2 * M * self.H * self.C)
            return None
        if out is None:
            out = torch.empty(self.n_out, ops.pad4(self.C), dtype=torch.float32, device=X.device)
            view = out[:, : self.C]
        self._timed("head", lambda: ops.gemm_head_rows(h, self.Wl, self.bl, ops.ACT_NONE, self.head, self._head_map, out,
                                                       K=self.H, N=self.C), nbytes=nb, flops=2 * M * self.H * self.C)
        return out if view is None else view

    def _tail_conv_fused(self, A, K, M, X, out, peer_ptrs):
        """Rest of the aligned forward in the conv_fused form: plain first transform, then one kernel per later layer."""
        ap, H = self.apack, self.H
        fold = self.fold_bias
        W0, b0 = (self.W0_fold, None) if fold else (self.W[0], self.b[0])
        if self.f16_layer0:
            W0 = self.W0_f16
        self.launches += 1
        h = self._timed("gemm0", lambda: ops.gcn_transform_aggregate_f16(A, W0, b0, ops.ACT_ELU, None, None, K=K, N=H),
                        nbytes=4 * M * K + 4 * K * H + 2 * M * H, flops=2 * M * K * H)
        for i in range(1, self.L):
            hi_, Wi, bi = h, self.W[i], self.b[i]
            self.launches += 1
            h = self._timed(f"conv{i}", lambda: ops.gcn_conv_aligned_f16(hi_, Wi, bi, ops.ACT_ELU, ap.agg_desc, ap.dinv, K=H, N=H),
                            nbytes=2 * M * H + 4 * H * H + 2 * M * H + 12 * M, flops=2 * M * H * H)
        self.launches += 1
        nb16 = 2 * M * H + 4 * H * self.C + 4 * self.n_out * self.C + 4 * M
        if peer_ptrs is not None:
            self._timed("head", lambda: ops.gemm_f16_head_rows_peers(h, self.Wl, self.bl, ops.ACT_NONE, self.head, self._head_map,
                                                                     peer_ptrs, ops.pad4(self.C), K=H, N=self.C),
                        nbytes=nb16 + 4 * (len(peer_ptrs) - 1) * self.n_out * self.C, flops=2 * M * H * self.C)
            return None
        view = None
        if out is None:
            out = torch.empty(self.n_out, ops.pad4(self.C), dtype=torch.float32, device=X.device)
            view = out[:, : self.C]
        self._timed("head", lambda: ops.gemm_f16(h, self.Wl, self.bl, ops.ACT_NONE, self.head, row_map=self._head_map, out=out,
                                                 K=H, N=self.C), nbytes=nb16, flops=2 * M * H * self.C)
        return out if view is None else view

    # -- forward -------------------------------------------------------------------------------
    @torch.no_grad()
    def __call__(self, X, out=None, peer_ptrs=None, packed=False):
        """X: [n_src, F] fp32 CUDA — every node once (+ one row per cluster for cluster mode, i.e. C·X); with
        packed=True: the output of pack_features (one row per pack row, no gid indirection).
        Returns [n_out, C] (or the last hidden [n_out, H] when with_head=False), rows in pack order.
        `out` ([n_out, C] fp32, e.g. this rank's slot of an all-gather buffer) receives the head output in place.
        `peer_ptrs` (dist.PeerGather.slot_ptrs; fused-aggregation schedule only): the head stores its rows into that slot
        of every rank's gather buffer instead (pitch pad4(C)) and nothing is returned."""
        if self.sage and peer_ptrs is not None:
            raise NotImplementedError("peer stores (dist.PeerGather) are built for GCNConv models only, not SAGEConv")
        assert peer_ptrs is None or self.apack is not None, "peer stores need the group-aligned schedule"
        assert self.out_map is None or (out is not None and peer_ptrs is None), "out_map needs the `out` tensor"
        p = self.pack
        assert X.is_cuda and X.dtype == torch.float32
        if self.sage:
            assert X.shape[0] == (p.n_rows if packed else p.n_src) and X.shape[1] in (self.F, ops.pad4(self.F), self.Fp), \
                tuple(X.shape)
            return self._forward_sage(X, out, packed)
        n_in = (self.apack if self.apack is not None else p).n_rows if packed else p.n_src
        assert X.shape[0] == n_in and X.shape[1] in (self.F, ops.pad4(self.F), self.Fp), tuple(X.shape)
        bf = self.precision == ops.GEMM_BF16X3
        if self.apack is not None:
            if not (X.is_contiguous() and X.shape[1] % 4 == 0):
                X = self.pad_features(X)
            return self._forward_aligned(X, out, peer_ptrs, packed)
        X = self.pad_features(X)
        gid0 = None if packed else p.gid
        h = None
        if self.f16_classic:
            return self._forward_classic_f16(X, gid0, out)
        for i in range(self.L):
            last = i == self.L - 1
            if i == 0 and self.transform_first:
                A = ops.split_bf16(X) if bf else X
                if bf:
                    self.launches += 1
                Z = self._gemm(A, self.W[0], None, ops.ACT_NONE, N=self.H, K=self.Fp, name="gemm0_unique_rows")
                h = self._spmm(Z, self.H, gid0, self.b[0], ops.ACT_ELU, last, split=False, name="spmm0")
            elif i == 0 and bf and self.fused_layer0 is not False and self.Fp <= 128 and self.H > 128 and not packed:
                h = self._fused_layer0(X, last)
                if h is None:  # not eligible for this shape: SpMM + GEMM below
                    A = self._spmm(X, self.Fp, gid0, None, ops.ACT_NONE, last, split=bf, name="spmm0")
                    h = self._gemm(A, self.W[0], self.b[0], ops.ACT_ELU, N=self.H, K=self.Fp, name="gemm0",
                                   split_out=bf and last and self.with_head and self.H % 8 == 0)
            else:
                src, width, idx = (X, self.Fp, gid0) if i == 0 else (h, self.H, None)
                A = self._spmm(src, width, idx, None, ops.ACT_NONE, last, split=bf, name=f"spmm{i}")
                # the last conv layer feeds only the head GEMM: emit its bf16 hi/lo planes straight from the epilogue
                to_head = bf and last and self.with_head and self.H % 8 == 0
                h = self._gemm(A, self.W[i], self.b[i], ops.ACT_ELU, N=self.H, K=width, name=f"gemm{i}",
                               split_out=to_head)
        return self._finish(h, out, X.device)

    def _finish(self, h, out, device):
        """Head of the classic schedule on the last hidden state h (fp32, or bf16 planes from the last transform)."""
        bf = self.precision == ops.GEMM_BF16X3
        if not self.with_head:
            return h
        if bf and not isinstance(h, tuple):
            h = self._timed("split_head", lambda: ops.split_bf16(h), nbytes=8 * h.numel())
            self.launches += 1
        view = None
        if self.out_map is not None:  # rows go to out[out_map]
            if bf:
                self.launches += 1
                self._timed("head", lambda: ops.gemm_head_rows(h, self.Wl, self.bl, ops.ACT_NONE, self.head, self.out_map, out,
                                                               K=self.H, N=self.C),
                            nbytes=4 * (self.n_out * self.H + self.H * self.C + self.n_out * self.C) + 4 * self.n_out,
                            flops=2 * self.n_out * self.H * self.C)
            else:
                res = self._gemm(h, self.Wl, self.bl, ops.ACT_NONE, self.head, N=self.C, K=self.H, name="head")
                out[self.out_map.long(), : self.C] = res
            return out
        if out is None and self.C % 4 != 0:
            # 16-byte aligned row pitch -> coalesced / TMA stores in the head epilogue; callers get the [:, :C] view
            out = torch.empty(self.n_out, ops.pad4(self.C), dtype=torch.float32, device=device)
            view = out[:, : self.C]
        res = self._gemm(h, self.Wl, self.bl, ops.ACT_NONE, self.head, N=self.C, K=self.H, name="head", out=out)
        return res if view is None else view

    def _forward_classic_f16(self, X, gid0, out):
        """Classic schedule (SpMM + transform per layer) with the hidden state as ONE fp16 plane (precision='fp16x2')."""
        p = self.pack
        H, Fp = self.H, self.Fp
        A = self._spmm(X, Fp, gid0, None, ops.ACT_NONE, False, split=True, name="spmm0")
        self.launches += 1
        M = p.n_rows
        h = self._timed("gemm0", lambda: ops.gcn_transform_aggregate_f16(A, self.W[0], self.b[0], ops.ACT_ELU, None, None,
                                                                         K=Fp, N=H),
                        nbytes=4 * M * Fp + 4 * Fp * H + 2 * M * H, flops=2 * M * Fp * H)
        for i in range(1, self.L):
            last = i == self.L - 1
            rows = self.out_rows if last else None
            hubs = self.hubs_out if last else self.hubs_all
            n_rows = self.n_out if last else p.n_rows
            src = h
            self.launches += 1 + (1 if hubs[1] > 0 else 0)
            A = self._timed(f"spmm{i}", lambda: ops.spmm_symnorm_f16(p.rowptr, p.col, p.dinv, src, H, None, None, ops.ACT_NONE,
                                                                      rows, hubs=hubs),
                            nbytes=self._spmm_bytes(H, None, last, p.n_rows, out_elem=2, in_elem=2))
            self.launches += 1
            h = self._timed(f"gemm{i}", lambda: ops.gemm_f16(A, self.W[i], self.b[i], ops.ACT_ELU, out_f16=True, K=H, N=H),
                            nbytes=2 * n_rows * H + 4 * H * H + 2 * n_rows * H, flops=2 * n_rows * H * H)
        n = self.n_out
        self.launches += 1
        nb = 2 * n * H + 4 * H * self.C + 4 * n * self.C
        fl = 2 * n * H * self.C
        if self.out_map is not None:
            self._timed("head", lambda: ops.gemm_f16(h, self.Wl, self.bl, ops.ACT_NONE, self.head, row_map=self.out_map, out=out,
                                                     K=H, N=self.C), nbytes=nb + 4 * n, flops=fl)
            return out
        view = None
        if out is None:
            out = torch.empty(n, ops.pad4(self.C), dtype=torch.float32, device=X.device)
        if out.shape[1] != self.C:
            view = out[:, : self.C]
        self._timed("head", lambda: ops.gemm_f16(h, self.Wl, self.bl, ops.ACT_NONE, self.head, out=out, K=H, N=self.C),
                    nbytes=nb, flops=fl)
        return out if view is None else view

    def capture(self, X_example):
        """CUDA-graph the whole forward (the small configs are launch-bound, SURVEY §7.5): returns run(X) that copies X
        into a static buffer, replays the captured launches and returns the static output tensor."""
        static_x = self.pad_features(X_example).clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                self(static_x)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            static_out = self(static_x)

        def run(X):
            static_x[:, : X.shape[1]].copy_(X)
            graph.replay()
            return static_out

        run.graph, run.static_out = graph, static_out
        return run

    def scatter_to_nodes(self, out, n_nodes=None):
        """Core-row outputs (pack order) -> [N, C] in global node order."""
        n_nodes = self.pack.n_nodes if n_nodes is None else n_nodes
        full = torch.empty(n_nodes, out.shape[1], dtype=out.dtype, device=out.device)
        full[self.pack.core_gid.long()] = out
        return full
