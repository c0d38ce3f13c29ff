"""Streamed / hybrid forward: the whole subgraph_list through the model in size-bounded shards.

The reference streams its subgraphs through the model 128 at a time (G_DataLoader(graphs, batch_size=128), run.py:336;
loops run.py:59-77 and :186-197), so its working set is one batch.  `PackedForward` runs a whole pack at once, which is
the fast way while the activations fit; two things break that:
  * cluster_node augmentation at ogbn-products scale: ~10^8 pack rows (N + nnz(Ac)), > 2^31 CSR entries, 209 GB for ONE
    512-wide fp32 activation -> the pack only exists as shards (pack.build_pack_stream) and the forward runs shard by
    shard, the caching allocator re-using the previous shard's activation buffers (stream-ordered);
  * heavy-tailed subgraph sizes (real coarsenings: core size p99 ~180, max ~500, SURVEY §7): ONE subgraph with more than 32
    rows used to drop the whole pack from the fused schedule (aggregation inside the transform's epilogue, engine.py) to
    the classic one.  Here every shard is split by subgraph size: subgraphs <= 32 rows run the fused group-aligned
    schedule, the rest the classic SpMM + GEMM schedule, and both write their rows of the SAME output tensor through
    row maps (fitgnn_gemm_head_rows), so the result is in subgraph_list order as before.
Results are those of PackedForward on the unsplit pack (same kernels per row; tests/test_gpu_stream.py)."""
from __future__ import annotations

import torch

from . import ops
from .engine import PackedForward, is_sage
from .infer import select_subgraphs
from .pack import Pack, PackStream


class StreamedForward:
    """Prepared forward over a PackStream (or a single Pack).  `rows`: 'core' only (node tasks)."""

    def __init__(self, packs, state_dict, head="log_softmax", precision="bf16x3", hybrid="auto", small_rows=32,
                 align_policy="degree", min_small_fraction=0.05):
        if is_sage(state_dict):
            raise NotImplementedError("StreamedForward runs GCNConv models only; run a SAGEConv model per pack with "
                                      "PackedForward")
        if isinstance(packs, Pack):
            packs = PackStream([packs], [0, packs.n_sub], packs.mode, packs.n_nodes, packs.n_src)
        self.stream = packs
        self.C = state_dict["lt1.weight"].shape[0]
        self.Cp = ops.pad4(self.C)
        self.parts = []   # PackedForward objects in execution order
        self.kinds = []   # 'fused' | 'classic' per part
        self.n_out = 0
        kw = dict(head=head, rows="core", precision=precision, align_policy=align_policy)
        for pack in packs.packs:
            base = self.n_out
            self.n_out += pack.n_core
            split = None
            if hybrid and precision in ("bf16x3", "fp16x2", "fp16") and pack.n_core == pack.n_rows and pack.n_sub > 1:
                # fused-schedule candidates: subgraphs of <= 32 rows whose rows have <= 12 neighbours (the epilogue's
                # aggregation descriptor, align.cu); one oversized subgraph or one high-degree row no longer drops the rest
                sizes = (pack.sub_ptr[1:] - pack.sub_ptr[:-1]).long()
                deg = (pack.rowptr[1:] - pack.rowptr[:-1]).long() - 1
                sub_of_row = torch.repeat_interleave(torch.arange(pack.n_sub, device=pack.device), sizes)
                max_deg = torch.zeros(pack.n_sub, dtype=torch.long, device=pack.device).scatter_reduce_(
                    0, sub_of_row, deg, reduce="amax", include_self=True)
                small = (sizes <= small_rows) & (max_deg <= 12)
                n_small_rows = int(sizes[small].sum())
                if 0 < n_small_rows < pack.n_rows and n_small_rows >= min_small_fraction * pack.n_rows:
                    split = small
            if split is None:
                fuse = "auto" if hybrid else False  # hybrid=False: the classic schedule everywhere
                f = PackedForward(pack, state_dict, fuse_aggregate=fuse, out_map=self._iota(base, pack.n_core, pack.device), **kw) \
                    if len(packs.packs) > 1 else PackedForward(pack, state_dict, fuse_aggregate=fuse, **kw)
                self._add(f, base)
                continue
            # position of every pack row among the core rows (= output row inside this shard)
            pos = torch.full((pack.n_rows,), -1, dtype=torch.long, device=pack.device)
            pos[pack.core_rows.long()] = torch.arange(pack.n_core, device=pack.device)
            for ids, fuse in ((torch.nonzero(split).view(-1), "auto"), (torch.nonzero(~split).view(-1), False)):
                sub, rows = select_subgraphs(pack, ids, return_rows=True)
                out_map = (pos[rows[sub.core_rows.long()]] + base).to(torch.int32)
                self._add(PackedForward(sub, state_dict, fuse_aggregate=fuse, out_map=out_map, **kw), base)
        self.prof = None

    @staticmethod
    def _iota(base, n, device):
        return torch.arange(base, base + n, dtype=torch.int32, device=device)

    def _add(self, f, base):
        f._out_base = base
        self.parts.append(f)
        self.kinds.append("fused" if f.apack is not None else "classic")

    @property
    def launches(self):
        return sum(f.launches for f in self.parts)

    def enable_profile(self, on=True):
        for f in self.parts:
            f.enable_profile(on)

    def profile_summary(self):
        """{op: dict(ms = per-step time summed over the parts, launches, bytes, flops)}; ops of the fused parts keep
        their names, those of the classic parts are prefixed 'c_' when both kinds are present."""
        both = len(set(self.kinds)) > 1
        out = {}
        for f, kind in zip(self.parts, self.kinds):
            for name, r in f.profile_summary().items():
                key = ("c_" + name) if (both and kind == "classic") else name
                a = out.setdefault(key, dict(ms=0.0, launches=0, bytes=0, flops=0))
                a["ms"] += r["ms"]; a["launches"] += r["launches"]; a["bytes"] += r["bytes"]; a["flops"] += r["flops"]
        return out

    def table_features(self, X):
        """The feature table in the pitch the parts read ([n_src, F] -> K-padded for the classic schedule)."""
        need_pad = any(f.apack is None for f in self.parts) or X.shape[1] % 4 != 0
        return self.parts[0].pad_features(X) if need_pad else X

    @torch.no_grad()
    def __call__(self, X, out=None):
        """X: [n_src, F] fp32 feature table (every node once, + C·X rows in cluster mode).  Returns [n_core, C] in
        subgraph_list order (a view of the [n_core, pad4(C)] buffer `out`)."""
        if len(self.parts) == 1 and self.parts[0].out_map is None:
            return self.parts[0](X, out=out)
        if out is None:
            out = torch.empty(self.n_out, self.Cp, dtype=torch.float32, device=X.device)
        assert out.shape[0] == self.n_out and out.stride(0) == self.Cp
        Xp = None
        for f in self.parts:
            if f.apack is not None and X.shape[1] % 4 == 0 and X.is_contiguous():
                f(X, out=out)
            else:
                if Xp is None:
                    Xp = f.pad_features(X)
                f(Xp, out=out)
        return out[:, : self.C]
