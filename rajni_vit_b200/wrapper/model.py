"""RAJNIViTWrapper — drop-in for rajni/wrapper/model.py:6-69, running on sm_100a kernels.

The class keeps the reference's constructor, attribute names (``m``, ``blocks``,
``pruning_schedule``, ``blk.attn`` swapped for ``RAJNIAttention``, ``blk.has_pruner``),
``forward`` and ``get_last_stats()``.  The body of ``forward`` does not call the base
model's modules: it reads their leaf parameters and launches the kernels of
``librajni_b200.so`` — pruned and un-pruned blocks, patch-embed and head alike.

Deliberate deviations from the reference (SURVEY.md section 5):
  * schedule keys may be ints or digit strings (the reference silently prunes
    nothing for the string keys that ``json.load`` produces);
  * activations are bf16 with fp32 accumulation, scores are fp32;
  * ties in the top-k are broken by lower index (torch.topk leaves it undefined);
  * unsupported base models raise instead of silently diverging.

Beyond the reference's models it runs the two DeiT families: LayerScale (DeiT-III's ``ls1`` / ``ls2``, folded into the
proj / fc2 weights), a class token without a position (``no_embed_class``), and a distillation token (distilled DeiT:
two prefix tokens, always kept, and the eval-mode average of ``head`` and ``head_dist``).  It also runs average-pooled
heads (``global_pool='avg'`` with ``fc_norm``, MAE fine-tunes: the mean of the patch tokens the last block kept, then
fc_norm, in one kernel) and a pre-norm stem (``norm_pre``, CLIP fine-tunes: one LayerNorm pass over the embedded tokens
that also writes block 0's LayerNorm statistics), with or without a patch-embedding bias.  A headless model (``head`` =
Identity, timm's ``num_classes=0``: DINO and other backbones) returns its pooled, normalised features [B, C], stored in fp32
by the final LayerNorm or pooling kernel itself.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional

import torch
import torch.nn as nn

from .. import ops
from ..packing import PackCache
from .attention import RAJNIAttention, keep_count


def _normalise_schedule(schedule: Dict) -> Dict[int, Dict]:
    out = {}
    for k, cfg in schedule.items():
        if isinstance(k, str):
            if not k.strip().lstrip("-").isdigit():
                raise ValueError(f"pruning_schedule key {k!r} is not a block index")
            k = int(k)
        if "keep_ratio" not in cfg:
            raise KeyError("keep_ratio")
        out[int(k)] = cfg
    return out


def _is_identity(m) -> bool:
    return m is None or isinstance(m, nn.Identity) or (isinstance(m, nn.Dropout) and m.p == 0.0)


def _is_layer_norm(m, C: int) -> bool:
    return isinstance(m, nn.LayerNorm) and tuple(m.normalized_shape) == (C,) and m.weight is not None and m.bias is not None


def _is_layer_scale(m, C: int) -> bool:
    """timm's LayerScale (x * gamma): a module of that name whose only parameter is ``gamma`` [C] and that holds nothing else."""
    if type(m).__name__ != "LayerScale" or list(m.children()) or list(m.buffers()):
        return False
    params = dict(m.named_parameters())
    return list(params) == ["gamma"] and tuple(params["gamma"].shape) == (C,)


AUTO_GRAPH_MAX_ROWS = 16384       # batch x tokens up to which forward() replays a CUDA graph by default


class RAJNIViTWrapper(nn.Module):
    def __init__(self, base_model: nn.Module, pruning_schedule: Dict[int, Dict]):
        super().__init__()
        self.m = base_model
        self.blocks = base_model.blocks
        self.pruning_schedule = pruning_schedule
        sched = _normalise_schedule(pruning_schedule)

        for i, blk in enumerate(self.blocks):
            if i in sched:
                cfg = sched[i]
                blk.attn = RAJNIAttention(blk.attn, keep_ratio=cfg["keep_ratio"], update=cfg.get("update", True))
                blk.has_pruner = True
            else:
                blk.has_pruner = False

        self._last_stats = None
        self._last_keep_idx: List[Optional[torch.Tensor]] = []
        self._packs = PackCache()
        self._ws = {}
        self._graphs = {}
        self._param_list = None
        # None = automatic: replay a captured CUDA graph when the batch is small enough to be launch-bound
        env = os.environ.get("RAJNI_CUDA_GRAPH", "")
        self.use_cuda_graph: Optional[bool] = None if env == "" else env != "0"
        self.prefix = 1                  # leading tokens that are always kept (set by _validate: 2 for a distilled DeiT)
        self.no_embed_class = False      # pos_embed covers the patches only (DeiT-III)
        self.pre_norm = False            # norm_pre LayerNorm after the embedding (CLIP)
        self.avg_pool = False            # head on fc_norm(mean of the patch tokens) (global_pool='avg', MAE)
        self.headless = False            # head = Identity: forward returns the features the head would read (num_classes=0)
        self.input_norm: Optional[tuple] = None       # (mean[3], std[3]) for uint8 images, see set_input_normalization
        # Stream-K tail of the fc2 GEMMs (gemm_tcgen05.cu): +1.4 % at 32 images per GPU, nothing at 64 and above.  OFF by default
        # because the fp32 summation order of a split tile depends on the tile count, i.e. on the batch size: without it an
        # image's logits are bit-identical whatever batch it is evaluated in (tests/test_gpu_e2e.py::test_full_batch_properties).
        self.stream_k: bool = os.environ.get("RAJNI_STREAM_K", "0") == "1"
        self._validate()

    def set_input_normalization(self, mean, std) -> "RAJNIViTWrapper":
        """Extension (not in the reference): accept raw uint8 pixels [B,3,S,S] and apply the loader's ToTensor + Normalize
        (run.py:62-70) inside the patch kernel - a quarter of the host-to-device bytes of fp32 images, same logits."""
        mean, std = tuple(float(v) for v in mean), tuple(float(v) for v in std)
        if len(mean) != 3 or len(std) != 3 or min(std) <= 0:
            raise ValueError("mean and std must have three entries, std positive")
        self.input_norm = (mean, std)
        self._graphs = {}
        return self

    # ------------------------------------------------------------------ contract checks
    def _validate(self):
        m = self.m
        proj = getattr(m.patch_embed, "proj", None)
        if not isinstance(proj, nn.Conv2d):
            raise NotImplementedError("patch_embed.proj must be Conv2d(3, C, kernel=p, stride=p)")
        p = proj.kernel_size[0]
        if (proj.kernel_size != (p, p) or proj.stride != (p, p) or p % 8 or proj.in_channels != 3
                or proj.padding != (0, 0) or proj.dilation != (1, 1) or proj.groups != 1):
            raise NotImplementedError(f"patch_embed.proj is Conv2d(in={proj.in_channels}, kernel={proj.kernel_size}, "
                                      f"stride={proj.stride}); supported: Conv2d(3, C, kernel=p, stride=p) with p a multiple of 8 "
                                      f"(8, 16, 24, 32, ...)")
        self.patch = p
        if not _is_identity(getattr(m.patch_embed, "norm", None)):
            raise NotImplementedError("patch_embed.norm is not supported")
        if not _is_identity(getattr(m, "patch_drop", None)):
            raise NotImplementedError(f"patch_drop = {type(m.patch_drop).__name__} is not supported")
        C = proj.out_channels
        # pre-norm stem (CLIP): a LayerNorm over the embedded tokens before block 0
        norm_pre = getattr(m, "norm_pre", None)
        if not _is_identity(norm_pre) and not _is_layer_norm(norm_pre, C):
            raise NotImplementedError(f"norm_pre = {type(norm_pre).__name__} is not supported (Identity or an affine LayerNorm [C])")
        self.pre_norm = not _is_identity(norm_pre)
        # head: the class token through `norm`, or the mean of the patch tokens through `fc_norm` (MAE fine-tunes)
        pool, fc_norm = getattr(m, "global_pool", "token"), getattr(m, "fc_norm", None)
        if pool == "avg":
            if getattr(m, "dist_token", None) is not None:
                raise NotImplementedError("global_pool='avg' with a distillation token is not supported")
            if _is_identity(fc_norm):
                raise NotImplementedError("global_pool='avg' without fc_norm (timm fc_norm=False) is not supported")
            if not _is_layer_norm(fc_norm, C):
                raise NotImplementedError(f"fc_norm = {type(fc_norm).__name__} is not supported (an affine LayerNorm [C])")
            if not _is_identity(m.norm):
                raise NotImplementedError(f"fc_norm together with norm = {type(m.norm).__name__} is not supported "
                                          "(timm's avg-pooled models have norm = Identity)")
        elif pool == "token":
            if not _is_identity(fc_norm):
                raise NotImplementedError(f"fc_norm = {type(fc_norm).__name__} with global_pool='token' is not supported")
            if not isinstance(m.norm, nn.LayerNorm):
                raise NotImplementedError("norm must be LayerNorm")
        else:
            raise NotImplementedError(f"global_pool={pool!r} is not supported ('token' or 'avg')")
        self.avg_pool = pool == "avg"
        if not isinstance(m.head, nn.Linear) and not _is_identity(m.head):
            raise NotImplementedError(f"head = {type(m.head).__name__} is not supported (Linear, or Identity for a headless model)")
        self.headless = _is_identity(m.head)
        # prefix tokens: CLS, or CLS + distillation token (distilled DeiT); register tokens are not supported
        if getattr(m, "cls_token", None) is None:
            raise NotImplementedError("a class token (cls_token) is required")
        if getattr(m, "reg_token", None) is not None or getattr(m, "num_reg_tokens", 0):
            raise NotImplementedError("register tokens (reg_token) are not supported")
        dist, head_dist = getattr(m, "dist_token", None), getattr(m, "head_dist", None)
        prefix = int(getattr(m, "num_prefix_tokens", 1))
        if dist is not None:
            if self.headless:
                raise NotImplementedError("a dist_token with head = Identity (headless) is not supported: timm would return the "
                                          "mean of the normalised class and distillation tokens")
            if not isinstance(head_dist, nn.Linear) or head_dist.weight.shape != m.head.weight.shape:
                raise NotImplementedError("a dist_token needs head_dist, a Linear of the head's shape")
            if prefix != 2:
                raise NotImplementedError(f"num_prefix_tokens = {prefix} with a dist_token: expected 2 (CLS + distillation)")
            if getattr(m, "distilled_training", False):
                raise NotImplementedError("distilled_training (the (x, x_dist) training output) is not supported")
        elif head_dist is not None and not _is_identity(head_dist):
            raise NotImplementedError("head_dist without a dist_token is not supported")
        elif prefix != 1:
            raise NotImplementedError(f"num_prefix_tokens = {prefix}: only CLS (1) or CLS + dist_token (2) are supported")
        self.prefix = prefix
        self.no_embed_class = bool(getattr(m, "no_embed_class", False))
        for i, blk in enumerate(self.blocks):
            for name in ("ls1", "ls2"):
                ls = getattr(blk, name, None)
                if not _is_identity(ls) and not _is_layer_scale(ls, C):
                    raise NotImplementedError(f"blocks[{i}].{name} = {type(ls).__name__} is not supported "
                                              "(Identity or LayerScale with gamma [C])")
            for name in ("drop_path1", "drop_path2"):
                if not _is_identity(getattr(blk, name, None)):
                    raise NotImplementedError(f"blocks[{i}].{name} = {type(getattr(blk, name)).__name__} is not supported")
            attn = blk.attn
            if attn.num_heads * 64 != C:
                raise NotImplementedError(f"blocks[{i}]: head dim must be 64 (C={C}, heads={attn.num_heads})")
            if abs(float(attn.scale) - 0.125) > 1e-12:
                raise NotImplementedError(f"blocks[{i}]: attention scale {attn.scale} != 64**-0.5")
            for name in ("q_norm", "k_norm"):
                if not _is_identity(getattr(attn, name, None)):
                    raise NotImplementedError(f"blocks[{i}].attn.{name} is not supported")
            act = blk.mlp.act
            if not isinstance(act, nn.GELU) or getattr(act, "approximate", "none") != "none":
                raise NotImplementedError(f"blocks[{i}].mlp.act = {type(act).__name__} is not supported: "
                                          f"blocks[{i}].mlp.act must be exact (erf) nn.GELU")
            if not _is_identity(getattr(blk.mlp, "norm", None)):
                raise NotImplementedError(f"blocks[{i}].mlp.norm is not supported")
            if not isinstance(blk.norm1, nn.LayerNorm) or not isinstance(blk.norm2, nn.LayerNorm):
                raise NotImplementedError(f"blocks[{i}]: norm1/norm2 must be LayerNorm")
            if blk.has_pruner:
                blk.attn.num_prefix_tokens = prefix

    def _apply(self, fn, *a, **kw):
        self._packs.clear()
        self._ws.clear()
        self._graphs = {}
        self._param_list = None
        return super()._apply(fn, *a, **kw)

    def load_state_dict(self, *a, **kw):
        self._graphs = {}
        self._param_list = None
        return super().load_state_dict(*a, **kw)

    def get_last_stats(self):
        return self._last_stats

    def _distilled(self) -> bool:
        return getattr(self.m, "dist_token", None) is not None

    # ------------------------------------------------------------------ workspace
    def _workspace(self, B: int, S: int, dev: torch.device):
        key = (B, S, dev, self.stream_k)
        ws = self._ws.get(key)
        if ws is not None:
            return ws
        m = self.m
        C = m.patch_embed.proj.out_channels
        p = self.patch
        G = S // p
        P = G * G
        P0 = self.prefix
        N0 = P + P0
        pos_off = 0 if self.no_embed_class else P0          # pos_embed row of patch 0
        if m.pos_embed.shape[1] < P + pos_off:
            raise ValueError(f"pos_embed has {m.pos_embed.shape[1]} positions, input needs {P + pos_off}")
        hidden = max(blk.mlp.fc1.out_features for blk in self.blocks)
        bf = dict(device=dev, dtype=torch.bfloat16)
        idx = torch.arange(B * P, device=dev, dtype=torch.int32)
        ws = dict(
            P=P, N0=N0, C=C,
            cols=torch.empty((B * P, 3 * p * p), **bf),
            xa=torch.empty((B * N0, C), **bf), xb=torch.empty((B * N0, C), **bf),
            qkv=torch.empty((B * N0, 3 * C), **bf),
            att=torch.empty((B * N0, C), **bf), hid=torch.empty((B * N0, hidden), **bf),
            # final-norm rows feeding the head: CLS, or [CLS | distillation token] side by side (K = 2C)
            cls=torch.empty((B, (2 if self._distilled() else 1) * C), **bf),
            embed_out_map=((idx // P) * N0 + P0 + idx % P).to(torch.int32),
            embed_pos_map=(pos_off + idx % P).to(torch.int32),
            # LayerNorm partial sums (sum, sum of squares) of the rows of x, one slot per (n-tile, column half)
            # of the GEMM that produced them; consumed by the LN-folded qkv / fc1 GEMMs
            stat_slots=ops.row_stats_slots(C),
            stats=torch.zeros((ops.row_stats_slots(C), B * N0, 2), device=dev, dtype=torch.float32),
            sel={},
            # stream-K scratch of the long-K GEMMs (fc2), only when asked for: owned here like every other pointer a captured
            # graph bakes in
            gemm_ws=ops.gemm_workspace(dev) if self.stream_k else None,
            # scratch of the split score path (small batches, and sequences too long for the one-launch kernel at any batch):
            # owned here, so a captured graph's pointer lives with the graph.  Sized for N0, the longest sequence of the step.
            score_ws=(torch.empty(max(ops.score_workspace_bytes(B, N0, C, blk.attn.num_heads) for blk in self.blocks),
                                  device=dev, dtype=torch.uint8)
                      if B <= ops.SPLIT_SCORE_MAX_BATCH or any(ops.needs_score_workspace(N0, blk.attn.num_heads) for blk in self.blocks)
                      else None),
        )
        self._ws = {key: ws}        # keep one shape resident
        self._graphs = {}           # a captured graph points into the workspace it was captured with
        return ws

    # ------------------------------------------------------------------ forward
    @torch.no_grad()
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """model.py:30-69.  The launch sequence of a given input shape can be captured once into a CUDA graph and replayed:
        the 68 launches of a step cost ~13 us of host time each, which dominates small batches (vit_tiny at batch 8:
        0.88 -> 0.53 ms per step).  ``use_cuda_graph`` = None (default) replays when the batch has at most
        ``AUTO_GRAPH_MAX_ROWS`` token rows, True / False force it (RAJNI_CUDA_GRAPH=1 / 0 in the environment do the same).
        A captured graph is dropped when any parameter changes (storage or version), on ``.to()`` / ``.bfloat16()`` /
        ``load_state_dict`` and when the input normalisation changes; results are bit-identical to the eager sequence."""
        if x.device.type == "cuda" and x.device.index is not None and x.device.index != torch.cuda.current_device():
            with torch.cuda.device(x.device):          # the C ABI launches on the current device
                return self.forward(x)
        use = self.use_cuda_graph
        if use is None and x.dim() == 4:
            use = x.shape[0] * ((x.shape[2] // self.patch) * (x.shape[3] // self.patch) + self.prefix) <= AUTO_GRAPH_MAX_ROWS
        if not use or x.device.type != "cuda" or x.dim() != 4 or ops._prof is not None:      # (the per-kernel profiler times eager launches)
            return self._forward_eager(x)
        # what _forward_eager reads besides the input: the schedule of the pruned blocks (attention.py:25-32) ...
        sched = tuple((blk.attn.keep_ratio, blk.attn.update) if blk.has_pruner else None for blk in self.blocks)
        key = (tuple(x.shape), x.dtype, x.device, self.training, sched, self.input_norm, self.stream_k)
        # ... and the parameters.  Storage changes go through _apply / load_state_dict (which drop the graphs); in-place
        # updates bump the tensors' version counters, summed here over a parameter list that is built once.
        if self._param_list is None:
            self._param_list = list(self.parameters())
        wsig = sum(q._version for q in self._param_list)
        entry = self._graphs.get(key)
        if entry is None or entry[5] != wsig:
            x_static = x.clone()
            self._forward_eager(x_static)                       # builds packs and workspace, warms every kernel
            torch.cuda.synchronize(x.device)
            graph = torch.cuda.CUDAGraph()
            # thread-local capture mode: a DataLoader's pin-memory thread may call into CUDA while this thread captures
            with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                y_static = self._forward_eager(x_static)
            entry = (graph, x_static, y_static, self._last_stats, self._last_keep_idx, wsig)
            self._graphs = {key: entry}                         # one shape resident, like the workspace
        graph, x_static, y_static, stats, keep, _ = entry
        x_static.copy_(x)
        graph.replay()
        self._last_stats, self._last_keep_idx = stats, keep
        return y_static.clone()

    @torch.no_grad()
    def _forward_eager(self, x: torch.Tensor) -> torch.Tensor:
        if x.dim() != 4 or x.shape[1] != 3 or x.shape[2] != x.shape[3] or x.shape[2] % self.patch:
            raise ValueError(f"expected images [B,3,S,S] with S a multiple of the patch size {self.patch}, got {tuple(x.shape)}")
        if x.device.type != "cuda":
            raise RuntimeError("RAJNIViTWrapper (B200) runs on CUDA tensors only; there is no CPU path")
        last = self.m.head if not self.headless else self.m.fc_norm if self.avg_pool else self.m.norm      # the last module with weights
        if self.m.pos_embed.device != x.device or last.weight.device != x.device:
            raise RuntimeError(f"Expected all tensors to be on the same device: input on {x.device}, model on "
                               f"{self.m.pos_embed.device} (call .to(device) on the wrapper first)")
        if self.training:
            for blk in self.blocks:
                for d in (blk.attn.proj_drop, getattr(blk.mlp, "drop1", None), getattr(blk.mlp, "drop2", None)):
                    if isinstance(d, nn.Dropout) and d.p > 0:
                        raise NotImplementedError("dropout in training mode is not supported (inference path)")
        m = self.m
        out_dtype = x.dtype if x.dtype.is_floating_point else torch.float32
        if x.dtype == torch.uint8:
            if self.input_norm is None:
                raise TypeError("uint8 images need set_input_normalization(mean, std) first (the reference takes normalised floats)")
        elif x.dtype not in (torch.float32, torch.bfloat16):
            x = x.float()
        x = x.contiguous()
        B, _, S, _ = x.shape
        ws = self._workspace(B, S, x.device)
        P, N, C = ws["P"], ws["N0"], ws["C"]
        pk = self._packs

        # ---- patch + CLS + pos (model.py:31-37): im2col, then one GEMM whose epilogue adds
        #      bias and pos_embed and scatters into rows P0..P0+P-1 of each image (P0 = 1, or 2 with a distillation token)
        pe_w, pe_b = pk.linear(m.patch_embed.proj)
        if pe_b is None:                # CLIP: no patch bias.  A zero bias keeps the GEMM's bias + residual epilogue, the one
            pe_b = pk.tensors(("pe_zero_bias",), (m.patch_embed.proj.weight,),          # that also writes row statistics
                              lambda: torch.zeros(C, device=x.device, dtype=torch.float32))
        P0 = self.prefix
        dist = getattr(m, "dist_token", None)

        def _pos_pack():
            pos_ = m.pos_embed.detach()[0, : P + (0 if self.no_embed_class else P0)].to(torch.bfloat16).contiguous()
            tok = [m.cls_token.detach()[0, 0]] + ([dist.detach()[0, 0]] if dist is not None else [])
            if not self.no_embed_class:                     # the tokens' own positions; DeiT-III adds none to its class token
                tok = [t + m.pos_embed.detach()[0, r] for r, t in enumerate(tok)]
            rows = torch.stack(tok).to(torch.bfloat16).contiguous()
            r32 = rows.to(torch.float32)
            sums = [float(r32[r].sum()) for r in range(P0)]               # one full reduction per row
            sqs = [float((r32[r] * r32[r]).sum()) for r in range(P0)]
            return pos_, rows, sums if P0 > 1 else sums[0], sqs if P0 > 1 else sqs[0]

        pos, prefix_rows, pre_sum, pre_sumsq = pk.tensors(("pos", P), (m.pos_embed, m.cls_token, dist), _pos_pack)
        cur, nxt = ws["xa"], ws["xb"]
        stats, slots = ws["stats"], ws["stat_slots"]
        kpe = ws["cols"].shape[1]                                                   # 3 p^2
        ops.patch_im2col(x, self.patch, ws["cols"], prefix_rows, cur, C, row_stats=stats, stats_slots=slots,
                         cls_sum=pre_sum, cls_sumsq=pre_sumsq, norm=self.input_norm if x.dtype == torch.uint8 else None,
                         prefix=P0)
        ops.gemm(ws["cols"], pe_w, pe_b, B * P, C, kpe, residual=pos, ldres=C, res_row_map=ws["embed_pos_map"],
                 out=cur, ldd=C, out_row_map=ws["embed_out_map"], row_stats=stats, tag="embed")
        if self.pre_norm:               # x = norm_pre(x) in place, with the row statistics block 0's LN-folded qkv GEMM reads
            gp, bp, ep = pk.norm(m.norm_pre)
            ops.layernorm(cur, gp, bp, ep, B * N, C, out=cur, row_stats=stats, stats_slots=slots)

        # Zig-zag traversal: every persistent kernel walks its row tiles in the direction opposite to the kernel that
        # produced its main operand, so it starts on the rows that kernel wrote last and that still sit in L2.
        zig = os.environ.get("RAJNI_NO_ZIGZAG") is None       # A/B switch for profiling
        rev = zig                      # the embed GEMM walked forward
        scores = None
        token_counts = []
        keep_log: List[Optional[torch.Tensor]] = []
        for i, blk in enumerate(self.blocks):
            token_counts.append(N)                                                   # model.py:43
            H = blk.attn.num_heads
            # norm1 / norm2 are folded into the qkv / fc1 GEMMs: x itself is the A operand, the row statistics
            # come from the epilogue of whichever GEMM stored x (embed, proj or fc2)
            # LayerScale (DeiT-III) is folded into the GEMMs that feed the residual: proj (ls1) and fc2 (ls2)
            qw, qb, qsum, e1 = pk.linear_ln(blk.attn.qkv, blk.norm1)
            ls1, ls2 = getattr(blk, "ls1", None), getattr(blk, "ls2", None)
            pw, pb = pk.linear(blk.attn.proj) if _is_identity(ls1) else pk.linear_ls(blk.attn.proj, ls1)
            f1w, f1b, f1sum, e2 = pk.linear_ln(blk.mlp.fc1, blk.norm2)
            f2w, f2b = pk.linear(blk.mlp.fc2) if _is_identity(ls2) else pk.linear_ls(blk.mlp.fc2, ls2)
            hidden = f1w.shape[0]
            M = B * N
            ops.gemm(cur, qw, qb, M, 3 * C, C, out=ws["qkv"], ln=(stats, slots, qsum, e1), tag="qkv", reverse=rev)   # model.py:51 + attention.py:22
            if blk.has_pruner:
                attn: RAJNIAttention = blk.attn
                keep = keep_count(N, attn.keep_ratio, P0)                             # attention.py:31-32
                if keep > N - P0:
                    raise RuntimeError("selected index k out of range")               # attention.py:35
                Np = keep + P0
                sel = ws["sel"].get(i)
                if sel is None or sel[0].shape[1] != Np:
                    sel = (torch.empty((B, Np), device=x.device, dtype=torch.int32),
                           torch.empty((B, Np), device=x.device, dtype=torch.float32),
                           torch.empty((B * Np,), device=x.device, dtype=torch.int32))
                    ws["sel"][i] = sel
                keep_idx, next_scores, row_map = sel
                if attn.update or scores is None:                                     # attention.py:25-28
                    ops.score_select(ws["qkv"][: B * N].view(B, N, 3 * C), H, keep, keep_idx=keep_idx, next_scores=next_scores,
                                     row_map=row_map, workspace=ws["score_ws"], prefix=P0)
                else:
                    ops.select(scores, keep, keep_idx=keep_idx, next_scores=next_scores, row_map=row_map, prefix=P0)
                if Np > ops.LONG_SEQ and "qkvc" not in ws:                             # compaction buffer, long sequences only
                    ws["qkvc"] = torch.empty((B * ws["N0"], 3 * C), device=x.device, dtype=torch.bfloat16)
                ops.attention(ws["qkv"], row_map, B, N, Np, C, H, float(attn.scale), out=ws["att"], reverse=zig and not rev,
                              compact=ws.get("qkvc"))
                # proj + gathered residual: x_new[b,j] = x[b, keep_idx[b,j]] + proj(att)   model.py:55-58
                ops.gemm(ws["att"], pw, pb, B * Np, C, C, residual=cur, ldres=C, res_row_map=row_map, out=nxt, ldd=C,
                         row_stats=stats, tag="proj", reverse=rev)
                cur, nxt = nxt, cur
                scores = next_scores                                                  # attention.py:58
                keep_log.append(keep_idx)
                N = Np
                M = B * N
            else:
                ops.attention(ws["qkv"], None, B, N, N, C, H, float(blk.attn.scale), out=ws["att"], reverse=zig and not rev)
                ops.gemm(ws["att"], pw, pb, M, C, C, residual=cur, ldres=C, out=cur, ldd=C, row_stats=stats, tag="proj", reverse=rev)   # in place
                scores = None                                                         # model.py:63
                keep_log.append(None)
            ops.gemm(cur, f1w, f1b, M, hidden, C, gelu=True, out=ws["hid"], ldd=hidden,
                     ln=(stats, slots, f1sum, e2), tag="fc1", reverse=zig and not rev)                                    # model.py:59 (norm2 + fc1 + GELU)
            ops.gemm(ws["hid"], f2w, f2b, M, C, hidden, residual=cur, ldres=C, out=cur, ldd=C, row_stats=stats, tag="fc2", reverse=rev,
                     workspace=ws["gemm_ws"] if self.stream_k else None)
            rev = zig and not rev

        # ---- final norm on the CLS rows only (LayerNorm is row-wise) + head   model.py:65-66
        if self.headless:               # the head's input is the output, stored in fp32 by the kernel that computes it
            logits = torch.empty((B, C), device=x.device, dtype=torch.float32)
            if self.avg_pool:
                ops.mean_pool_layernorm(cur, B, N, C, *pk.norm(m.fc_norm), prefix=P0, out=logits)
            else:
                ops.layernorm(cur, *pk.norm(m.norm), B, C, in_row_stride=N * C, out=logits)
        elif self.avg_pool:             # timm forward_head, global_pool='avg': head(fc_norm(mean of the kept patch tokens))
            gf, bf_, ef = pk.norm(m.fc_norm)
            hw, hb = pk.linear(m.head)
            ops.mean_pool_layernorm(cur, B, N, C, gf, bf_, ef, prefix=P0, out=ws["cls"])
            logits = ops.gemm(ws["cls"], hw, hb, B, hw.shape[0], C, out_f32=True, tag="head")
        elif dist is None:
            gn, bn, en = pk.norm(m.norm)
            hw, hb = pk.linear(m.head)
            ops.layernorm(cur, gn, bn, en, B, C, in_row_stride=N * C, out=ws["cls"])
            logits = ops.gemm(ws["cls"], hw, hb, B, hw.shape[0], C, out_f32=True, tag="head")
        else:
            # distilled: (head(LN(x0)) + head_dist(LN(x1))) / 2 as ONE GEMM over [LN(x0) | LN(x1)] (K = 2C) with the weights
            # [W_head | W_dist] / 2 (halving is exact in bf16) and the bias (b + b_dist) / 2
            gn, bn, en = pk.norm(m.norm)
            hw, hb = pk.tensors(("head2",), (m.head.weight, m.head.bias, m.head_dist.weight, m.head_dist.bias), self._head_pack)
            for r in range(2):
                ops.layernorm(cur, gn, bn, en, B, C, in_row_stride=N * C, in_offset=r * C, out=ws["cls"],
                              out_row_stride=2 * C, out_offset=r * C)
            logits = ops.gemm(ws["cls"], hw, hb, B, hw.shape[0], 2 * C, out_f32=True, tag="head")

        self._last_stats = {"token_counts": token_counts}                            # model.py:68
        self._last_keep_idx = keep_log
        return logits if out_dtype == torch.float32 else logits.to(out_dtype)

    def _head_pack(self):
        m = self.m
        w = torch.cat([m.head.weight.detach(), m.head_dist.weight.detach()], dim=1).to(torch.bfloat16) / 2
        b = [t.detach().to(torch.float32) if t is not None else torch.zeros(m.head.out_features, device=m.head.weight.device)
             for t in (m.head.bias, m.head_dist.bias)]
        return w.contiguous(), ((b[0] + b[1]) / 2).contiguous()
