"""Config-driven decoder-only transformer shared by the Llama / Qwen2 / Qwen3 / Mixtral / Qwen-MoE /
ChatGLM families (the per-architecture modules in this package only translate HF configs and
checkpoint names into a `ModelSpec`).

Block dataflow (B200-first, differs from the reference's module-per-op structure):

    normed, residual ──► QKV GEMM ──► fused [q/k-norm + RoPE + paged-KV write] ──► paged attention
        ──► O-proj GEMM ⊕ TP-reduce ⊕ residual-add ⊕ RMSNorm        (one TPComm call)
        ──► gate/up GEMM with SiLU-gate epilogue  |  MoE block
        ──► down GEMM ⊕ TP-reduce ⊕ residual-add ⊕ *next layer's* RMSNorm   (one TPComm call)

so every row-parallel GEMM is handed to the TP strategy together with the norm that consumes it —
that is what lets `FusedTPComm` run GEMM⊕reduce-scatter and all-gather⊕GEMM on token-sharded
activations. Reference equivalents: gllm/models/qwen2.py:36-261, llama.py, qwen3.py.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Callable, Dict, List, Optional

import torch
from torch import nn

from gllm_b200.layers import functional as Fn
from gllm_b200.layers.rotary import RopeSpec, build_rope
from gllm_b200.models import weight_utils as wu
from gllm_b200.ops import ref
from gllm_b200.parallel import state as ps
from gllm_b200.parallel.tp import TPComm


_NVTX = __import__("os").environ.get("GLLM_NVTX", "0") == "1"   # per-layer NVTX ranges for nsys / ncu --nvtx


@dataclass
class MoESpec:
    num_experts: int
    top_k: int
    intermediate_size: int
    norm_topk_prob: bool = True
    shared_intermediate_size: int = 0
    shared_gate: bool = False           # sigmoid-gated shared expert (Qwen2-MoE)
    scoring: str = "softmax"            # or "sigmoid" (DeepSeek-V3)
    n_group: int = 0
    topk_group: int = 0
    routed_scaling: float = 1.0
    has_bias_correction: bool = False


@dataclass
class ModelSpec:
    arch: str
    hidden_size: int
    num_layers: int
    num_heads: int
    num_kv_heads: int
    head_dim: int
    intermediate_size: int
    vocab_size: int
    rms_eps: float = 1e-6
    qkv_bias: bool = False
    o_bias: bool = False
    qk_norm: bool = False
    tie_word_embeddings: bool = False
    max_position: int = 8192
    rope_theta: float = 10000.0
    rope_scaling: Optional[dict] = None
    rot_dim: Optional[int] = None
    rope_neox: bool = True
    moe: Optional[MoESpec] = None
    moe_layers: Optional[List[int]] = None  # global layer ids that are MoE (None + moe => all)
    dtype: torch.dtype = torch.bfloat16
    use_mla: bool = False
    # HF checkpoint name templates
    names: Dict[str, str] = field(default_factory=dict)
    eos_token_id: Optional[object] = None
    extra: dict = field(default_factory=dict)
    quant: Optional[str] = None  # "fp8": block-scaled e4m3 linears (HF quantization_config, 128x128 blocks)

    def is_moe_layer(self, layer_id: int) -> bool:
        if self.moe is None:
            return False
        return True if self.moe_layers is None else layer_id in self.moe_layers


DEFAULT_NAMES = {
    "embed": "model.embed_tokens.weight",
    "final_norm": "model.norm.weight",
    "lm_head": "lm_head.weight",
    "layer": "model.layers.{i}.",
    "input_norm": "input_layernorm.weight",
    "post_norm": "post_attention_layernorm.weight",
    "q": "self_attn.q_proj", "k": "self_attn.k_proj", "v": "self_attn.v_proj", "o": "self_attn.o_proj",
    "q_norm": "self_attn.q_norm.weight", "k_norm": "self_attn.k_norm.weight",
    "gate": "mlp.gate_proj", "up": "mlp.up_proj", "down": "mlp.down_proj",
    "router": "mlp.gate.weight",
    "expert": "mlp.experts.{e}.", "e_gate": "gate_proj.weight", "e_up": "up_proj.weight", "e_down": "down_proj.weight",
    "shared": "mlp.shared_expert.", "shared_gate": "mlp.shared_expert_gate.weight",
}


def _param(*shape, dtype, device, std=0.02, fill=None):
    if fill is not None:
        t = torch.full(shape, fill, dtype=dtype, device=device)
    else:
        t = torch.empty(shape, dtype=dtype, device=device)
    return nn.Parameter(t, requires_grad=False)


def _linear_params(n: int, k: int, spec: ModelSpec, device):
    """(weight, scale_inv | None): bf16 [n, k], or e4m3 [n, k] + fp32 block scales for fp8 checkpoints."""
    if spec.quant == "fp8" and k % 128 == 0:      # activations are quantised per 128-wide K group
        w = nn.Parameter(torch.zeros(n, k, dtype=torch.float8_e4m3fn, device=device), requires_grad=False)
        s = nn.Parameter(torch.ones((n + 127) // 128, (k + 127) // 128, dtype=torch.float32, device=device),
                         requires_grad=False)
        return w, s
    return _param(n, k, dtype=spec.dtype, device=device), None


def _qw(w, s):
    """Weight handle passed to the linear ops: plain tensor, or (e4m3, scale_inv) for fp8."""
    return w if s is None else (w, s)


def _store_linear(w_param, s_param, w: torch.Tensor):
    """Copy a (sharded) weight into its parameter; fp8 parameters are block-quantised here (128x128 blocks,
    scale_inv = amax / 448). Re-quantising the de-quantised tensor of an fp8 checkpoint is lossless as long
    as shard boundaries fall on block boundaries (they do: head_dim 128, intermediate % 128 == 0)."""
    if s_param is None:
        w_param.data.copy_(w)
        return
    w = w.float()
    n, k = w.shape
    nb, kb = (n + 127) // 128, (k + 127) // 128
    wp = torch.zeros(nb * 128, kb * 128, dtype=torch.float32, device=w.device)
    wp[:n, :k] = w
    blk = wp.view(nb, 128, kb, 128)
    sc = (blk.abs().amax(dim=(1, 3)) / 448.0).clamp_min(1e-12)
    q = (blk / sc.view(nb, 1, kb, 1)).view(nb * 128, kb * 128)[:n, :k].to(torch.float8_e4m3fn)
    w_param.data.copy_(q)
    s_param.data.copy_(sc)


class Attention(nn.Module):
    def __init__(self, spec: ModelSpec, layer_id: int, rope: RopeSpec, device):
        super().__init__()
        st = ps.get_state()
        tp, tr = st.tp_size, st.tp_rank
        self.layer_id = layer_id
        self.head_dim = spec.head_dim
        assert spec.num_heads % tp == 0, f"{spec.num_heads} heads not divisible by tp={tp}"
        self.num_heads = spec.num_heads // tp
        _, self.num_kv_heads = wu.kv_head_range(spec.num_kv_heads, tr, tp)
        self.q_size = self.num_heads * self.head_dim
        self.kv_size = self.num_kv_heads * self.head_dim
        self.scaling = self.head_dim ** -0.5 * rope.attn_mscale
        self.rope = rope
        self.eps = spec.rms_eps
        h, dt = spec.hidden_size, spec.dtype
        self.qkv_w, self.qkv_ws = _linear_params(self.q_size + 2 * self.kv_size, h, spec, device)
        self.qkv_b = _param(self.q_size + 2 * self.kv_size, dtype=dt, device=device) if spec.qkv_bias else None
        self.o_w, self.o_ws = _linear_params(h, self.q_size, spec, device)
        self.o_b = _param(h, dtype=dt, device=device) if spec.o_bias else None
        self.q_norm_w = _param(self.head_dim, dtype=dt, device=device, fill=1.0) if spec.qk_norm else None
        self.k_norm_w = _param(self.head_dim, dtype=dt, device=device, fill=1.0) if spec.qk_norm else None

    def qkv_proj(self, h: torch.Tensor, tpc: TPComm) -> torch.Tensor:
        return tpc.col_linear(h, _qw(self.qkv_w, self.qkv_ws), self.qkv_b)

    def forward(self, inp, h: torch.Tensor, kv_cache, tpc: TPComm, qkv: Optional[torch.Tensor] = None) -> torch.Tensor:
        """h [T, H] (normed) -> attention output [T, q_size] (input of the row-parallel O-proj).
        `qkv` may be supplied pre-computed (tile-streamed pipeline input)."""
        if qkv is None:
            qkv = self.qkv_proj(h, tpc)
        t = qkv.shape[0]
        d = self.head_dim
        q = qkv[:, : self.q_size].view(t, self.num_heads, d)
        k = qkv[:, self.q_size: self.q_size + self.kv_size].view(t, self.num_kv_heads, d)
        v = qkv[:, self.q_size + self.kv_size:].view(t, self.num_kv_heads, d)
        if kv_cache is None:
            # memory-profiling run without a KV cache (reference: gllm/layers/attention.py:34-36)
            return qkv[:, : self.q_size].contiguous()
        kc, vc = kv_cache.k_cache[self.layer_id], kv_cache.v_cache[self.layer_id]
        Fn.rope_kv_write(q, k, v, inp.positions, self.rope.cos_sin, self.rope.rot_dim, self.rope.neox,
                         self.q_norm_w, self.k_norm_w, self.eps, kc, vc, inp.slot_mapping,
                         self.rope.mrope_section)
        return Fn.paged_attention(qkv[:, : self.q_size], kc, vc, inp, self.scaling, self.num_heads, d)


class DenseMLP(nn.Module):
    def __init__(self, hidden: int, intermediate: int, dtype, device, shard: bool = True,
                 spec: Optional[ModelSpec] = None):
        super().__init__()
        tp = ps.get_tp_size() if shard else 1
        assert intermediate % tp == 0
        self.inter = intermediate // tp
        fp8 = spec is not None and spec.quant == "fp8"
        # fused SiLU-gate epilogue needs the gate/up rows interleaved per 128 (bf16 kernel only)
        self.fused_act = self.inter % 128 == 0 and not fp8
        if fp8:
            self.gate_up_w, self.gate_up_ws = _linear_params(2 * self.inter, hidden, spec, device)
            self.down_w, self.down_ws = _linear_params(hidden, self.inter, spec, device)
        else:
            self.gate_up_w, self.gate_up_ws = _param(2 * self.inter, hidden, dtype=dtype, device=device), None
            self.down_w, self.down_ws = _param(hidden, self.inter, dtype=dtype, device=device), None

    def set_gate_up(self, gate_up: torch.Tensor):
        """gate_up [2*inter, H] = [gate rows; up rows] for this rank."""
        if self.fused_act:
            gate_up = ref.interleave_gate_up(gate_up, 128)
        _store_linear(self.gate_up_w, self.gate_up_ws, gate_up)

    def down_weight(self):
        return _qw(self.down_w, self.down_ws)

    def act(self, h: torch.Tensor, tpc: TPComm) -> torch.Tensor:
        if self.fused_act:
            return tpc.col_linear_silu_mul(h, self.gate_up_w)
        return Fn.silu_and_mul(tpc.col_linear(h, _qw(self.gate_up_w, self.gate_up_ws)))


class DecoderLayer(nn.Module):
    def __init__(self, spec: ModelSpec, layer_id: int, local_id: int, rope: RopeSpec, device, moe_factory=None):
        super().__init__()
        self.spec = spec
        self.layer_id = layer_id      # global index (weights)
        self.local_id = local_id      # index into this stage's KV cache
        dt, h = spec.dtype, spec.hidden_size
        self.input_norm_w = _param(h, dtype=dt, device=device, fill=1.0)
        self.post_norm_w = _param(h, dtype=dt, device=device, fill=1.0)
        self.attn = Attention(spec, local_id, rope, device)
        self.is_moe = spec.is_moe_layer(layer_id)
        if self.is_moe:
            self.mlp = moe_factory(spec, layer_id, device)
        else:
            self.mlp = DenseMLP(h, spec.intermediate_size, dt, device, spec=spec)

    def forward(self, inp, h: torch.Tensor, residual: torch.Tensor, kv_cache, tpc: TPComm,
                next_norm_w: Optional[torch.Tensor], qkv: Optional[torch.Tensor] = None):
        """h = RMSNorm'ed block input, residual = running residual stream.
        Returns (normed input of the next block, residual) — or (un-normed block output, residual)
        when `next_norm_w` is None (last layer of a non-final pipeline stage)."""
        eps = self.spec.rms_eps
        a = self.attn(inp, h, kv_cache, tpc, qkv=qkv)
        h, residual = tpc.row_linear_add_norm(a, _qw(self.attn.o_w, self.attn.o_ws), residual, self.post_norm_w, eps, self.attn.o_b)
        if self.is_moe:
            if next_norm_w is None:
                return tpc.all_reduce(self.mlp(tpc.materialize(h), tpc)), residual
            return tpc.moe_add_norm(self.mlp, h, residual, next_norm_w, eps)
        act = self.mlp.act(h, tpc)
        if next_norm_w is None:
            return tpc.row_linear(act, self.mlp.down_weight()), residual
        return tpc.row_linear_add_norm(act, self.mlp.down_weight(), residual, next_norm_w, eps)


class CausalLM(nn.Module):
    """This pipeline stage's slice of the model (+ embedding on the first stage, final norm and
    LM head on the last)."""

    ret_residual = True  # PP sends (hidden, residual)

    def __init__(self, spec: ModelSpec, device="cpu", moe_factory=None):
        super().__init__()
        self.spec = spec
        st = ps.get_state()
        self.device = torch.device(device)
        self.layers_range = ps.get_pp_layers(spec.num_layers)
        self.is_first, self.is_last = ps.is_first_pp_rank(), ps.is_last_pp_rank()
        self.tp_size, self.tp_rank = st.tp_size, st.tp_rank
        self.rope = build_rope(spec.head_dim, spec.max_position, spec.rope_theta, spec.rope_scaling, spec.rot_dim,
                               spec.rope_neox, device=device)
        dt, h = spec.dtype, spec.hidden_size
        self.vocab_padded = wu.pad_vocab(spec.vocab_size, self.tp_size)
        self.vocab_per_rank = self.vocab_padded // self.tp_size
        self.vocab_start = self.tp_rank * self.vocab_per_rank
        need_embed = self.is_first or (spec.tie_word_embeddings and self.is_last)
        self.embed_w = _param(self.vocab_per_rank, h, dtype=dt, device=device) if need_embed else None
        self.layers = nn.ModuleList([
            DecoderLayer(spec, gid, lid, self.rope, device, moe_factory)
            for lid, gid in enumerate(self.layers_range)])
        if self.is_last:
            self.final_norm_w = _param(h, dtype=dt, device=device, fill=1.0)
            self.lm_head_w = self.embed_w if spec.tie_word_embeddings else _param(self.vocab_per_rank, h, dtype=dt,
                                                                                   device=device)
        else:
            self.final_norm_w = self.lm_head_w = None

    # -- attributes the runner needs (reference: models/qwen2.py:183-258) -------------------------
    @property
    def num_layers(self): return len(self.layers)

    @property
    def num_kv_heads(self): return self.layers[0].attn.num_kv_heads if len(self.layers) else 0

    @property
    def head_dim(self): return self.spec.head_dim

    @property
    def hidden_size(self): return self.spec.hidden_size

    # -- forward ----------------------------------------------------------------------------------
    def embed(self, inp, tpc: TPComm) -> torch.Tensor:
        x = Fn.embedding(inp.tokens, self.embed_w, self.vocab_start, self.vocab_start + self.vocab_per_rank)
        return tpc.all_reduce(x)

    def forward(self, inp, kv_cache, tpc: TPComm, hidden: Optional[torch.Tensor] = None,
                residual: Optional[torch.Tensor] = None, inputs_embeds: Optional[torch.Tensor] = None,
                recv_tiles=None, deepstack=None):
        """First stage: tokens -> ... ; later stages: (hidden, residual) from the previous stage.
        Returns (hidden, residual): on the last stage `hidden` is the final-normed activation."""
        eps = self.spec.rms_eps
        n = len(self.layers)
        if self.is_first:
            x = inputs_embeds if inputs_embeds is not None else self.embed(inp, tpc)
            if n == 0:
                return x, None
            h, residual = tpc.first_norm(x, self.layers[0].input_norm_w, eps)
        qkv0 = None
        else_branch = not self.is_first
        if else_branch:
            if n == 0:
                if recv_tiles:
                    for _, _, works in recv_tiles:
                        for w in works:
                            w.wait()
                return hidden, residual
            if getattr(tpc, "fused", False):
                # fused TP inside a pipeline stage: the stage input arrives replicated; fold the previous stage's
                # block output into the residual stream, then enter the token-sharded dataflow exactly like the
                # embedding output does on the first stage (normed gather buffer + residual shard)
                if recv_tiles:
                    for _, _, works in recv_tiles:
                        for w in works:
                            w.wait()
                _, res_full = Fn.rmsnorm(hidden, self.layers[0].input_norm_w, eps, residual)
                h, residual = tpc.first_norm(res_full, self.layers[0].input_norm_w, eps)
            elif recv_tiles and len(recv_tiles) > 1 and hasattr(self.layers[0].attn, "qkv_proj"):
                # tile-streamed pipeline input: add+RMSNorm and the QKV GEMM run per row tile as the tiles
                # land, overlapping the NCCL transfer of the following tiles (SURVEY §2.4 X5)
                h = torch.empty_like(hidden)
                at = self.layers[0].attn
                for r0, r1, works in recv_tiles:
                    for w in works:
                        w.wait()  # stream-level wait on this tile only
                    Fn.rmsnorm(hidden[r0:r1], self.layers[0].input_norm_w, eps, residual[r0:r1], out=h[r0:r1])
                    q = at.qkv_proj(h[r0:r1], tpc)
                    if qkv0 is None:
                        qkv0 = torch.empty(hidden.shape[0], q.shape[1], dtype=q.dtype, device=q.device)
                    qkv0[r0:r1].copy_(q)
            else:
                if recv_tiles:
                    for _, _, works in recv_tiles:
                        for w in works:
                            w.wait()
                h, residual = Fn.rmsnorm(hidden, self.layers[0].input_norm_w, eps, residual)
        nvtx = _NVTX and h.is_cuda
        for i, layer in enumerate(self.layers):
            if nvtx:
                if i:
                    torch.cuda.nvtx.range_pop()
                torch.cuda.nvtx.range_push(f"layer{layer.layer_id}")
            if i + 1 < n:
                nxt = self.layers[i + 1].input_norm_w
            else:
                nxt = self.final_norm_w if self.is_last else None
            if deepstack is not None and i < len(deepstack[1]):
                # DeepStack (Qwen3-VL): intermediate ViT features are added to the block output at the
                # visual token rows before the next block's norm (reference: models/qwen3_vl.py:525-568)
                out, residual = layer(inp, h, residual, kv_cache, tpc, None)
                out.index_add_(0, deepstack[0], deepstack[1][i])
                h, residual = Fn.rmsnorm(out, nxt, eps, residual)
            elif i == 0 and qkv0 is not None:
                h, residual = layer(inp, h, residual, kv_cache, tpc, nxt, qkv=qkv0)
            else:
                h, residual = layer(inp, h, residual, kv_cache, tpc, nxt)
        if nvtx and n:
            torch.cuda.nvtx.range_pop()
        if not self.is_last:
            residual = tpc.stage_exit(residual)
        return h, residual

    def compute_logits(self, inp, hidden: torch.Tensor, tpc: TPComm, all_rows: bool = False,
                       local: bool = False) -> torch.Tensor:
        """Logits of the last token of every emitting sequence -> [E, V]; `local=True` returns this rank's vocab
        shard [E, Vp/tp] instead (vocab-parallel sampling: the runner reduces winners, not logits)."""
        hidden = tpc.materialize(hidden)
        rows = hidden if all_rows else Fn.gather_rows(hidden, inp.logits_idx)
        shard = Fn.linear(rows, self.lm_head_w)
        if local:
            return shard
        return tpc.gather_logits(shard, self.spec.vocab_size)

    # -- weights ----------------------------------------------------------------------------------
    def process_weights(self):
        """Post-load preparation of derived tensors (padded routers, absorbed MLA matrices, ...): every
        sub-module that defines `process_weights` is visited. Runs after loading, before graph capture."""
        for m in self.modules():
            if m is not self and hasattr(m, "process_weights"):
                m.process_weights()

    def init_dummy(self, seed: int = 0):
        """`--load-format dummy`: random weights of the right shapes (reference: model_loader.py:154)."""
        rank_seed = seed + 1000 * self.tp_rank + 7 * ps.get_pp_rank()
        g = torch.Generator(device="cpu").manual_seed(rank_seed)
        gd = None    # seeded on-device RNG: the same dummy weights in every run, so that runs can be compared
        for name, p in self.named_parameters():
            if p.is_cuda and gd is None:
                gd = torch.Generator(device=p.device).manual_seed(rank_seed)
            if name.endswith("norm_w"):
                p.data.fill_(1.0)
            elif p.dim() == 1:
                p.data.zero_()
            elif name.endswith("router_w") or name.endswith("shared_gate_w"):
                # replicated parameters must be identical on every rank
                gr = torch.Generator(device="cpu").manual_seed(seed + 31 + len(name))
                p.data.copy_((torch.randn(p.shape, generator=gr) * 0.3).to(p.dtype))
            elif p.dtype == torch.float8_e4m3fn:
                step = 1 << 26
                flat = p.data.view(-1)
                for s0 in range(0, flat.numel(), step):
                    e0 = min(s0 + step, flat.numel())
                    flat[s0:e0].copy_((torch.randn(e0 - s0, device=p.device, generator=gd if p.is_cuda else None)
                                       * 100.0).clamp_(-448.0, 448.0)
                                     .to(torch.float8_e4m3fn))   # e4m3fn has no inf: out-of-range casts give NaN
            elif name.endswith("_ws"):
                p.data.fill_(0.02 / 100.0)
            elif p.is_cuda:
                p.data.normal_(mean=0.0, std=0.02, generator=gd)  # on-device RNG: 8B params in well under a second
            else:
                flat = p.data.view(-1)
                step = 1 << 24
                for s in range(0, flat.numel(), step):
                    e = min(s + step, flat.numel())
                    flat[s:e].copy_((torch.randn(e - s, generator=g) * 0.02).to(p.dtype))

    def load_weights(self, reader: wu.CheckpointReader, progress: Optional[Callable[[int, int], None]] = None):
        spec, nm = self.spec, {**DEFAULT_NAMES, **self.spec.names}
        tp, tr = self.tp_size, self.tp_rank
        d = spec.head_dim
        total = len(self.layers) + 2
        done = 0

        def tick():
            nonlocal done
            done += 1
            if progress is not None:
                progress(done, total)

        def put(param, tensor):
            assert tuple(param.shape) == tuple(tensor.shape), (tuple(param.shape), tuple(tensor.shape))
            param.data.copy_(tensor)

        if self.embed_w is not None:
            put(self.embed_w, wu.shard_vocab(reader.get(nm["embed"]), tr, tp))
        tick()
        for layer in self.layers:
            pre = nm["layer"].format(i=layer.layer_id)
            at = layer.attn
            put(layer.input_norm_w, reader.get(pre + nm["input_norm"]))
            put(layer.post_norm_w, reader.get(pre + nm["post_norm"]))
            self._load_attention(reader, pre, nm, at)
            if layer.is_moe:
                layer.mlp.load_weights(reader, pre, nm)
            else:
                self._load_dense_mlp(reader, pre, nm, layer.mlp)
            tick()
        if self.is_last:
            put(self.final_norm_w, reader.get(nm["final_norm"]))
            if not spec.tie_word_embeddings:
                name = nm["lm_head"] if reader.has(nm["lm_head"]) else nm["embed"]
                put(self.lm_head_w, wu.shard_vocab(reader.get(name), tr, tp))
        tick()

    def _load_attention(self, reader, pre, nm, at: Attention):
        spec, tp, tr, d = self.spec, self.tp_size, self.tp_rank, self.spec.head_dim
        if "qkv_fused" in nm:  # ChatGLM: one [ (hq + 2 hkv) * D, H ] tensor
            w = reader.get(pre + nm["qkv_fused"] + ".weight")
            q, k, v = w.split([spec.num_heads * d, spec.num_kv_heads * d, spec.num_kv_heads * d], dim=0)
        else:
            q = reader.get(pre + nm["q"] + ".weight")
            k = reader.get(pre + nm["k"] + ".weight")
            v = reader.get(pre + nm["v"] + ".weight")
        _store_linear(at.qkv_w, at.qkv_ws, wu.shard_qkv(q, k, v, spec.num_heads, spec.num_kv_heads, d, tr, tp))
        if at.qkv_b is not None:
            if "qkv_fused" in nm:
                b = reader.get(pre + nm["qkv_fused"] + ".bias")
                qb, kb, vb = b.split([spec.num_heads * d, spec.num_kv_heads * d, spec.num_kv_heads * d], dim=0)
            else:
                qb, kb, vb = (reader.get(pre + nm[x] + ".bias") for x in ("q", "k", "v"))
            at.qkv_b.data.copy_(wu.shard_qkv(qb, kb, vb, spec.num_heads, spec.num_kv_heads, d, tr, tp))
        _store_linear(at.o_w, at.o_ws, wu.shard_cols(reader.get(pre + nm["o"] + ".weight"), tr, tp))
        if at.o_b is not None:
            at.o_b.data.copy_(reader.get(pre + nm["o"] + ".bias"))
        if at.q_norm_w is not None:
            at.q_norm_w.data.copy_(reader.get(pre + nm["q_norm"]))
            at.k_norm_w.data.copy_(reader.get(pre + nm["k_norm"]))

    def _load_dense_mlp(self, reader, pre, nm, mlp: DenseMLP):
        tp, tr = self.tp_size, self.tp_rank
        if "gate_up_fused" in nm:  # ChatGLM dense_h_to_4h = [gate; up]
            w = reader.get(pre + nm["gate_up_fused"] + ".weight")
            gate, up = w.chunk(2, dim=0)
        else:
            gate = reader.get(pre + nm["gate"] + ".weight")
            up = reader.get(pre + nm["up"] + ".weight")
        mlp.set_gate_up(wu.shard_gate_up(gate, up, tr, tp))
        _store_linear(mlp.down_w, mlp.down_ws, wu.shard_cols(reader.get(pre + nm["down"] + ".weight"), tr, tp))
