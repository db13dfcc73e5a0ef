"""Drop-in module surface of the reference (``aecf/AECFLayer.py``), dispatching to the sm_100a kernels.

Same class names, constructor and ``forward`` signatures, attribute names, ``state_dict`` keys,
``info`` keys/shapes/detach status and exception types as the reference; the arithmetic runs in the
C-ABI library (``include/aecf_b200.h``).  CUDA tensors only -- there is no CPU or eager fallback.

Deliberate differences (DESIGN.md "reference quirks"):
  * ``info`` tensors are fp32 even when the module runs in bf16 (the reference computes entropy in
    bf16, which collapses it to a handful of distinct values; SURVEY.md section 0 item 8).
  * ``use_checkpoint=`` is accepted and ignored: the fused backward always recomputes the attention
    weights, and because dropout is counter-based the recompute is exact (the reference's is not,
    ``aecf/AECFLayer.py:510-512``).
  * exact ties in the ``min_active`` top-k go to the lowest index (the reference inherits an
    implementation-defined choice from ``torch.topk`` for more than 3 tokens).
"""
from __future__ import annotations

import math
import os
import threading
from typing import Any, Dict, Optional, Tuple, Union

import torch
import torch.nn as nn

from . import ops
from .fused_pool import (CurriculumMaskFunction, EntropyFunction, EntropyLossFunction, FusedPoolFunction, PoolConfig,
                         SdpaFunction, SideStream)

__all__ = ["CurriculumMasking", "MultimodalAttentionPool", "multimodal_attention_pool", "create_fusion_pool",
           "set_rng_state", "get_rng_state"]


# ---------------------------------------------------------------------------------------------
# Philox call counter.  seed follows torch.manual_seed(); every forward that draws random numbers
# takes the next offset, so a run is reproducible after seeding, like the reference's torch RNG use.
# ---------------------------------------------------------------------------------------------
class _PhiloxState:
    """Hands out one (seed, call offset) pair per forward that draws random numbers.

    On a CUDA device the pair comes from torch's own Philox generator for that device -- the seed
    set by ``torch.manual_seed`` and the generator's running offset, which is advanced like any torch
    random op would -- so re-seeding restarts the stream exactly as it does for the reference's
    ``torch.bernoulli`` / dropout draws.  ``set_rng_state`` pins an explicit pair instead (parity tests).
    """

    def __init__(self):
        self.lock = threading.Lock()
        self.explicit_seed: Optional[int] = None
        self.seen_seed: Optional[int] = None
        self.offset = 0
        # CUDA-graph capture: per-device int64 tensor {seed, next offset} that captured forwards read and
        # advance ON THE DEVICE (a by-value pair would be frozen into the graph); see aecf_b200.graphs
        self.device_states: Dict[int, torch.Tensor] = {}

    def prepare_device_state(self, device: torch.device) -> torch.Tensor:
        """Create (or refresh) the device-side {seed, next offset} pair from the host-side state.  Must run
        outside capture: captured forwards then draw from it and advance it with captured kernels."""
        seed, offset = self.next(device)
        index = device.index if device.index is not None else torch.cuda.current_device()
        host = torch.tensor([seed - (1 << 64) if seed >= (1 << 63) else seed, offset], dtype=torch.int64)
        with self.lock:
            state = self.device_states.get(index)
            if state is None:
                state = self.device_states[index] = host.to(device)
            else:
                state.copy_(host)
        return state

    def captured(self, device: torch.device) -> torch.Tensor:
        """Inside capture: a snapshot of the device-side pair for this call (the backward's recompute reads
        the same snapshot), after which the device-side offset moves on -- both as captured kernels."""
        index = device.index if device.index is not None else torch.cuda.current_device()
        state = self.device_states.get(index)
        if state is None:
            raise RuntimeError(
                "aecf_b200: a forward that draws random numbers is being captured into a CUDA graph, but the "
                "device-side Philox state does not exist yet. Call aecf_b200.graphs.prepare(device) before the "
                "capture (aecf_b200.graphs.capture_step does it for you).")
        used = state.clone()
        state[1:2].add_(1)
        return used

    def next(self, device: Optional[torch.device] = None) -> Tuple[int, int]:
        with self.lock:
            if self.explicit_seed is None and device is not None and device.type == "cuda":
                gen = torch.cuda.default_generators[device.index if device.index is not None
                                                    else torch.cuda.current_device()]
                off = gen.get_offset()
                gen.set_offset(off + 4)                          # one Philox block, like a torch random op
                return gen.initial_seed() & 0xFFFFFFFFFFFFFFFF, (off // 4) & 0xFFFFFFFF
            seed = self.explicit_seed if self.explicit_seed is not None else torch.initial_seed()
            if self.explicit_seed is None and seed != self.seen_seed:
                self.seen_seed, self.offset = seed, 0
            off = self.offset
            self.offset = (self.offset + 1) & 0xFFFFFFFF
            return seed & 0xFFFFFFFFFFFFFFFF, off


_rng = _PhiloxState()


def set_rng_state(seed: Optional[int], offset: int = 0) -> None:
    """Pin the Philox (seed, next offset) used for masks and dropout; ``seed=None`` follows torch again."""
    with _rng.lock:
        _rng.explicit_seed = seed
        _rng.seen_seed = None
        _rng.offset = int(offset) & 0xFFFFFFFF
        stale = list(_rng.device_states)
    if seed is not None and stale and not torch.cuda.is_current_stream_capturing():
        for index in stale:                                  # graphs captured earlier follow the new pair too
            s64 = seed & 0xFFFFFFFFFFFFFFFF
            host = torch.tensor([s64 - (1 << 64) if s64 >= (1 << 63) else s64, _rng.offset], dtype=torch.int64)
            _rng.device_states[index].copy_(host)


def get_rng_state() -> Tuple[int, int]:
    with _rng.lock:
        seed = _rng.explicit_seed if _rng.explicit_seed is not None else torch.initial_seed()
        return seed, _rng.offset


class CurriculumMasking(nn.Module):
    """Entropy-driven curriculum masking of attention weights (reference ``aecf/AECFLayer.py:33-319``).

    Inside :class:`MultimodalAttentionPool` this stage is part of the fused forward kernel; the
    parameters below are read at call time, so mutating them between steps works as in the reference
    (``README.md:341-350``).
    """

    def __init__(self, base_mask_prob: float = 0.15, entropy_target: float = 0.7, min_active: int = 1):
        super().__init__()
        if not 0.0 < base_mask_prob <= 1.0:
            raise ValueError(f"base_mask_prob must be in (0, 1], got {base_mask_prob}")
        if not 0.0 < entropy_target <= 1.0:
            raise ValueError(f"entropy_target must be in (0, 1], got {entropy_target}")
        if min_active < 1:
            raise ValueError(f"min_active must be >= 1, got {min_active}")
        self.base_mask_prob = base_mask_prob
        self.entropy_target = entropy_target
        self.min_active = min_active
        self.register_buffer("_eps", torch.tensor(1e-8))     # state_dict key 'curriculum_masking._eps'
        self._last_seq_len = 2                                # reference :99

    def compute_entropy(self, weights: torch.Tensor) -> torch.Tensor:
        """Shannon entropy over the last dimension, clamped to [0, log L] (reference :101-128)."""
        return self.compute_entropy_fused(weights)

    def compute_entropy_fused(self, weights: torch.Tensor) -> torch.Tensor:
        ops.require_cuda(weights)
        return EntropyFunction.apply(weights)

    def forward(self, weights: torch.Tensor) -> Tuple[torch.Tensor, Dict[str, torch.Tensor]]:
        """Standalone masking of caller-supplied weights (..., L), L <= 64 (reference :130-283).

        Inside MultimodalAttentionPool this stage runs fused in the pool kernel instead.  The masked weights
        returned here in training mode keep their graph, like the reference's ``final_weights`` (the mask itself and
        the entropy carry no gradient).
        """
        ops.require_cuda(weights)
        lead, length = weights.shape[:-1], weights.shape[-1]
        if not self.training:                                             # :150-156
            return weights, {"entropy": EntropyFunction.apply(weights),
                             "mask_rate": torch.zeros(lead, device=weights.device, dtype=weights.dtype)}
        if length <= 1:                                                   # :159-167
            zeros = torch.zeros(lead, device=weights.device, dtype=weights.dtype)
            return weights, {"entropy": zeros, "mask_rate": zeros.clone(), "target_entropy": zeros.clone()}
        self._last_seq_len = length                                       # :187
        seed, offset = _rng.next(weights.device)
        masked, entropy, mask_rate = CurriculumMaskFunction.apply(weights, self.base_mask_prob, self.min_active, seed, offset)
        entropy = entropy.reshape(lead).to(weights.dtype)
        info = {"entropy": entropy, "mask_rate": mask_rate.reshape(lead).to(weights.dtype),
                "target_entropy": torch.full_like(entropy, math.log(float(length)) * self.entropy_target)}
        return masked, info

    def _loss_target(self) -> float:
        seq_len = getattr(self, "_last_seq_len", 2)
        return (math.log(float(seq_len)) if seq_len > 1 else 0.0) * self.entropy_target

    def entropy_loss(self, entropy: torch.Tensor) -> torch.Tensor:
        """mean((entropy - entropy_target * log(L))^2), L = tokens of the last training forward (:285-314).

        For the ``info['entropy']`` tensor of the pool's last training-mode forward the value was already produced by that
        forward's kernel (the per-sample term is fused there, ``aecf_pool_desc::loss_out``) and is returned as is -- in
        training mode the reference's entropy is detached (:278), so there is no gradient to carry.  Any other tensor
        (eval mode, user-made, modified in place since) takes the stand-alone kernels."""
        target = self._loss_target()
        fused = getattr(entropy, "_aecf_fused_loss", None)      # attached to the very tensor object the forward returned
        if fused is not None:
            version, fused_target, loss = fused
            if entropy._version == version and fused_target == target and not entropy.requires_grad:
                return loss.reshape(()).to(entropy.dtype)
        ops.require_cuda(entropy)
        return EntropyLossFunction.apply(entropy, target)

    def extra_repr(self) -> str:
        return (f"base_mask_prob={self.base_mask_prob}, entropy_target={self.entropy_target}, "
                f"min_active={self.min_active}")


class _OutProj(nn.Module):
    """Holds ``out_proj.weight`` / ``out_proj.bias`` under the names nn.MultiheadAttention uses."""

    def __init__(self, embed_dim: int, bias: bool, device, dtype):
        super().__init__()
        lin = nn.Linear(embed_dim, embed_dim, bias=bias, device=device, dtype=dtype)   # same RNG draws as MHA's
        self.weight = lin.weight
        if bias:
            self.bias = lin.bias
        else:
            self.register_parameter("bias", None)


class _AttentionParams(nn.Module):
    """Parameter container with nn.MultiheadAttention's names, shapes and default initialisation
    (torch/nn/modules/activation.py:1189-1242), so ``state_dict`` round-trips with the reference."""

    def __init__(self, embed_dim: int, num_heads: int, dropout: float, bias: bool, device, dtype):
        super().__init__()
        self.embed_dim, self.num_heads, self.dropout = embed_dim, num_heads, dropout
        self.head_dim = embed_dim // num_heads
        self.in_proj_weight = nn.Parameter(torch.empty((3 * embed_dim, embed_dim), device=device, dtype=dtype))
        if bias:
            self.in_proj_bias = nn.Parameter(torch.empty(3 * embed_dim, device=device, dtype=dtype))
        else:
            self.register_parameter("in_proj_bias", None)
        self.out_proj = _OutProj(embed_dim, bias, device, dtype)
        nn.init.xavier_uniform_(self.in_proj_weight)
        if bias:
            nn.init.constant_(self.in_proj_bias, 0.0)
            nn.init.constant_(self.out_proj.bias, 0.0)


class MultimodalAttentionPool(nn.Module):
    """Attention pooling over modality tokens (reference ``aecf/AECFLayer.py:322-552``).

    ``forward(query, key, value=None, key_padding_mask=None, attn_mask=None, return_info=False,
    use_checkpoint=False)``; ``query`` is ``[B, S, D]`` -- S = 1 (one fusion token per sample, usually an expand of
    one ``[1, 1, D]`` parameter) is the hot path, S > 1 runs the multi-query kernels.
    """

    def __init__(self, embed_dim: int, num_heads: int = 1, dropout: float = 0.0, bias: bool = True,
                 curriculum_masking: Optional[CurriculumMasking] = None, batch_first: bool = True,
                 device: Optional[torch.device] = None, dtype: Optional[torch.dtype] = None):
        super().__init__()
        if embed_dim <= 0:
            raise ValueError(f"embed_dim must be positive, got {embed_dim}")
        if num_heads <= 0:
            raise ValueError(f"num_heads must be positive, got {num_heads}")
        if embed_dim % num_heads != 0:
            raise ValueError(f"embed_dim ({embed_dim}) must be divisible by num_heads ({num_heads})")
        if not 0.0 <= dropout <= 1.0:
            raise ValueError(f"dropout must be in [0, 1], got {dropout}")
        self.embed_dim = embed_dim
        self.num_heads = num_heads
        self.batch_first = batch_first
        self.curriculum_masking = curriculum_masking
        self.attention = _AttentionParams(embed_dim, num_heads, dropout, bias, device, dtype)
        # data-parallel state (aecf_b200.dp): global index of local row 0, gradient-ready callback
        self.row_offset = 0
        self._grad_ready = None
        self._grad_buffers = None
        self._dp = None                               # data parallelism: aecf_b200.dp.FusedGradSum
        self._side = None                             # SideStream of the backward's gradient tail, made on first use
        self._want_mask_bits = False
        # Folded key projection (include/aecf_b200.h): None = automatic -- on for bf16 whenever one fusion query
        # is shared by all rows and key is value (AECF_FOLD=0 in the environment turns the automatic choice off);
        # True forces it wherever it applies (also fp32), False keeps the K projection.
        self.fold_key_projection: Optional[bool] = None

    # -- validation: same exception types and messages as the reference (:450-498) -----------
    def _validate(self, query, key, value):
        if not isinstance(query, torch.Tensor):
            raise TypeError(f"Expected query to be torch.Tensor, got {type(query)}")
        if not isinstance(key, torch.Tensor):
            raise TypeError(f"Expected key to be torch.Tensor, got {type(key)}")
        if value is not None and not isinstance(value, torch.Tensor):
            raise TypeError(f"Expected value to be torch.Tensor or None, got {type(value)}")
        val = key if value is None else value
        tag = "True" if self.batch_first else "False"
        for name, t in (("query", query), ("key", key), ("value", val)):
            if t.dim() != 3:
                raise ValueError(f"Expected 3D {name} tensor with batch_first={tag}, got {t.dim()}D")
        bdim, sdim = (0, 1) if self.batch_first else (1, 0)
        batch, embed = query.shape[bdim], query.shape[2]
        if key.shape[sdim] == 0:
            raise ValueError("Key sequence length cannot be zero")
        if key.shape[bdim] != batch or key.shape[2] != embed:
            if self.batch_first:
                raise RuntimeError(f"Key shape {key.shape} incompatible with query shape {query.shape}")
            raise RuntimeError(f"Shape mismatch: query {query.shape}, key {key.shape}")
        if val.shape[bdim] != batch or val.shape[sdim] != key.shape[sdim] or val.shape[2] != embed:
            raise RuntimeError(f"Value shape {val.shape} incompatible with key shape {key.shape}")
        return batch, query.shape[sdim], key.shape[sdim], embed

    def _shared_query_source(self, query: torch.Tensor, batch: int):
        """If every row of ``query`` is the same vector (the documented ``fusion_query.expand(B,-1,-1)``
        pattern), return the D-element tensor to differentiate instead of the B x D expansion."""
        bdim = 0 if self.batch_first else 1
        D = query.shape[2]
        if batch == 1:
            return query
        if query.stride(bdim) != 0 or query.stride(2) != 1:
            return None
        base = query._base
        if (base is not None and base.numel() == D and base.is_contiguous() and base.dtype == query.dtype
                and base.device == query.device and query.storage_offset() == base.storage_offset()):
            return base                      # the Parameter itself: its gradient arrives already reduced
        return query.narrow(bdim, 0, 1)      # generic stride-0 view: autograd expands the reduced gradient

    def _score_bias(self, key_padding_mask, attn_mask, batch, tokens, device, tgt_len=1):
        """Merge key_padding_mask and attn_mask into one additive fp32 bias the way torch does
        (torch/nn/functional.py:6608-6620).  Returns (tensor or None, (stride_b, stride_h, stride_s)): a contiguous
        [b, h, s, tokens] tensor whose broadcast dimensions have size 1 and stride 0."""
        def as_float(mask):
            if mask.dtype == torch.bool:
                return torch.zeros(mask.shape, dtype=torch.float32, device=device).masked_fill_(mask, float("-inf"))
            return mask.to(torch.float32)

        H, S = self.num_heads, tgt_len
        bias = None
        if attn_mask is not None:
            am = as_float(attn_mask.to(device))
            if am.dim() == 2:
                if am.shape != (S, tokens):
                    raise RuntimeError(f"The shape of the 2D attn_mask is {tuple(am.shape)}, but should be {(S, tokens)}.")
                bias = am.reshape(1, 1, S, tokens)
            elif am.dim() == 3:
                if am.shape != (batch * H, S, tokens):
                    raise RuntimeError(
                        f"The shape of the 3D attn_mask is {tuple(am.shape)}, but should be {(batch * H, S, tokens)}.")
                bias = am.reshape(batch, H, S, tokens)
            else:
                raise RuntimeError(f"attn_mask's dimension {am.dim()} is not supported")
        if key_padding_mask is not None:
            if key_padding_mask.shape != (batch, tokens):
                raise RuntimeError(
                    f"expecting key_padding_mask shape of {(batch, tokens)}, but got {tuple(key_padding_mask.shape)}")
            kpm = as_float(key_padding_mask.to(device)).reshape(batch, 1, 1, tokens)
            bias = kpm if bias is None else bias + kpm
        if bias is None:
            return None, (0, 0, 0)
        bias = bias.contiguous()
        b, h, s, _ = bias.shape
        return bias, (h * s * tokens if b > 1 else 0, s * tokens if h > 1 else 0, tokens if s > 1 else 0)

    def _side_stream(self, device: torch.device):
        """The second stream the folded backward's gradient tail runs on (AECF_SIDE_STREAM=0: everything in order)."""
        if os.environ.get("AECF_SIDE_STREAM", "1") == "0" or device.type != "cuda":
            return None
        if self._side is None or self._side.device != device:
            if torch.cuda.is_current_stream_capturing():
                return None                             # streams and events are made outside captures (the warm-up steps)
            self._side = SideStream(device)
        return self._side

    def forward(self, query: torch.Tensor, key: torch.Tensor, value: Optional[torch.Tensor] = None,
                key_padding_mask: Optional[torch.Tensor] = None, attn_mask: Optional[torch.Tensor] = None,
                return_info: bool = False, use_checkpoint: bool = False, sample_index: Optional[torch.Tensor] = None,
                ) -> Union[torch.Tensor, Tuple[torch.Tensor, Dict[str, Any]]]:
        """Same arguments as the reference (``aecf/AECFLayer.py:409-418``) plus one extension, ``sample_index``: a 1-D integer
        tensor of DISTINCT batch indices.  Only those samples are pooled -- exactly as if the reference had been called on
        ``query[idx], key[idx]`` (same Philox rows, info tensors of ``len(idx)`` rows) -- but in place: the output keeps the
        full batch layout ``[B, 1, D]``, rows of unlisted samples hold ``out_proj.bias`` (the projection of a zero context; mask
        them, e.g. with ``torch.where``) and get no gradient.  This is the reference x-ray model's gather -> pool -> scatter
        (``xrays/train_xrays_example.py:202-222``) without the two indexing copies.  Needs the shared fusion query and no masks."""
        batch, tgt_len, tokens, embed = self._validate(query, key, value)
        if value is key:
            value = None
        ops.require_cuda(query, key, value, self.attention.in_proj_weight)
        if embed != self.embed_dim:
            raise RuntimeError(f"was expecting embedding dimension of {self.embed_dim}, but got {embed}")
        # several queries per sample run on their own kernels (csrc/pool_multi.cuh)
        multi = tgt_len > 1
        att = self.attention
        pdt = att.in_proj_weight.dtype
        q_src = None if multi else self._shared_query_source(query, batch)
        q_shared = q_src is not None
        # Mixed precision: fp32 parameters, bf16 key / value (what torch.autocast hands over from bf16 encoders).  The step
        # runs in bf16 on a bf16 rounding of the parameters, made on every call, and the parameter gradients are fp32.  The
        # query is then either bf16 rows of its own or the shared fp32 fusion query (a parameter, rounded like the others).
        dt = key.dtype
        if q_shared and batch == 1 and pdt == torch.float32 and dt == torch.bfloat16 and query.dtype == torch.bfloat16:
            q_src, q_shared = None, False                       # one sample: a bf16 query is that row's own
        mixed = (pdt == torch.float32 and dt == torch.bfloat16
                 and query.dtype == (torch.float32 if q_shared else torch.bfloat16))
        if not mixed:
            dt = pdt
        if (not mixed and (query.dtype != dt or key.dtype != dt)) or (value is not None and value.dtype != dt):
            raise RuntimeError(f"expected query/key/value of dtype {pdt} (the module's parameter dtype), "
                               f"got {query.dtype}/{key.dtype}")
        if multi:
            q_src = query.contiguous()             # [B, S, D] or [S, B, D], used in place (rows (b, s) by strides)
        elif not q_shared:
            q_src = (query if self.batch_first else query.transpose(0, 1)).contiguous()
        key_c = key.contiguous()
        value_c = None if value is None else value.contiguous()
        bias, bias_strides = self._score_bias(key_padding_mask, attn_mask, batch, tokens, key.device, tgt_len)
        index = None
        if sample_index is not None:
            if not q_shared or multi or bias is not None or not self.batch_first:
                raise ops._lib.UnsupportedShapeError(
                    ops._lib.ERR_UNSUPPORTED, "MultimodalAttentionPool",
                    "sample_index needs the shared fusion query (an expand of one [1, 1, D] tensor), batch_first and no masks")
            if sample_index.dim() != 1 or sample_index.dtype not in (torch.int64, torch.int32) or sample_index.device != key.device:
                raise ValueError("sample_index must be a 1-D int64 / int32 tensor on the inputs' device")
            index = sample_index.to(torch.int64).contiguous()

        cm = self.curriculum_masking
        fused_cm = cm is not None and type(cm).forward is CurriculumMasking.forward
        masking = 0
        if fused_cm:
            masking = 1 if cm.training else 2
            if cm.training and tokens > 1:
                cm._last_seq_len = tokens                               # reference :187
        can_fold = q_shared and value_c is None and self.num_heads <= 32 and not multi
        if self.fold_key_projection is None:
            fold = can_fold and dt == torch.bfloat16 and os.environ.get("AECF_FOLD", "1") != "0"
        else:
            fold = can_fold and bool(self.fold_key_projection)
        draws = (att.training and att.dropout > 0.0) or masking == 1
        rng_state = None
        if draws and torch.cuda.is_current_stream_capturing():
            seed, offset, rng_state = 0, 0, _rng.captured(key.device)
        else:
            seed, offset = _rng.next(key.device) if draws else (0, 0)
        cfg = PoolConfig(
            num_heads=self.num_heads, dropout_p=att.dropout, training=att.training, masking=masking,
            base_mask_prob=cm.base_mask_prob if fused_cm else 0.15,
            entropy_target=cm.entropy_target if fused_cm else 0.7,
            min_active=cm.min_active if fused_cm else 1,
            seed=seed, offset=offset, rng_state=rng_state, row0=int(self.row_offset), q_shared=q_shared,
            seq_first=not self.batch_first, fold=fold, want_mask_bits=self._want_mask_bits, bias_strides=bias_strides,
            tgt_len=tgt_len, grad_ready=self._grad_ready, grad_buffers=self._grad_buffers,
            loss_target=cm._loss_target() if (masking == 1 and return_info) else None,
            side=self._side_stream(key.device) if fold else None, dp=self._dp, sample_index=index, mixed=mixed)
        info_rows = batch if index is None else int(index.numel())
        out, pooled, entropy, mask_rate, masked, bits, fused_loss = FusedPoolFunction.apply(
            q_src, key_c, value_c, att.in_proj_weight, att.in_proj_bias, att.out_proj.weight, att.out_proj.bias,
            bias, cfg)

        attn_output = out.reshape(batch, tgt_len, embed) if self.batch_first else out.reshape(tgt_len, batch, embed)
        pooled_weights = pooled.reshape(info_rows, tgt_len, tokens)     # [B, S, M] whatever batch_first (functional.py:6657)
        info: Dict[str, Any] = {}
        if cm is not None:
            if fused_cm:
                info["entropy"] = entropy.reshape(info_rows, tgt_len)
                if fused_loss.numel() == 1:             # entropy_loss(info['entropy']) is already known: see there
                    info["entropy"]._aecf_fused_loss = (info["entropy"]._version, cfg.loss_target, fused_loss)
                info["mask_rate"] = mask_rate.reshape(info_rows, tgt_len)
                if cm.training:                                         # eval mode has no target (:153-156)
                    target = math.log(float(tokens)) * cm.entropy_target if tokens > 1 else 0.0
                    info["target_entropy"] = torch.full_like(info["entropy"], target)
                masked_weights = masked.reshape(info_rows, tgt_len, tokens)
            else:
                masked_weights, mask_info = cm(pooled_weights)          # user-overridden forward (README.md:341-350)
                info.update(mask_info)
            info["attention_weights"] = pooled_weights                  # keeps its gradient (:538)
            if return_info:
                info["masked_attention_weights"] = masked_weights.detach()
                if self._want_mask_bits:
                    info["mask_bits"] = bits.reshape(info_rows, tgt_len) if multi else bits
        elif return_info:
            info["attention_weights"] = pooled_weights
        if return_info:
            return attn_output, info
        return attn_output

    def extra_repr(self) -> str:
        return (f"embed_dim={self.embed_dim}, num_heads={self.num_heads}, batch_first={self.batch_first}, "
                f"curriculum_masking={self.curriculum_masking is not None}")


def multimodal_attention_pool(query: torch.Tensor, key: torch.Tensor, value: Optional[torch.Tensor] = None,
                              embed_dim: Optional[int] = None, num_heads: int = 1, dropout: float = 0.0,
                              curriculum_masking: Optional[CurriculumMasking] = None,
                              training: bool = False) -> torch.Tensor:
    """Functional interface (reference ``aecf/AECFLayer.py:584-652``).

    Fast path (eval, single head, no masking, no dropout): projection-free scaled dot-product
    attention, one kernel, any source/target length; differentiable (a two-kernel recompute backward).  Otherwise a freshly initialised
    :class:`MultimodalAttentionPool` is built per call, as in the reference -- but on the inputs'
    device and dtype (the reference builds it on CPU/fp32 and cannot take CUDA inputs; quirk D6).
    """
    if embed_dim is None:
        embed_dim = query.size(-1)
    if value is None:
        value = key
    if not training and curriculum_masking is None and dropout == 0.0 and num_heads == 1:
        ops.require_cuda(query, key, value)
        if query.dim() != 3 or key.dim() != 3 or value.dim() != 3:
            raise ValueError("expected 3D query, key and value tensors")
        if query.dtype != key.dtype or query.dtype != value.dtype:
            raise RuntimeError(f"expected query/key/value of one dtype, got {query.dtype}/{key.dtype}/{value.dtype}")
        return SdpaFunction.apply(query.contiguous(), key.contiguous(), value.contiguous())
    pool = MultimodalAttentionPool(embed_dim=embed_dim, num_heads=num_heads, dropout=dropout,
                                   curriculum_masking=curriculum_masking, batch_first=True,
                                   device=query.device, dtype=query.dtype)
    pool.train(training)
    return pool(query, key, value)


def create_fusion_pool(embed_dim: int, num_modalities: int, mask_prob: float = 0.15,
                       **kwargs) -> Tuple[nn.Parameter, MultimodalAttentionPool]:
    """Factory (reference ``aecf/AECFLayer.py:655-728``): a (1, 1, E) fusion query drawn from
    N(0, sqrt(2/E)) and a pool with ``CurriculumMasking(mask_prob)``.  ``kwargs`` go to the pool
    (``num_heads`` defaults to 1); ``device``/``dtype`` kwargs also apply to the query here, whereas
    the reference leaves it on CPU/fp32 (quirk D7)."""
    if not isinstance(embed_dim, int) or embed_dim <= 0:
        raise ValueError(f"embed_dim must be a positive integer, got {embed_dim}")
    if not isinstance(num_modalities, int) or num_modalities <= 0:
        raise ValueError(f"num_modalities must be a positive integer, got {num_modalities}")
    if not isinstance(mask_prob, (int, float)) or not (0.0 < mask_prob <= 1.0):
        raise ValueError(f"mask_prob must be in (0, 1], got {mask_prob}")
    fusion_query = nn.Parameter(torch.empty(1, 1, embed_dim))
    nn.init.normal_(fusion_query, 0.0, (2.0 / embed_dim) ** 0.5)        # drawn on CPU: same values as the reference
    if kwargs.get("device") is not None or kwargs.get("dtype") is not None:
        fusion_query = nn.Parameter(fusion_query.detach().to(device=kwargs.get("device"), dtype=kwargs.get("dtype")))
    masking = CurriculumMasking(base_mask_prob=mask_prob)
    pool = MultimodalAttentionPool(embed_dim=embed_dim, curriculum_masking=masking, **kwargs)
    return fusion_query, pool
