"""``custom_pretrained_transformer`` token embedder on the sm_100a encoder.

Drop-in for MemVul/custom_PTM_embedder.py:22-242 (registered name, constructor keywords and
``forward(token_ids, mask, type_ids, segment_concat_mask)`` are the reference's).  The reference
calls HF ``BertModel`` (:224-228) and returns ``last_hidden_state`` (:235); here the same tensor is
produced by ``memvul_encoder_forward`` (tcgen05 GEMMs + fused attention, include/memvul_b200.h).

Differences that are visible to a caller, all on padded positions only: hidden rows of masked
(padded) tokens are unspecified (the reference computes garbage-but-finite values there that nothing
on this path reads; ModelMemory takes row 0 only, model_memory.py:99).  Masks must be prefix masks
(what AllenNLP's padding produces).  The long-sequence fold/unfold path (:244-381) is unreachable in
the reference configs (``max_length`` unset, SURVEY.md F8) and raises here.
"""
from __future__ import annotations

import os
from typing import Any, Dict, Optional

import torch

from . import native
from .modules import BertConfigLite, BertWeights, params_version
from .registrable import TokenEmbedder

_PACKED_DEFAULT = os.environ.get("MEMVUL_ENC_PACKED", "1") != "0"


@TokenEmbedder.register("custom_pretrained_transformer")
class PretrainedTransformerEmbedder(TokenEmbedder):
    authorized_missing_keys = [r"position_ids$"]

    def __init__(
        self,
        model_name: str = None,
        *,
        max_length: int = None,
        sub_module: str = None,
        train_parameters: bool = True,
        eval_mode: bool = False,
        last_layer_only: bool = True,
        override_weights_file: Optional[str] = None,
        override_weights_strip_prefix: Optional[str] = None,
        gradient_checkpointing: Optional[bool] = None,
        tokenizer_kwargs: Optional[Dict[str, Any]] = None,
        transformer_kwargs: Optional[Dict[str, Any]] = None,
        pretrained_model_path: str = "out_wwm/",
        config: Optional[BertConfigLite] = None,
        precision: Optional[str] = None,
    ) -> None:
        super().__init__()
        # Not a reference keyword: "fp16" (default) = fp16 GEMM operands / fp32 accumulation; "split_fp16" = the opt-in
        # accuracy mode (MEMVUL_ENC_PRECISE: every operand split into two fp16 numbers, fp32 between the GEMMs) for
        # checkpoints whose heads amplify the fp16-operand error beyond the 1e-3 logit tolerance.  MEMVUL_PRECISION
        # overrides the default of models that do not pass the keyword (archives written by the reference never do).
        precision = precision or os.environ.get("MEMVUL_PRECISION", "fp16")
        if precision not in ("fp16", "split_fp16"):
            raise ValueError(f"precision must be 'fp16' or 'split_fp16', got {precision!r}")
        self.precision = precision
        if sub_module:
            raise NotImplementedError("sub_module is not used by the MemVul configs")
        if not last_layer_only:
            raise NotImplementedError("scalar-mix of all layers is not used by the MemVul configs")
        # custom_PTM_embedder.py:99 loads the further-pretrained BERT from a local directory.  Without
        # that directory (this image has no weights) the tree is created with HF's init and is expected
        # to be overwritten by the archive's weights.th through load_state_dict.
        if pretrained_model_path and os.path.isfile(os.path.join(pretrained_model_path, "config.json")) \
                and os.path.isfile(os.path.join(pretrained_model_path, "pytorch_model.bin")):
            self.transformer_model = BertWeights.from_pretrained(pretrained_model_path)
        else:
            self.transformer_model = BertWeights(config or BertConfigLite(**(transformer_kwargs or {})))
        self.config = self.transformer_model.config
        self._max_length = max_length
        self.output_dim = self.config.hidden_size
        self.train_parameters = train_parameters
        if not train_parameters:
            for p in self.transformer_model.parameters():
                p.requires_grad = False
        self.eval_mode = eval_mode
        self._packed: Optional[native.PackedBert] = None
        self._packed_version = None
        self._workspace: Optional[torch.Tensor] = None

    def get_output_dim(self) -> int:
        return self.output_dim

    def _number_of_token_type_embeddings(self) -> int:
        return self.config.type_vocab_size

    # ------------------------------------------------------------------ native plumbing
    def packed(self) -> native.PackedBert:
        """fp16 GEMM-layout copy of the fp32 master weights, rebuilt when they change."""
        dev = self.transformer_model.embeddings.word_embeddings.weight.device
        if dev.type != "cuda":
            raise native.NativeError("memvul_b200 runs on a CUDA device only (model is on %s); there is no CPU path" % dev)
        ver = (params_version(self.transformer_model), dev, self.precision)
        if self._packed is None or self._packed_version != ver:
            sd = {"m." + k: v for k, v in self.transformer_model.state_dict().items()}
            self._packed = native.PackedBert(sd, "m.", dev, ln_eps=self.config.layer_norm_eps,
                                             precise=self.precision == "split_fp16")
            self._packed_version = ver
        return self._packed

    def workspace(self, B: int, S: int, device: torch.device, flags: int = 0) -> torch.Tensor:
        need = self.packed().workspace_bytes(B, S, flags)
        if self._workspace is None or self._workspace.numel() < need or self._workspace.device != device:
            # reused for every batch shape and never initialised (include/memvul_b200.h: each call writes every row it
            # reads); grown geometrically so a stream of growing batches does not reallocate every step
            grow = 0 if self._workspace is None or self._workspace.device != device else self._workspace.numel() * 5 // 4
            self._workspace = None
            self._workspace = torch.empty(max(need, grow), dtype=torch.uint8, device=device)
        return self._workspace

    def encode(self, token_ids: torch.Tensor, lens: torch.Tensor, type_ids: Optional[torch.Tensor] = None,
               out: Optional[torch.Tensor] = None, cls_only: bool = False,
               row_start: Optional[torch.Tensor] = None, bad: Optional[torch.Tensor] = None) -> torch.Tensor:
        """[B,S] ids + per-sequence lengths -> fp32 [B,S,H]; asynchronous on the current stream.
        ``cls_only``: only ``[:, 0]`` is the final layer's output (enough for BertPooler).
        ``row_start``: packed var-len execution (padded tokens are never computed)."""
        B, S = token_ids.shape
        flags = native.encoder_flags(self.packed(), cls_only, row_start is not None)
        return native.encoder_forward(self.packed(), token_ids.contiguous(), lens,
                                      None if type_ids is None else type_ids.contiguous(),
                                      self.workspace(B, S, token_ids.device, flags), out, cls_only=cls_only,
                                      row_start=row_start, bad=bad)

    # ------------------------------------------------------------------ reference interface
    def forward(self, token_ids: torch.LongTensor, mask: torch.BoolTensor,
                type_ids: Optional[torch.LongTensor] = None,
                segment_concat_mask: Optional[torch.BoolTensor] = None, *, cls_only: bool = False) -> torch.Tensor:
        if self._max_length is not None and token_ids.size(1) > self._max_length:
            raise NotImplementedError("fold/unfold of long sequences (custom_PTM_embedder.py:244-381) is unreachable "
                                      "in the MemVul configs and not implemented")
        if token_ids.shape != mask.shape:
            raise ValueError("token_ids and mask must have the same shape")
        if type_ids is not None and token_ids.shape != type_ids.shape:
            raise ValueError("token_ids and type_ids must have the same shape")       # :205-206
        # Packed (token-major, var-len) execution is the default: the reference pads every batch to its longest member
        # (config_memory.json:50-57) and pays for the padding in every GEMM; here padded tokens are never computed and
        # the row count stays on the device (no host sync).  MEMVUL_ENC_PACKED=0 selects the padded execution.
        if _PACKED_DEFAULT:
            lens, row_start, bad = native.mask_to_lens(mask.contiguous(), with_row_start=True)
        else:
            (lens, bad), row_start = native.mask_to_lens(mask.contiguous()), None
        hidden = self.encode(token_ids, lens, type_ids, cls_only=cls_only, row_start=row_start, bad=bad)
        # The reference's `type_ids.max()` (:199-202) is a host sync per batch, and torch.embedding raises on an
        # out-of-range id; here both checks (and the prefix-mask check) set bits of a device flag that the caller reads
        # with its results (ModelMemory bundles it with the result copy; native.raise_for_flag turns it into the error).
        self.last_bad_mask_flag = bad
        return hidden

    def check_last_batch(self) -> None:
        """Synchronising check of the deferred flag of the last ``forward`` (mask not a prefix mask / id out of range)."""
        native.raise_for_flag(int(self.last_bad_mask_flag.item()))
