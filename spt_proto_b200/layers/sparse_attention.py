"""PQ sparse attention layers (reference naive_gpt/layers/sparse/attention.py).

V1 = dense attention + PQ training loss (how the codebooks are learned); V2 = the sparse hot path:
    q, k -> PQ codes -> lookup (top S/sparse_coeff keys per query, fixed-stride CSR)
         -> sddmm -> clamp(scaling * ., -10, 10) -> causal CSR softmax -> spmm with v.
Constructors, buffers (`trigger`, `loss`) and `from_pretrained` match the reference; `sparse_coeff`
(hard-wired to 8 in the reference, attention.py:110,115) is an attribute here."""
from __future__ import annotations

import torch

from .. import ext, kernels
from ..kernels import layout
from .basic import PQV1, PQV2, RotaryAttention, VanillaAttention


class _PQTrainMixin:
    """V1 behaviour: dense attention, PQ loss recorded on every forward (attention.py:34-44,181-193)."""

    def _init_pq(self, d_codeword, n_codewords, n_subspaces):
        self.d_codeword, self.n_codewords, self.n_subspaces = d_codeword, n_codewords, n_subspaces
        self.quantizer = PQV1(d_codeword=d_codeword, n_codewords=n_codewords, n_subspaces=n_subspaces)
        self.register_buffer("trigger", torch.scalar_tensor(False, dtype=torch.bool))

    def _record_loss(self, q, k):
        loss = self.quantizer("train", z=q)[-1] + self.quantizer("train", z=k)[-1]
        self.register_buffer("loss", loss, persistent=False)


class SparseVanillaAttentionV1(_PQTrainMixin, VanillaAttention):
    def __init__(self, d_head: int, p_dropout: float, d_codeword: int, n_codewords: int, n_subspaces: int):
        VanillaAttention.__init__(self, d_head=d_head, p_dropout=p_dropout)
        self._init_pq(d_codeword, n_codewords, n_subspaces)

    def _get_attn(self, q, k, attn_mask):
        self._record_loss(q, k)
        return VanillaAttention._get_attn(self, q, k, attn_mask)


class SparseRotaryAttentionV1(_PQTrainMixin, RotaryAttention):
    def __init__(self, d_head: int, p_dropout: float, d_codeword: int, n_codewords: int, n_subspaces: int):
        RotaryAttention.__init__(self, d_head=d_head, p_dropout=p_dropout)
        # the reference ignores n_subspaces here and derives it (attention.py:165-169)
        self._init_pq(d_codeword, n_codewords, d_head // d_codeword)
        self.n_subspaces = n_subspaces

    def _get_attn(self, q, k, attn_mask):
        q, k = self._rotate(q), self._rotate(k)
        self._record_loss(q, k)
        return VanillaAttention._get_attn(self, q, k, attn_mask)


class _SparseV2Mixin:
    """The hot path shared by the vanilla and rotary V2 layers (attention.py:84-142, 233-299)."""

    sparse_coeff: int = 8
    # The shipped reference un-transposes the 3-D result with `y.transpose(1, 2).contiguous()
    # .view(v_size)` (attention.py:139-142), which swaps S and E instead of S and H: its output is
    # a re-interpretation of [N*H, E, S] memory as [N, S, H, E] (invisible to its all-ones layer
    # test).  True (default) reproduces the shipped layer bit for bit — checkpoints fine-tuned with
    # the reference learned `linear_o` / LoRA against that layout, so the drop-in must return it;
    # False is the opt-in corrected layout (identical to the reference's dense VanillaAttention on
    # the same pattern).  Also a constructor keyword.  INTEGRATION.md, "Output layout".
    reference_output_layout: bool = True
    # bf16 or fp16, d_head 64, 80 or 128, S % 128 == 0 on CUDA: run lookup -> bitmask -> fused masked-dense attention
    # on the tensor cores instead of the stage chain (same result up to bf16 / fp16 rounding; DESIGN.md sec. 5).
    # False keeps the stage chain for every shape (fp16 operands run it in fp32 and the result is returned in fp16).
    use_fused: bool = True
    # The reference reads its device-side `trigger` buffer with `is_nonzero()` on every forward
    # (attention.py:98) — a device->host synchronisation per layer call.  None (default) keeps that
    # behaviour (a training loop arms the layer with `trigger.fill_(True)`, script/4-sparse-tuning-0.py:
    # 71-78).  Setting host_trigger to a bool makes the decision on the host, with no synchronisation:
    # True = compute the PQ loss on the next forward (then resets to False), False = skip it.
    host_trigger = None
    # Above this length (S, or max_seqlen of a packed batch) the fused path keeps the PQ codes (S m 4 bytes per head)
    # between forward and backward and runs the lookup again in the backward, instead of keeping the bitmask (S^2 / 8
    # bytes per head: 8 MiB at S 8192, 128 MiB at S 32768).  Same gradients bit for bit.
    recompute_mask_above: int = 8192
    # "fused" | "stage": which implementation the last forward() used; forward_packed: "fused_packed" | "per_sequence"
    # (diagnostics / benches)
    last_path = None

    def _init_v2(self, d_head, d_codeword, n_codewords):
        self.quantizer = PQV2(d_codeword=d_codeword, n_codewords=n_codewords, n_subspaces=d_head // d_codeword)
        self.register_buffer("trigger", torch.scalar_tensor(False, dtype=torch.bool))
        self._indptr_cache = {}

    @classmethod
    def _from_v1(cls, source, v1_type):
        assert isinstance(source, v1_type)
        model = cls(d_head=source.d_head, d_codeword=source.d_codeword,
                    n_codewords=source.n_codewords, p_dropout=0.0)
        result = model.load_state_dict(source.state_dict(), strict=False)
        if len(result.missing_keys) != 0:
            raise RuntimeError
        return model

    def _fixed_indptr(self, seq_length: int, top_k: int, device) -> torch.Tensor:
        key = (seq_length, top_k, str(device))
        hit = self._indptr_cache.get(key)
        if hit is None:  # the reference rebuilds this arange on every call (attention.py:116-119)
            hit = torch.arange(0, top_k * seq_length + 1, step=top_k, dtype=torch.int32, device=device)
            self._indptr_cache[key] = hit
        return hit

    @staticmethod
    def _to_heads(x: torch.Tensor) -> torch.Tensor:  # [N, S, H, E] -> [N*H, S, E]
        x = layout.swap12(x)                         # transpose(1, 2).contiguous() as 16-byte-word row moves
        return x.view(-1, x.size(-2), x.size(-1))

    def _fused_ok(self, q) -> bool:
        return (self.use_fused and q.is_cuda and q.dtype in (torch.bfloat16, torch.float16) and q.size(-1) in (64, 80, 128)
                and q.size(1) % 128 == 0 and q.size(1) % self.sparse_coeff == 0
                and (q.size(1) // self.sparse_coeff) % 4 == 0 and q.size(1) // self.sparse_coeff >= 8
                and q.size(1) <= ext.LOOKUP_MAX_SEQ)

    @staticmethod
    def _kv_group(q, k, v) -> int:
        """G = H // Hkv for grouped-query / multi-query attention: q [N, S, H, E] (packed: [1, T, H, E]) with k, v
        [N, S, Hkv, E], H % Hkv == 0; query head h attends with key / value head h // G (the contiguous grouping of HF
        LLaMA / Mistral repeat_kv, i.e. torch.repeat_interleave(k, G, dim=2)).  1 when q, k, v share one shape.
        Raises ValueError naming the broken rule."""
        if q.shape == k.shape == v.shape:
            return 1
        if k.shape != v.shape:
            raise ValueError(f"k and v must have the same shape (got k {tuple(k.shape)}, v {tuple(v.shape)})")
        if q.dim() != 4 or k.dim() != 4 or q.shape[:2] != k.shape[:2] or q.size(3) != k.size(3):
            raise ValueError(f"grouped-query attention needs q [N, S, H, E] and k, v [N, S, Hkv, E] with the same N, S and "
                             f"E (got q {tuple(q.shape)}, k {tuple(k.shape)})")
        if k.size(2) < 1 or q.size(2) % k.size(2):
            raise ValueError(f"the query head count H = {q.size(2)} must be a multiple of the key / value head count "
                             f"Hkv = {k.size(2)}")
        return q.size(2) // k.size(2)

    @staticmethod
    def _repeat_kv(k, v, G: int):
        """k, v repeated to H heads (HF repeat_kv): the multi-head input the grouped-query result is defined by."""
        return (k, v) if G == 1 else (k.repeat_interleave(G, dim=2), v.repeat_interleave(G, dim=2))

    @staticmethod
    def _encode_qk(q, k, weight):
        """quantizer('encode') of q and k: one launch for both when they share a shape, else (fewer key heads) one each."""
        if q.shape == k.shape:
            return ext.pq_encode_pair(q, k, weight)
        return ext.pq_encode(q, weight), ext.pq_encode(k, weight)

    def _maybe_train_loss(self, q, k):
        if self.host_trigger is not None:
            armed, self.host_trigger = bool(self.host_trigger), False
        else:
            armed = self.trigger.is_nonzero()  # one-shot PQ training loss, armed by the training loop
            if armed:
                self.trigger.logical_not_()
        if armed:
            loss = self.quantizer("train", z=q)[-1] + self.quantizer("train", z=k)[-1]
            self.register_buffer("loss", loss, persistent=False)

    def _fused_forward(self, q, k, v):
        # everything runs on the layer's native [N, S, H, E] layout: PQ encode is row-wise, lookup and
        # the attention kernels stride over the interleaved heads, so none of the reference's
        # transpose(1, 2).contiguous() copies (attention.py:92-95,138-142) is made
        q, k, v = q.contiguous(), k.contiguous(), v.contiguous()
        # PQ loss is a mean over rows: layout-invariant.  With fewer key heads (grouped-query attention) it runs on the
        # un-repeated k, whose mean equals that of the repeated k: every row appears G times there.
        self._maybe_train_loss(q, k)
        q_c, k_c = self._encode_qk(q, k, self.quantizer.weight)   # [N, S, H, m] and [N, S, Hkv, m]
        n_codewords = self.quantizer.weight.size(1)
        # [N, S, H, E]; with reference_output_layout the kernel writes the shipped layer's re-interpretation of
        # [N*H, E, S] memory itself (forward epilogue / backward row prologue): no permute pass either way
        if q.size(1) > self.recompute_mask_above:
            return kernels.sparse_attention_recompute(q, k, v, q_c, k_c, self.sparse_coeff, self.scaling,
                                                      reference_layout=self.reference_output_layout,
                                                      n_codewords=n_codewords)
        mask, extra0, _ = ext.lookup_mask(q_c, k_c, self.sparse_coeff, n_codewords=n_codewords)
        return kernels.sparse_attention(q, k, v, mask, extra0, self.scaling,
                                        reference_layout=self.reference_output_layout)

    def _packed_fused_ok(self, q, max_seqlen: int) -> bool:
        m = self.quantizer.weight.size(0)
        return (self.use_fused and q.is_cuda and q.dtype in (torch.bfloat16, torch.float16) and q.size(-1) in (64, 80, 128)
                and max_seqlen <= ext.lookup_mask_varlen_max_seqlen(m))

    def _rotate_packed(self, x, cu, max_seqlen=None):      # the rotary layer restarts positions at every sequence start
        return x

    def forward_packed(self, q, k, v, cu_seqlens, max_seqlen=None):
        """Packed variable-length sequences (INTEGRATION.md, "Packed sequences"): q, k, v [T, H, E] or [1, T, H, E] hold
        n sequences concatenated along the token axis; cu_seqlens [n + 1] their offsets (cu[0] = 0, cu[n] = T).  Sequence
        i (rows cu[i] .. cu[i+1]) gets exactly what forward() gives for it alone as a batch of one, in the same output
        layout; y has q's shape.
        cu_seqlens is a host list / CPU tensor (validated, then copied to the device: not capturable), or an int32 CUDA
        tensor together with max_seqlen (trusted, never synchronised on: capturable).  Lengths must be multiples of
        4 * sparse_coeff and of 32, and at least 8 * sparse_coeff.  Outside the fused envelope (or with use_fused =
        False) every sequence runs forward() on its own, after one synchronisation to read the offsets."""
        squeeze = q.dim() == 3
        q, k, v = (t.unsqueeze(0) if squeeze else t for t in (q, k, v))
        if q.dim() != 4 or q.size(0) != 1 or k.dim() != 4 or v.dim() != 4:
            raise ValueError("forward_packed: q, k, v must all be [T, H, E] or [1, T, H, E] (k, v: [T, Hkv, E] or "
                             "[1, T, Hkv, E] with H % Hkv == 0)")
        self._kv_group(q, k, v)
        T = q.size(1)
        if isinstance(cu_seqlens, torch.Tensor) and cu_seqlens.is_cuda:
            if max_seqlen is None:
                raise ValueError("forward_packed: a device cu_seqlens needs max_seqlen")
            cu, max_seqlen = cu_seqlens, int(max_seqlen)
        else:
            longest = ext.check_cu_seqlens(cu_seqlens, T, self.sparse_coeff, max_seqlen)
            max_seqlen = longest if max_seqlen is None else int(max_seqlen)
            host = cu_seqlens.tolist() if isinstance(cu_seqlens, torch.Tensor) else list(cu_seqlens)
            cu = torch.tensor([int(x) for x in host], dtype=torch.int32, device=q.device)
        if self._packed_fused_ok(q, max_seqlen):
            self.last_path = "fused_packed"
            q, k, v = self._rotate_packed(q, cu, max_seqlen), self._rotate_packed(k, cu, max_seqlen), v.contiguous()
            q, k = q.contiguous(), k.contiguous()
            self._maybe_train_loss(q, k)      # over all T rows (un-repeated k: see _fused_forward)
            q_c, k_c = self._encode_qk(q, k, self.quantizer.weight)
            n_codewords = self.quantizer.weight.size(1)
            if max_seqlen > self.recompute_mask_above:
                y = kernels.sparse_attention_varlen_recompute(q, k, v, q_c, k_c, cu, max_seqlen, self.sparse_coeff,
                                                              self.scaling, reference_layout=self.reference_output_layout,
                                                              n_codewords=n_codewords)
            else:
                mask, extra0 = ext.lookup_mask_varlen(q_c, k_c, cu, max_seqlen, self.sparse_coeff, n_codewords=n_codewords)
                y = kernels.sparse_attention_varlen(q, k, v, mask, extra0, cu, max_seqlen, self.scaling,
                                                    reference_layout=self.reference_output_layout)
        else:
            offs = [int(x) for x in cu.tolist()]
            y = torch.cat([self.forward(q[:, a:b], k[:, a:b], v[:, a:b]) for a, b in zip(offs[:-1], offs[1:])], dim=1)
            self.last_path = "per_sequence"
        return y.squeeze(0) if squeeze else y

    def _sparse_get_attn(self, q, k):
        assert q.size() == k.size()
        seq_length = q.size(1)
        q, k = self._to_heads(q), self._to_heads(k)
        self._maybe_train_loss(q, k)
        q_c = self.quantizer("encode", z=q)
        k_c = self.quantizer("encode", z=k)
        topk = kernels.lookup(q_c, k_c, sparse_coeff=self.sparse_coeff)
        csr_indices = topk.flatten(start_dim=1)
        indptr = self._fixed_indptr(seq_length, seq_length // self.sparse_coeff, q.device)
        # sddmm + scale + clamp(-10, 10) of attention.py:122-127 in one kernel each way (no eager elementwise passes)
        # (kernels.sddmm_softmax = kernels.sddmm_scaled + kernels.softmax with a one-pass backward from the gradient of
        # the probabilities to the gradient of the raw scores)
        values = kernels.sddmm_softmax(indptr, csr_indices, q, k, self.scaling, 10.0)
        return indptr, csr_indices, values

    def _stage_forward(self, q, k, v, attn_mask):
        # the stage kernels take fp32 / bf16: fp16 operands run the chain in fp32 and the result goes back to fp16
        if q.dtype == torch.float16:
            return VanillaAttention.forward(self, q.float(), k.float(), v.float(), attn_mask).to(q.dtype)
        return VanillaAttention.forward(self, q, k, v, attn_mask)

    def _apply_attn(self, attn, v):
        v_size = v.size()
        indptr, indices, values = attn
        y = kernels.spmm(indptr, indices, values, self._to_heads(v))
        if self.reference_output_layout:
            return layout.transpose_last2(y).view(v_size)
        return layout.swap12(y.view(v_size[0], v_size[2], v_size[1], v_size[3])).view(v_size)


class SparseVanillaAttentionV2(_SparseV2Mixin, VanillaAttention):
    def __init__(self, d_head: int, d_codeword: int, n_codewords: int, p_dropout: float,
                 reference_output_layout: bool = True):
        VanillaAttention.__init__(self, d_head=d_head, p_dropout=p_dropout)
        self._init_v2(d_head, d_codeword, n_codewords)
        self.reference_output_layout = reference_output_layout

    @staticmethod
    def from_pretrained(source: SparseVanillaAttentionV1):
        return SparseVanillaAttentionV2._from_v1(source, SparseVanillaAttentionV1)

    def _get_attn(self, q, k, attn_mask):  # attn_mask is ignored: the path is always causal
        return self._sparse_get_attn(q, k)

    def forward(self, q, k, v, attn_mask=None):
        G = self._kv_group(q, k, v)
        if self._fused_ok(q):
            self.last_path = "fused"
            return self._fused_forward(q, k, v)
        self.last_path = "stage"
        return self._stage_forward(q, *self._repeat_kv(k, v, G), attn_mask)


class SparseRotaryAttentionV2(_SparseV2Mixin, RotaryAttention):
    def __init__(self, d_head: int, p_dropout: float, d_codeword: int, n_codewords: int,
                 reference_output_layout: bool = True):
        RotaryAttention.__init__(self, d_head=d_head, p_dropout=p_dropout)
        self._init_v2(d_head, d_codeword, n_codewords)
        self.reference_output_layout = reference_output_layout

    @staticmethod
    def from_pretrained(source: SparseRotaryAttentionV1):
        return SparseRotaryAttentionV2._from_v1(source, SparseRotaryAttentionV1)

    def _get_attn(self, q, k, attn_mask):
        return self._sparse_get_attn(self._rotate(q), self._rotate(k))

    def _rotate_packed(self, x, cu, max_seqlen=None):
        # position of token t = t - cu[sequence of t], built on the device (no host synchronisation); max_seqlen (> every
        # position) extends the rotation tables where it exceeds them
        t = torch.arange(x.size(1), dtype=torch.int32, device=x.device)
        ids = (t - cu[torch.searchsorted(cu, t, right=True) - 1]).long()
        return self.embedding(x, ids=ids, n_positions=max_seqlen).to(x.dtype)

    def forward(self, q, k, v, attn_mask=None):
        G = self._kv_group(q, k, v)
        if self._fused_ok(q):
            self.last_path = "fused"
            # fp32 rotation tables promote a bf16 input to fp32 (as in the reference); the fused kernels take the rotated
            # operands in the input's own dtype (k at its own head count)
            return self._fused_forward(self._rotate(q).to(q.dtype), self._rotate(k).to(k.dtype), v)
        self.last_path = "stage"
        return self._stage_forward(q, *self._repeat_kv(k, v, G), attn_mask)
