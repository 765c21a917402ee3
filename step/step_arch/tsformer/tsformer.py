"""TSFormer on the B200-native kernels (drop-in for the reference module of the same name).

Same constructor / ``forward`` signature and the same 72 state-dict keys as the reference
(``step/step_arch/tsformer/tsformer.py:21-191``, checkpoint contract in SURVEY.md Appx C), so
``tsformer_ckpt/*.pt`` load with ``strict=True``.  The sub-modules below only *hold parameters*
under the reference's names; the arithmetic is ``step_b200.ops.ts_encoder_forward`` (hand-written
sm_100a kernels).  There is no PyTorch fallback.
"""
import math
import os

import torch
from torch import nn

from step_b200 import ops


class _AttnParams(nn.Module):
    """Parameter holder with nn.MultiheadAttention's names (in_proj_weight/in_proj_bias/out_proj)."""

    def __init__(self, dim):
        super().__init__()
        self.in_proj_weight = nn.Parameter(torch.empty(3 * dim, dim))
        self.in_proj_bias = nn.Parameter(torch.zeros(3 * dim))
        self.out_proj = nn.Linear(dim, dim)
        nn.init.xavier_uniform_(self.in_proj_weight)
        nn.init.zeros_(self.out_proj.bias)


class _EncoderLayerParams(nn.Module):
    """Parameter holder with nn.TransformerEncoderLayer's names."""

    def __init__(self, dim, hidden):
        super().__init__()
        self.self_attn = _AttnParams(dim)
        self.linear1 = nn.Linear(dim, hidden)
        self.linear2 = nn.Linear(hidden, dim)
        self.norm1 = nn.LayerNorm(dim)
        self.norm2 = nn.LayerNorm(dim)

    def kernel_weights(self):
        return {"in_proj_w": self.self_attn.in_proj_weight, "in_proj_b": self.self_attn.in_proj_bias,
                "out_proj_w": self.self_attn.out_proj.weight, "out_proj_b": self.self_attn.out_proj.bias,
                "lin1_w": self.linear1.weight, "lin1_b": self.linear1.bias,
                "lin2_w": self.linear2.weight, "lin2_b": self.linear2.bias,
                "norm1_w": self.norm1.weight, "norm1_b": self.norm1.bias,
                "norm2_w": self.norm2.weight, "norm2_b": self.norm2.bias}


class _LayerList(nn.Module):
    def __init__(self, dim, hidden, depth):
        super().__init__()
        self.layers = nn.ModuleList([_EncoderLayerParams(dim, hidden) for _ in range(depth)])


class TransformerLayers(nn.Module):
    """Holds ``transformer_encoder.layers.{i}.*`` (reference: tsformer/transformer_layers.py:6-20)."""

    def __init__(self, hidden_dim, nlayers, mlp_ratio, num_heads=4, dropout=0.1):
        super().__init__()
        self.d_model = hidden_dim
        self.num_heads = num_heads
        self.dropout = dropout
        self.transformer_encoder = _LayerList(hidden_dim, hidden_dim * mlp_ratio, nlayers)

    def kernel_weights(self):
        return [layer.kernel_weights() for layer in self.transformer_encoder.layers]


class PatchEmbedding(nn.Module):
    """Holds ``input_embedding.{weight,bias}`` (reference: tsformer/patch.py:4-42)."""

    def __init__(self, patch_size, in_channel, embed_dim, norm_layer=None):
        super().__init__()
        self.len_patch = patch_size
        self.input_channel = in_channel
        self.output_channel = embed_dim
        self.input_embedding = nn.Conv2d(in_channel, embed_dim, kernel_size=(patch_size, 1), stride=(patch_size, 1))


class PositionalEncoding(nn.Module):
    """Holds ``position_embedding`` (reference: tsformer/positional_encoding.py:5-35)."""

    def __init__(self, hidden_dim, dropout=0.1, max_len: int = 1000):
        super().__init__()
        self.p = dropout
        self.position_embedding = nn.Parameter(torch.empty(max_len, hidden_dim), requires_grad=True)


class MaskGenerator(nn.Module):
    """Uniform random patch masking (reference: tsformer/mask.py:6-29): a shuffled ``range(num_tokens)`` from
    Python's ``random`` module, the first ``int(num_tokens * mask_ratio)`` entries are masked; both index lists are
    returned sorted.  ``fixed`` (a pair of index lists) pins the draw for parity tests."""

    def __init__(self, num_tokens, mask_ratio):
        super().__init__()
        self.num_tokens, self.mask_ratio, self.sort = num_tokens, mask_ratio, True
        self.fixed = None
        self.masked_tokens, self.unmasked_tokens = None, None

    def uniform_rand(self):
        import random
        order = list(range(int(self.num_tokens)))
        random.shuffle(order)
        n_masked = int(self.num_tokens * self.mask_ratio)
        masked, unmasked = order[:n_masked], order[n_masked:]
        if self.sort:
            masked, unmasked = sorted(masked), sorted(unmasked)
        self.masked_tokens, self.unmasked_tokens = masked, unmasked
        return unmasked, masked

    def forward(self):
        if self.fixed is not None:
            self.unmasked_tokens, self.masked_tokens = list(self.fixed[0]), list(self.fixed[1])
            return self.unmasked_tokens, self.masked_tokens
        return self.uniform_rand()


class TSFormer(nn.Module):
    """Masked-patch transformer for long time series; ``mode="forecasting"`` is the STEP hot path."""

    def __init__(self, patch_size, in_channel, embed_dim, num_heads, mlp_ratio, dropout, num_token, mask_ratio,
                 encoder_depth, decoder_depth, mode="pre-train"):
        super().__init__()
        assert mode in ["pre-train", "forecasting"], "Error mode."
        if (patch_size, in_channel, embed_dim, num_heads, mlp_ratio) != (12, 1, 96, 4, 4):
            raise NotImplementedError(
                "step_b200 kernels are specialised for the STEP configuration patch_size=12, in_channel=1, "
                "embed_dim=96, num_heads=4, mlp_ratio=4 (every shipped STEP_*.py / TSFormer_*.py config)")
        self.patch_size, self.in_channel, self.embed_dim, self.num_heads = patch_size, in_channel, embed_dim, num_heads
        self.num_token, self.mask_ratio, self.encoder_depth, self.mode, self.mlp_ratio = \
            num_token, mask_ratio, encoder_depth, mode, mlp_ratio
        self.dropout_p = dropout
        self.selected_feature = 0
        self.encoder_norm = nn.LayerNorm(embed_dim)
        self.decoder_norm = nn.LayerNorm(embed_dim)
        self.patch_embedding = PatchEmbedding(patch_size, in_channel, embed_dim, norm_layer=None)
        self.positional_encoding = PositionalEncoding(embed_dim, dropout=dropout)
        self.mask = MaskGenerator(num_token, mask_ratio)
        self.encoder = TransformerLayers(embed_dim, encoder_depth, mlp_ratio, num_heads, dropout)
        self.enc_2_dec_emb = nn.Linear(embed_dim, embed_dim, bias=True)
        self.mask_token = nn.Parameter(torch.zeros(1, 1, 1, embed_dim))
        self.decoder = TransformerLayers(embed_dim, decoder_depth, mlp_ratio, num_heads, dropout)
        self.output_layer = nn.Linear(embed_dim, patch_size)
        # kernel launch options
        self.chunk_seqs = 0          # fp32 path: sequences per L2-resident chunk (0 = all at once)
        # "bf16": tcgen05 tensor-core kernels (bf16 operands, fp32 accumulation/statistics) - the performance path;
        # "fp32": CUDA-core kernels that meet the 1e-4 parity bar against the reference.
        self.precision = os.environ.get("STEP_B200_PRECISION", "bf16")
        # stage-1 training (pretrain_forward_autograd) only: "bf16" runs the attention of every layer with P' <= 352 on
        # tcgen05 (bf16 operands, fp32 accumulation/statistics); "fp32" keeps the CUDA-core attention kernels.
        self.pretrain_precision = os.environ.get("STEP_B200_PRETRAIN_PRECISION", "fp32")
        self._tc_images = None
        self._tc_key = None
        self.seq_image = None        # bf16 Gram operand of the last bf16 forward ([B][P*12][R][8]); None in fp32 mode
        # node-sharded mode (STEP_PEMS07 on several GPUs): (rank, world) -> this rank encodes only its node range and
        # the hidden states are assembled with one NCCL all-gather (step_b200.parallel.all_gather_nodes)
        self.node_shard = None
        self.gathered_patches = None  # node-parallel bf16 path: P of the sequence image (hidden then holds the last patch only)
        self._calls = 0
        self.initialize_weights()

    def initialize_weights(self):
        nn.init.uniform_(self.positional_encoding.position_embedding, -.02, .02)
        nn.init.trunc_normal_(self.mask_token, std=.02)

    def _next_seed(self):
        self._calls += 1
        return (torch.initial_seed() + 0x9E3779B1 * self._calls) & (2 ** 63 - 1)

    def encoding(self, long_term_history, mask=False):
        """long_term_history: [B, N, 1, P*L] view -> hidden states [B, N, P, d] (no masking on this path)."""
        if mask:
            raise NotImplementedError("the masked encoding is fused into pretrain_forward(); call forward() in mode='pre-train'")
        series = long_term_history[:, :, 0, :].permute(0, 2, 1)      # [B, P*L, N] view, no copy
        num_nodes = series.shape[2]
        if self.node_shard is not None:
            from step_b200 import parallel
            rank, world = self.node_shard
            n0, n1 = parallel.node_shard_bounds(num_nodes, rank, world)
            series = series[:, :, n0:n1]
        drop = self.dropout_p if self.training else 0.0
        seed = self._next_seed() if drop > 0 else 0
        emb = self.patch_embedding.input_embedding
        layers = self.encoder.kernel_weights()
        if self.precision not in ("bf16", "fp32"):
            raise ValueError(f"TSFormer.precision must be 'bf16' or 'fp32', got {self.precision!r}")
        if self.precision == "bf16" and series.shape[1] // self.patch_size <= 352:
            key = (series.device, tuple(int(w._version) for lw in layers for w in lw.values()),
                   tuple(w.data_ptr() for lw in layers for w in lw.values()))
            if self._tc_key != key:           # frozen weights: packed into UMMA images once
                self._tc_images = ops.ts_pack_layer_images(layers)
                self._tc_key = key
            hidden, self.seq_image = ops.ts_encoder_forward_bf16(
                series, emb.weight, emb.bias, self.positional_encoding.position_embedding, layers, self._tc_images,
                self.encoder_norm.weight, self.encoder_norm.bias, drop_p=drop, seed=seed, want_seq_image=True)
        else:
            # fp32 kernels (also serve P > 352: the tensor-core attention holds at most two 176-key blocks in TMEM)
            self.seq_image = None
            hidden = ops.ts_encoder_forward(series, emb.weight, emb.bias, self.positional_encoding.position_embedding, layers,
                                            self.encoder_norm.weight, self.encoder_norm.bias, drop_p=drop, seed=seed,
                                            chunk_seqs=self.chunk_seqs)
        if self.node_shard is not None and self.node_shard[1] > 1:
            from step_b200 import parallel
            rank, world = self.node_shard
            if self.precision == "bf16" and self.seq_image is not None:
                # node-parallel, bf16 path: ONE all-gather of the bf16 Gram operand image (half the bytes of the fp32 states)
                # plus the last-patch states the forecaster consumes ([B,N,1,96], 0.3 % of the states).  STEP only reads
                # hidden[:, :, -1, :] (reference step.py:58), which this [B,N,1,96] tensor serves.
                B, P = hidden.shape[0], hidden.shape[2]
                self.seq_image = parallel.all_gather_seq_image(self.seq_image, B, P * 12, num_nodes, rank, world)
                hidden = parallel.gather_node_rows(hidden[:, :, -1:, :], num_nodes, rank, world)
                self.gathered_patches = P
            else:
                hidden = parallel.all_gather_nodes(hidden, num_nodes, rank, world)
                self.seq_image = ops.tc_hidden_to_seq_image(hidden) if self.precision == "bf16" and hidden.shape[2] * 12 % 8 == 0 else None
        return hidden, None, None

    @torch.no_grad()
    def pretrain_forward(self, history_data):
        """``mode="pre-train"`` forward (reference tsformer.py:71-160): embed all patches, encode the unmasked 25 %,
        ``enc_2_dec_emb``, append mask tokens (+ positional embedding of the masked positions), one decoder layer,
        ``decoder_norm``, ``output_layer``; returns (reconstruction of the masked patches, their ground truth), both
        ``[B, r*P*L, N]``.  Inference flavour on the fused fp32 kernels (no autograd graph); training goes through
        :meth:`pretrain_forward_autograd`.
        history_data: [B, N, 1, P*L] view."""
        B, N, _, T = history_data.shape
        L, d = self.patch_size, self.embed_dim
        P = T // L
        S = B * N
        series = history_data[:, :, 0, :].permute(0, 2, 1)          # [B, P*L, N] view
        drop = self.dropout_p if self.training else 0.0
        seed = self._next_seed() if drop > 0 else 0
        emb, pos = self.patch_embedding.input_embedding, self.positional_encoding.position_embedding
        unmasked, masked = self.mask()
        dev = history_data.device
        ui = torch.as_tensor(unmasked, device=dev, dtype=torch.long)
        mi = torch.as_tensor(masked, device=dev, dtype=torch.long)
        # --- encoder over the unmasked tokens (tokens already carry the sqrt(d) scale of transformer_layers.py:15)
        tokens = ops.ts_embed(series, emb.weight, emb.bias, pos, drop_p=drop, seed=seed).view(S, P, d)
        enc_in = tokens.index_select(1, ui).reshape(S * len(unmasked), d)
        hidden_u = ops.ts_layers(enc_in, S, len(unmasked), self.encoder.kernel_weights(), self.encoder_norm.weight,
                                 self.encoder_norm.bias, drop_p=drop, seed=seed + 1)
        # --- decoder over [unmasked | mask tokens]
        dec_u = ops.linear(hidden_u, self.enc_2_dec_emb.weight, self.enc_2_dec_emb.bias).view(S, len(unmasked), d)
        dec_m = (self.mask_token.view(1, 1, d) + pos[mi].unsqueeze(0)).expand(S, len(masked), d)
        if drop > 0:
            dec_m = torch.nn.functional.dropout(dec_m, drop, training=True)      # positional_encoding.py:32
        full = (torch.cat([dec_u, dec_m], dim=1) * math.sqrt(d)).reshape(S * P, d)
        hidden_f = ops.ts_layers(full, S, P, self.decoder.kernel_weights(), self.decoder_norm.weight,
                                 self.decoder_norm.bias, drop_p=drop, seed=seed + 2)
        recon = ops.linear(hidden_f, self.output_layer.weight, self.output_layer.bias).view(B, N, P, L)
        # --- masked tokens vs ground truth (tsformer.py:138-160)
        recon_masked = recon[:, :, len(unmasked):, :].reshape(B, N, -1).transpose(1, 2)
        label = history_data[:, :, self.selected_feature, :].reshape(B, N, P, L).index_select(2, mi)
        label_masked = label.reshape(B, N, -1).transpose(1, 2)
        return recon_masked, label_masked

    def _pretrain_tc_attention(self, seq_len: int) -> bool:
        """Whether stage-1 training runs the attention of a layer over `seq_len` tokens on the tensor cores: pretrain_precision
        "bf16" and seq_len <= 352 (longer sequences keep the fp32 kernels, as in :meth:`encoding`)."""
        if self.pretrain_precision not in ("bf16", "fp32"):
            raise ValueError(f"TSFormer.pretrain_precision must be 'bf16' or 'fp32', got {self.pretrain_precision!r}")
        return self.pretrain_precision == "bf16" and seq_len <= 352

    def pretrain_forward_autograd(self, history_data):
        """The same ``mode="pre-train"`` computation as :meth:`pretrain_forward`, built from differentiable ops (every one
        a hand-written kernel behind ``step_b200.ops``: split-bf16 tcgen05 GEMMs for the dense layers, fp32 attention /
        LayerNorm / dropout kernels with hand-written backward; with ``pretrain_precision="bf16"`` the attention runs on
        tcgen05 instead) so that stage 1 of STEP - the masked auto-encoder of reference tsformer.py:71-160 - trains on
        the GPU.  Gradients reach all 72 parameters."""
        B, N, _, T = history_data.shape
        L, d = self.patch_size, self.embed_dim
        P = T // L
        S = B * N
        drop = self.dropout_p if self.training else 0.0
        seed = self._next_seed() if drop > 0 else 0
        emb, pos = self.patch_embedding.input_embedding, self.positional_encoding.position_embedding
        unmasked, masked = self.mask()
        dev = history_data.device
        ui = torch.as_tensor(unmasked, device=dev, dtype=torch.long)
        mi = torch.as_tensor(masked, device=dev, dtype=torch.long)
        nu, nm = len(unmasked), len(masked)
        tc_attn = self._pretrain_tc_attention
        # --- patch + positional embedding (dropout on every token, positional_encoding.py:32), keep the unmasked 25 %
        patches = history_data[:, :, self.selected_feature, :].reshape(S * P, L)
        tok = ops.Linear.apply(patches, emb.weight.view(d, L), emb.bias, False).view(S, P, d) + pos[:P]
        tok = ops.dropout(tok.reshape(S * P, d), drop, seed, 1).view(S, P, d)
        z = (tok.index_select(1, ui) * math.sqrt(d)).reshape(S * nu, d)
        for i, lw in enumerate(self.encoder.kernel_weights()):
            z = ops.transformer_layer_train(z, S, nu, lw, drop, seed, 16 * (i + 1), tc_attention=tc_attn(nu))
        z = ops.AddLayerNorm.apply(z, None, self.encoder_norm.weight, self.encoder_norm.bias)
        # --- decoder over [unmasked | mask tokens + positional embedding of the masked positions]
        dec_u = ops.Linear.apply(z, self.enc_2_dec_emb.weight, self.enc_2_dec_emb.bias, False).view(S, nu, d)
        dec_m = (self.mask_token.view(1, 1, d) + pos[mi].unsqueeze(0)).expand(S, nm, d)
        dec_m = ops.dropout(dec_m.reshape(S * nm, d), drop, seed, 2).view(S, nm, d)
        z = (torch.cat([dec_u, dec_m], dim=1) * math.sqrt(d)).reshape(S * P, d)
        for i, lw in enumerate(self.decoder.kernel_weights()):
            z = ops.transformer_layer_train(z, S, P, lw, drop, seed, 160 + 16 * i, tc_attention=tc_attn(P))
        z = ops.AddLayerNorm.apply(z, None, self.decoder_norm.weight, self.decoder_norm.bias)
        recon = ops.Linear.apply(z, self.output_layer.weight, self.output_layer.bias, False).view(B, N, P, L)
        recon_masked = recon[:, :, nu:, :].reshape(B, N, -1).transpose(1, 2)
        label = history_data[:, :, self.selected_feature, :].reshape(B, N, P, L).index_select(2, mi)
        return recon_masked, label.reshape(B, N, -1).transpose(1, 2)

    def forward(self, history_data: torch.Tensor, future_data: torch.Tensor = None, batch_seen: int = None,
                epoch: int = None, **kwargs) -> torch.Tensor:
        """history_data: [B, L*P, N, 1].  forecasting mode -> [B, N, P, d]."""
        history_data = history_data.permute(0, 2, 3, 1)     # B, N, 1, L*P (view)
        if self.mode == "pre-train":
            if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
                return self.pretrain_forward_autograd(history_data)       # stage-1 training
            return self.pretrain_forward(history_data)                    # inference: fused kernels, no graph
        with torch.no_grad():
            hidden_states_full, _, _ = self.encoding(history_data, mask=False)
        return hidden_states_full
