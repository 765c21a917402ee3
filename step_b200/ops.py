"""Tensor-level wrappers and autograd glue over the C ABI (include/step_b200.h).

PyTorch is used here only for device memory, streams and autograd bookkeeping; every
numeric hot op below is a hand-written sm_100a kernel reached through ctypes.  No op in this
file has a PyTorch/CPU fallback: a CPU tensor or a missing library raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence

import torch

from . import lib as _lib
from .lib import GwLayerGrads, GwLayerParams, TsLayerWeights, check

Tensor = torch.Tensor

# counters the benchmark reads: how many of OUR kernels were launched (host-side count)
launch_counter = {"kernels": 0}


def _L():
    return _lib.load()


def _f32(t: Tensor, name: str) -> Tensor:
    if not t.is_cuda:
        raise _lib.StepB200Error(f"{name}: expected a CUDA tensor - step_b200 has no CPU path")
    if t.dtype != torch.float32:
        raise _lib.StepB200Error(f"{name}: expected float32, got {t.dtype}")
    return t.contiguous()


def _p(t: Optional[Tensor]):
    return None if t is None else t.data_ptr()


def _enter(t: Tensor):
    """Select the tensor's device in the library's CUDA runtime and return the current torch stream."""
    check(_L().step_set_device(t.device.index), "step_set_device")
    return torch.cuda.current_stream(t.device).cuda_stream


# --------------------------------------------------------------------------- #
# TSFormer encoder
# --------------------------------------------------------------------------- #
def ts_layer_struct(layers: Sequence[Dict[str, Tensor]]):
    arr = (TsLayerWeights * len(layers))()
    keep = []
    for i, lw in enumerate(layers):
        for name in ("in_proj_w", "in_proj_b", "out_proj_w", "out_proj_b", "lin1_w", "lin1_b", "lin2_w", "lin2_b",
                     "norm1_w", "norm1_b", "norm2_w", "norm2_b"):
            t = _f32(lw[name], name)
            keep.append(t)
            setattr(arr[i], name, t.data_ptr())
    return arr, keep


def ts_encoder_forward(series: Tensor, patch_w: Tensor, patch_b: Tensor, pos: Tensor, layers: Sequence[Dict[str, Tensor]],
                       norm_w: Tensor, norm_b: Tensor, drop_p: float = 0.0, seed: int = 0, chunk_seqs: int = 0) -> Tensor:
    """series: [B, P*12, N] float32 view (any strides) -> hidden [B, N, P, 96]."""
    if not series.is_cuda or series.dtype != torch.float32:
        raise _lib.StepB200Error("ts_encoder_forward: series must be a float32 CUDA tensor")
    B, T, N = series.shape
    if T % 12 != 0:
        raise _lib.StepB200Error(f"ts_encoder_forward: history length {T} is not a multiple of the patch size 12")
    P = T // 12
    st = _enter(series)
    hidden = torch.empty(B, N, P, 96, device=series.device, dtype=torch.float32)
    S = B * N
    chunk = S if chunk_seqs <= 0 else min(chunk_seqs, S)
    ws_bytes = _L().step_ts_encoder_workspace_bytes(chunk, P)
    ws = torch.empty(ws_bytes, device=series.device, dtype=torch.uint8)
    arr, keep = ts_layer_struct(layers)
    pw, pb, ps = _f32(patch_w.reshape(96, 12), "patch_w"), _f32(patch_b, "patch_b"), _f32(pos, "pos")
    nw, nb = _f32(norm_w, "norm_w"), _f32(norm_b, "norm_b")
    sB, sT, sN = series.stride()
    check(_L().step_ts_encoder_fwd(series.data_ptr(), sB, sT, sN, B, N, P, pw.data_ptr(), pb.data_ptr(), ps.data_ptr(),
                                   arr, len(layers), nw.data_ptr(), nb.data_ptr(), hidden.data_ptr(), ws.data_ptr(),
                                   ws_bytes, chunk, float(drop_p), int(seed) & (2**64 - 1), st), "step_ts_encoder_fwd")
    n_chunks = (S + chunk - 1) // chunk
    launch_counter["kernels"] += 1 + n_chunks * len(layers) * 5
    return hidden


def ts_embed(series: Tensor, patch_w: Tensor, patch_b: Tensor, pos: Tensor, drop_p: float = 0.0, seed: int = 0) -> Tensor:
    """Patch + positional embedding (x sqrt(96), positional dropout): series [B, P*12, N] view -> tokens [B*N*P, 96]."""
    if not series.is_cuda or series.dtype != torch.float32:
        raise _lib.StepB200Error("ts_embed: series must be a float32 CUDA tensor")
    B, T, N = series.shape
    if T % 12 != 0:
        raise _lib.StepB200Error(f"ts_embed: history length {T} is not a multiple of the patch size 12")
    P = T // 12
    st = _enter(series)
    x = torch.empty(B * N * P, 96, device=series.device, dtype=torch.float32)
    pw, pb, ps = _f32(patch_w.reshape(96, 12), "patch_w"), _f32(patch_b, "patch_b"), _f32(pos, "pos")
    sB, sT, sN = series.stride()
    check(_L().step_ts_embed_fwd(series.data_ptr(), sB, sT, sN, B, N, P, pw.data_ptr(), pb.data_ptr(), ps.data_ptr(),
                                 x.data_ptr(), float(drop_p), int(seed) & (2**64 - 1), st), "step_ts_embed_fwd")
    launch_counter["kernels"] += 1
    return x


def ts_layers(x: Tensor, S: int, P: int, layers: Sequence[Dict[str, Tensor]], norm_w: Optional[Tensor] = None,
              norm_b: Optional[Tensor] = None, drop_p: float = 0.0, seed: int = 0) -> Tensor:
    """Transformer layer stack (+ optional final LayerNorm) on tokens x [S*P, 96] (already x sqrt(96)); returns a new tensor."""
    x = _f32(x, "x").clone()
    if x.shape != (S * P, 96):
        raise _lib.StepB200Error(f"ts_layers: x must be [{S * P}, 96], got {tuple(x.shape)}")
    st = _enter(x)
    ws_bytes = _L().step_ts_encoder_workspace_bytes(S, P)
    ws = torch.empty(ws_bytes, device=x.device, dtype=torch.uint8)
    arr, keep = ts_layer_struct(layers)
    nw = _f32(norm_w, "norm_w") if norm_w is not None else None
    nb = _f32(norm_b, "norm_b") if norm_b is not None else None
    check(_L().step_ts_layers_fwd(x.data_ptr(), S, P, arr, len(layers), _p(nw), _p(nb), ws.data_ptr(), ws_bytes,
                                  float(drop_p), int(seed) & (2**64 - 1), st), "step_ts_layers_fwd")
    launch_counter["kernels"] += len(layers) * 5
    return x


def linear(a: Tensor, w: Tensor, bias: Optional[Tensor], epilogue: int = 0, residual: Optional[Tensor] = None,
           ln_w: Optional[Tensor] = None, ln_b: Optional[Tensor] = None, drop_p: float = 0.0, seed: int = 0) -> Tensor:
    a = _f32(a, "a"); w = _f32(w, "w")
    M, K = a.shape
    Nout = w.shape[0]
    st = _enter(a)
    c = torch.empty(M, Nout, device=a.device, dtype=torch.float32)
    check(_L().step_linear_f32(a.data_ptr(), w.data_ptr(), _p(bias), c.data_ptr(), M, K, Nout, epilogue, _p(residual),
                               _p(ln_w), _p(ln_b), float(drop_p), int(seed) & (2**64 - 1), 7, st), "step_linear_f32")
    launch_counter["kernels"] += 1
    return c


def attention(qkv: Tensor, S: int, P: int, drop_p: float = 0.0, seed: int = 0) -> Tensor:
    qkv = _f32(qkv, "qkv")
    st = _enter(qkv)
    out = torch.empty(S * P, 96, device=qkv.device, dtype=torch.float32)
    check(_L().step_attn_fwd_f32(qkv.data_ptr(), out.data_ptr(), S, P, float(drop_p), int(seed), 0, st), "step_attn_fwd_f32")
    launch_counter["kernels"] += 1
    return out


# --------------------------------------------------------------------------- #
# differentiable building blocks of the TSFormer pre-training path (stage 1)
# --------------------------------------------------------------------------- #
class Attention(torch.autograd.Function):
    """softmax(q k^T / sqrt(24)) v over S sequences of P tokens, 4 heads (fp32 kernels), with hand-written backward;
    attention-probability dropout is regenerated in backward from (seed, site 0)."""

    @staticmethod
    def forward(ctx, qkv, S, P, drop_p, seed):
        qkv = _f32(qkv, "qkv")
        out = attention(qkv, S, P, drop_p, seed)
        ctx.save_for_backward(qkv, out)
        ctx.cfg = (int(S), int(P), float(drop_p), int(seed))
        return out

    @staticmethod
    def backward(ctx, dout):
        qkv, out = ctx.saved_tensors
        S, P, drop_p, seed = ctx.cfg
        dout = _f32(dout, "dout")
        st = _enter(qkv)
        scratch = torch.empty(S * 4 * P * 2, device=qkv.device, dtype=torch.float32)
        dqkv = torch.empty_like(qkv)
        check(_L().step_attn_bwd_f32(qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), S, P, drop_p, seed, 0, scratch.data_ptr(),
                                     dqkv.data_ptr(), st), "step_attn_bwd_f32")
        launch_counter["kernels"] += 2
        return dqkv, None, None, None, None


ATTN_TC_MAX_P = 352     # longest sequence the tensor-core attention holds (K and V of one head stay in shared memory)


def attention_tc_pack(qkv: Tensor, S: int, P: int, bound: bool = False):
    """fp32 qkv rows [S*P, 288] -> (q_img, k_img, v_img[, bound]) bf16 operand images of the tensor-core attention."""
    qkv = _f32(qkv, "qkv")
    st = _enter(qkv)
    L = _L()
    q_img = torch.empty(L.step_tc_attn_image_bytes(S, P, 0), device=qkv.device, dtype=torch.uint8)
    k_img = torch.empty(L.step_tc_attn_image_bytes(S, P, 1), device=qkv.device, dtype=torch.uint8)
    v_img = torch.empty_like(k_img)
    bnd = torch.empty(L.step_tc_attn_image_bytes(S, P, 2) // 4, device=qkv.device, dtype=torch.float32) if bound else None
    check(L.step_tc_attn_train_pack(qkv.data_ptr(), S, P, q_img.data_ptr(), k_img.data_ptr(), v_img.data_ptr(), _p(bnd), st),
          "step_tc_attn_train_pack")
    launch_counter["kernels"] += 1
    return (q_img, k_img, v_img, bnd) if bound else (q_img, k_img, v_img)


def attention_tc_keep_mask(S: int, P: int, drop_p: float, seed: int, device) -> Tensor:
    """[S, 4, P, P] uint8, 1 where AttentionTC keeps the attention probability (query row, key column) - for tests."""
    mask = torch.empty(S, 4, P, P, device=device, dtype=torch.uint8)
    st = _enter(mask)
    check(_L().step_tc_attn_train_keep_mask(S, P, float(drop_p), int(seed) & (2**64 - 1), mask.data_ptr(), st),
          "step_tc_attn_train_keep_mask")
    return mask


class AttentionTC(torch.autograd.Function):
    """Same contract as :class:`Attention` (qkv [S*P, 288] -> [S*P, 96]) on tcgen05: bf16 Q/K/V operands, fp32 accumulation
    and softmax statistics, P <= 352.  Keeps the operand images, O and the per-row log2-sum-exp for the backward, which
    recomputes the probabilities on the tensor cores.  Attention-probability dropout uses the tensor-core counter hash
    (not :class:`Attention`'s Philox stream: same distribution, different masks)."""

    @staticmethod
    def forward(ctx, qkv, S, P, drop_p, seed):
        S, P = int(S), int(P)
        if P > ATTN_TC_MAX_P:
            raise _lib.StepB200Error(f"AttentionTC: P={P} > {ATTN_TC_MAX_P}; use Attention")
        q_img, k_img, v_img = attention_tc_pack(qkv, S, P)
        out = torch.empty(S * P, 96, device=qkv.device, dtype=torch.float32)
        lse = torch.empty(S * 4 * P, device=qkv.device, dtype=torch.float32)
        seed = int(seed) & (2**64 - 1)
        st = _enter(qkv)
        check(_L().step_tc_attn_train_fwd(q_img.data_ptr(), k_img.data_ptr(), v_img.data_ptr(), S, P, float(drop_p), seed,
                                          out.data_ptr(), lse.data_ptr(), st), "step_tc_attn_train_fwd")
        launch_counter["kernels"] += 1
        ctx.save_for_backward(q_img, k_img, v_img, out, lse)
        ctx.cfg = (S, P, float(drop_p), seed)
        return out

    @staticmethod
    def backward(ctx, dout):
        q_img, k_img, v_img, out, lse = ctx.saved_tensors
        S, P, drop_p, seed = ctx.cfg
        dout = _f32(dout, "dout")
        st = _enter(dout)
        dqkv = torch.empty(S * P, 288, device=dout.device, dtype=torch.float32)
        check(_L().step_tc_attn_train_bwd(q_img.data_ptr(), k_img.data_ptr(), v_img.data_ptr(), out.data_ptr(), lse.data_ptr(),
                                          dout.data_ptr(), S, P, drop_p, seed, dqkv.data_ptr(), st), "step_tc_attn_train_bwd")
        launch_counter["kernels"] += 1
        return dqkv, None, None, None, None


class AddLayerNorm(torch.autograd.Function):
    """LayerNorm96(x + r) (r may be None): the post-norm residual blocks and the final norms of the transformer."""

    @staticmethod
    def forward(ctx, x, r, w, b):
        x, w, b = _f32(x, "x"), _f32(w, "ln.weight"), _f32(b, "ln.bias")
        r = None if r is None else _f32(r, "r")
        M = x.shape[0]
        st = _enter(x)
        s_, stat, y = torch.empty_like(x), torch.empty(M, 2, device=x.device, dtype=torch.float32), torch.empty_like(x)
        check(_L().step_add_layernorm96_fwd(x.data_ptr(), _p(r), w.data_ptr(), b.data_ptr(), M, s_.data_ptr(), stat.data_ptr(),
                                            y.data_ptr(), st), "step_add_layernorm96_fwd")
        launch_counter["kernels"] += 1
        ctx.save_for_backward(s_, stat, w)
        ctx.has_r = r is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        s_, stat, w = ctx.saved_tensors
        dy = _f32(dy, "dy")
        st = _enter(dy)
        dx = torch.empty_like(dy)
        dw, db = torch.empty(96, device=dy.device, dtype=torch.float32), torch.empty(96, device=dy.device, dtype=torch.float32)
        check(_L().step_add_layernorm96_bwd(dy.data_ptr(), s_.data_ptr(), stat.data_ptr(), w.data_ptr(), dy.shape[0], dx.data_ptr(),
                                            dw.data_ptr(), db.data_ptr(), st), "step_add_layernorm96_bwd")
        launch_counter["kernels"] += 1
        return dx, (dx if ctx.has_r else None), dw, db


class Dropout(torch.autograd.Function):
    """Inverted dropout from the counter-based generator; the backward is the same kernel on the gradient."""

    @staticmethod
    def forward(ctx, x, p, seed, site):
        ctx.cfg = (float(p), int(seed) & (2**64 - 1), int(site))
        return Dropout._run(_f32(x, "x"), *ctx.cfg)

    @staticmethod
    def _run(x, p, seed, site):
        st = _enter(x)
        y = torch.empty_like(x)
        check(_L().step_dropout_f32(x.data_ptr(), x.numel(), p, seed, site, y.data_ptr(), st), "step_dropout_f32")
        launch_counter["kernels"] += 1
        return y

    @staticmethod
    def backward(ctx, dy):
        return Dropout._run(_f32(dy, "dy"), *ctx.cfg), None, None, None


def dropout(x: Tensor, p: float, seed: int, site: int) -> Tensor:
    return Dropout.apply(x, p, seed, site) if p > 0.0 else x


def transformer_layer_train(z: Tensor, S: int, P: int, lw: Dict[str, Tensor], drop_p: float, seed: int, site: int,
                            tc_attention: bool = False) -> Tensor:
    """One post-norm nn.TransformerEncoderLayer(96, 4, 384) on tokens z [S*P, 96] with autograd (stage-1 training path;
    the forecasting path uses the fused inference kernels).  tc_attention: attention on tcgen05 (:class:`AttentionTC`,
    P <= 352) instead of the fp32 kernels."""
    qkv = Linear.apply(z, lw["in_proj_w"], lw["in_proj_b"], False)
    attn = AttentionTC if tc_attention else Attention
    o = attn.apply(qkv, S, P, drop_p, (seed + 7919 * site) & (2**63 - 1))
    o = dropout(Linear.apply(o, lw["out_proj_w"], lw["out_proj_b"], False), drop_p, seed, site + 2)
    z1 = AddLayerNorm.apply(z, o, lw["norm1_w"], lw["norm1_b"])
    f = dropout(Linear.apply(z1, lw["lin1_w"], lw["lin1_b"], True), drop_p, seed, site + 3)
    f = dropout(Linear.apply(f, lw["lin2_w"], lw["lin2_b"], False), drop_p, seed, site + 4)
    return AddLayerNorm.apply(z1, f, lw["norm2_w"], lw["norm2_b"])


# --------------------------------------------------------------------------- #
# kNN prior
# --------------------------------------------------------------------------- #
def cosine_gram(x: Tensor) -> Tensor:
    x = _f32(x, "x")
    B, N, D = x.shape
    st = _enter(x)
    norms = torch.empty(B, N, device=x.device, dtype=torch.float32)
    sim = torch.empty(B, N, N, device=x.device, dtype=torch.float32)
    check(_L().step_cosine_gram_f32(x.data_ptr(), B, N, D, norms.data_ptr(), sim.data_ptr(), st), "step_cosine_gram_f32")
    launch_counter["kernels"] += 2
    return sim


def topk_mask(sim: Tensor, k: int) -> Tensor:
    sim = _f32(sim, "sim")
    B, N, _ = sim.shape
    st = _enter(sim)
    adj = torch.empty_like(sim)
    check(_L().step_topk_mask_f32(sim.data_ptr(), B, N, int(k), adj.data_ptr(), st), "step_topk_mask_f32")
    launch_counter["kernels"] += 1
    return adj


def knn_prior(hidden: Tensor, k_total: int) -> Tensor:
    """hidden [B,N,P,d] -> adj_knn [B,N,N] (no gradient: discrete_graph_learning.py:108-110)."""
    B, N = hidden.shape[:2]
    with torch.no_grad():
        return topk_mask(cosine_gram(hidden.reshape(B, N, -1)), k_total)


# --------------------------------------------------------------------------- #
# edge logits + Gumbel sample
# --------------------------------------------------------------------------- #
class EdgeLogits(torch.autograd.Function):
    """(ut [F,N], v [N,F], cat_w [2,F], cat_b [2]) -> (logits [N,N,2], theta [N,N])."""

    @staticmethod
    def forward(ctx, ut, v, cat_w, cat_b):
        ut, v, cat_w, cat_b = _f32(ut, "ut"), _f32(v, "v"), _f32(cat_w, "cat_w"), _f32(cat_b, "cat_b")
        F_, N = ut.shape
        st = _enter(ut)
        logits = torch.empty(N, N, 2, device=ut.device, dtype=torch.float32)
        theta = torch.empty(N, N, device=ut.device, dtype=torch.float32)
        check(_L().step_edge_logits_fwd(ut.data_ptr(), v.data_ptr(), cat_w.data_ptr(), cat_b.data_ptr(), N, F_,
                                        logits.data_ptr(), theta.data_ptr(), st), "step_edge_logits_fwd")
        launch_counter["kernels"] += 1
        ctx.save_for_backward(ut, v, cat_w, theta)
        return logits, theta

    @staticmethod
    def backward(ctx, dlogits, dtheta):
        ut, v, cat_w, theta = ctx.saved_tensors
        F_, N = ut.shape
        dl = torch.zeros(N, N, 2, device=ut.device, dtype=torch.float32) if dlogits is None else dlogits.contiguous().clone()
        if dtheta is not None:
            t = dtheta * theta * (1.0 - theta)       # d softmax_0 / d(l0 - l1)
            dl[..., 0] += t
            dl[..., 1] -= t
        st = _enter(ut)
        dut = torch.empty_like(ut); dv = torch.empty_like(v)
        dcw = torch.empty_like(cat_w); dcb = torch.empty(2, device=ut.device, dtype=torch.float32)
        check(_L().step_edge_logits_bwd(dl.data_ptr(), ut.data_ptr(), v.data_ptr(), cat_w.data_ptr(), N, F_, dut.data_ptr(),
                                        dv.data_ptr(), dcw.data_ptr(), dcb.data_ptr(), st), "step_edge_logits_bwd")
        launch_counter["kernels"] += 2
        return dut, dv, dcw, dcb


class GumbelSample(torch.autograd.Function):
    """logits [N,N,2] -> sampled adjacency [B,N,N] in {0,1} with straight-through gradient."""

    @staticmethod
    def forward(ctx, logits, uniform, B, tau, seed):
        logits = _f32(logits, "logits")
        N = logits.shape[0]
        if uniform is not None:
            uniform = _f32(uniform, "uniform")
            if uniform.numel() != B * N * N * 2:
                raise _lib.StepB200Error("gumbel_sample: uniform must hold B*N*N*2 values")
        st = _enter(logits)
        sampled = torch.empty(B, N, N, device=logits.device, dtype=torch.float32)
        y0 = torch.empty(B, N, N, device=logits.device, dtype=torch.float32)
        check(_L().step_gumbel_sample_fwd(logits.data_ptr(), _p(uniform), B, N, float(tau), int(seed) & (2**64 - 1),
                                          sampled.data_ptr(), y0.data_ptr(), st), "step_gumbel_sample_fwd")
        launch_counter["kernels"] += 1
        ctx.save_for_backward(y0)
        ctx.tau = float(tau)
        return sampled

    @staticmethod
    def backward(ctx, dsampled):
        (y0,) = ctx.saved_tensors
        B, N, _ = y0.shape
        dsampled = _f32(dsampled, "dsampled")
        st = _enter(y0)
        dl = torch.empty(N, N, 2, device=y0.device, dtype=torch.float32)
        check(_L().step_gumbel_sample_bwd(dsampled.data_ptr(), y0.data_ptr(), B, N, ctx.tau, 0, dl.data_ptr(), st),
              "step_gumbel_sample_bwd")
        launch_counter["kernels"] += 1
        return dl, None, None, None, None


# --------------------------------------------------------------------------- #
# Graph WaveNet layer stack
# --------------------------------------------------------------------------- #
_GW_FIELDS = ("filter_w", "filter_b", "gate_w", "gate_b", "skip_w", "skip_b", "mlp_w", "mlp_b", "bn_w", "bn_b")


def _gw_time_extents(n_layers: int):
    t, outs = 13, []
    for i in range(n_layers):
        t -= 1 if i % 2 == 0 else 2
        outs.append(t)
    return outs


class GWNetStack(torch.autograd.Function):
    """x0 [B,13,N,32], P1/P2 [B,N,N], P3 [N,N], per-layer parameters -> (skip [B,N,256], bn_stats [L,4,32]).

    flat parameter order per layer: filter_w, filter_b, gate_w, gate_b, skip_w, skip_b, mlp_w, mlp_b, bn_w, bn_b
    (mlp_w/mlp_b/bn_w/bn_b = None for the last layer, whose gcn output is dead in the reference:
    step/step_arch/graphwavenet/model.py:217-218)."""

    @staticmethod
    def forward(ctx, x0, P1, P2, P3, training, drop_p, seed, bn_eval_stats, n_layers, *flat):
        x0, P1, P2, P3 = _f32(x0, "x0"), _f32(P1, "P1"), _f32(P2, "P2"), _f32(P3, "P3")
        B, T0, N, Cc = x0.shape
        if T0 != 13 or Cc != 32:
            raise _lib.StepB200Error(f"gwnet_stack: x0 must be [B,13,N,32], got {tuple(x0.shape)}")
        assert len(flat) == n_layers * 10
        params = [None if t is None else _f32(t, "gw param") for t in flat]
        st = _enter(x0)
        arr = (GwLayerParams * n_layers)()
        for i in range(n_layers):
            for j, name in enumerate(_GW_FIELDS):
                t = params[i * 10 + j]
                setattr(arr[i], name, None if t is None else t.data_ptr())
        skip = torch.empty(B, N, 256, device=x0.device, dtype=torch.float32)
        if training:
            bn_stats = torch.zeros(n_layers, 4, 32, device=x0.device, dtype=torch.float32)
        else:
            bn_stats = _f32(bn_eval_stats, "bn_eval_stats")
        stash = torch.empty(_L().step_gwnet_stash_floats(B, N, n_layers), device=x0.device, dtype=torch.float32)
        check(_L().step_gwnet_stack_fwd(x0.data_ptr(), P1.data_ptr(), P2.data_ptr(), P3.data_ptr(), arr, n_layers, B, N,
                                        1 if training else 0, float(drop_p), int(seed) & (2**64 - 1), skip.data_ptr(),
                                        bn_stats.data_ptr(), stash.data_ptr(), st), "step_gwnet_stack_fwd")
        n_gcn = sum(1 for i in range(n_layers) if params[i * 10 + 6] is not None)
        launch_counter["kernels"] += n_layers + (n_gcn if training else 0)
        ctx.save_for_backward(x0, P1, P2, P3, bn_stats, stash, *[p for p in params if p is not None])
        ctx.mask = [p is not None for p in params]
        ctx.cfg = (training, float(drop_p) if training else 0.0, int(seed) & (2**64 - 1), n_layers)
        ctx.mark_non_differentiable(bn_stats)
        return skip, bn_stats

    @staticmethod
    def backward(ctx, dskip, _dstats):
        training, drop_p, seed, n_layers = ctx.cfg
        if not training:
            raise _lib.StepB200Error("gwnet_stack: backward is only defined in training mode (batch statistics)")
        saved = list(ctx.saved_tensors)
        x0, P1, P2, P3, bn_stats, stash = saved[:6]
        it = iter(saved[6:])
        params = [next(it) if m else None for m in ctx.mask]
        B, _, N, _ = x0.shape
        dskip = _f32(dskip, "dskip")
        st = _enter(x0)
        P1t, P2t, P3t = P1.transpose(1, 2).contiguous(), P2.transpose(1, 2).contiguous(), P3.t().contiguous()
        arr = (GwLayerParams * n_layers)()
        garr = (GwLayerGrads * n_layers)()
        grads: List[Optional[Tensor]] = []
        for i in range(n_layers):
            for j, name in enumerate(_GW_FIELDS):
                t = params[i * 10 + j]
                setattr(arr[i], name, None if t is None else t.data_ptr())
                g = None if t is None else torch.empty_like(t)
                grads.append(g)
                setattr(garr[i], name, None if g is None else g.data_ptr())
        dx0 = torch.empty_like(x0)
        dP1, dP2, dP3 = torch.empty_like(P1), torch.empty_like(P2), torch.empty_like(P3)
        check(_L().step_gwnet_stack_bwd(dskip.data_ptr(), x0.data_ptr(), P1.data_ptr(), P2.data_ptr(), P3.data_ptr(),
                                        P1t.data_ptr(), P2t.data_ptr(), P3t.data_ptr(), arr, garr, n_layers, B, N,
                                        drop_p, seed, bn_stats.data_ptr(), stash.data_ptr(), dx0.data_ptr(),
                                        dP1.data_ptr(), dP2.data_ptr(), dP3.data_ptr(), st), "step_gwnet_stack_bwd")
        n_gcn = sum(1 for i in range(n_layers) if params[i * 10 + 6] is not None)
        launch_counter["kernels"] += 2 * n_layers + n_gcn + (n_layers - 1)
        return (dx0, dP1, dP2, dP3, None, None, None, None, None, *grads)


# --------------------------------------------------------------------------- #
# general split-bf16 tcgen05 GEMM + the dense layers built on it
# --------------------------------------------------------------------------- #
GE_NONE, GE_RELU, GE_MASK, GE_RELU_ADD_RELU = 0, 1, 2, 3


def gemm(A: Tensor, B: Tensor, transA: bool = False, transB: bool = False, alpha: float = 1.0, bias: Optional[Tensor] = None,
         epilogue: int = GE_NONE, aux: Optional[Tensor] = None, aux_out: Optional[Tensor] = None, out: Optional[Tensor] = None,
         accumulate: bool = False, ksplit: int = 1) -> Tensor:
    """C[M,N] = alpha * opA opB^T (+ bias, epilogue) with fp32-class accuracy on tcgen05 (csrc/tc_gemm.cu).
    A: [M,K] (or [K,M] if transA); B: [N,K] (an nn.Linear weight; or [K,N] if transB)."""
    A, B = _f32(A, "A"), _f32(B, "B")
    M, K = (A.shape[1], A.shape[0]) if transA else A.shape
    N, Kb = (B.shape[1], B.shape[0]) if transB else B.shape
    if K != Kb:
        raise _lib.StepB200Error(f"gemm: inner dimensions differ ({K} vs {Kb})")
    st = _enter(A)
    C_ = torch.empty(M, N, device=A.device, dtype=torch.float32) if out is None else out
    if aux is not None:
        aux = _f32(aux, "aux")
    check(_L().step_gemm_f32(A.data_ptr(), A.shape[1], int(transA), B.data_ptr(), B.shape[1], int(transB), M, N, K, float(alpha),
                             _p(None if bias is None else _f32(bias, "bias")), int(epilogue), _p(aux),
                             0 if aux is None else aux.shape[1], _p(aux_out), int(accumulate), int(ksplit), C_.data_ptr(),
                             C_.shape[1], st), "step_gemm_f32")
    launch_counter["kernels"] += 1
    return C_


def _ksplit(M: int, N: int, K: int) -> int:
    """Split-K factor for weight-gradient GEMMs (tiny M x N, long K): fill ~2 CTAs per SM."""
    tiles = ((M + 127) // 128) * ((N + 127) // 128)
    return max(1, min((K + 255) // 256, 296 // tiles))


def colsum(x: Tensor) -> Tensor:
    x = _f32(x, "x")
    st = _enter(x)
    out = torch.empty(x.shape[1], device=x.device, dtype=torch.float32)
    check(_L().step_colsum_f32(x.data_ptr(), x.shape[0], x.shape[1], x.shape[1], out.data_ptr(), st), "step_colsum_f32")
    launch_counter["kernels"] += 1
    return out


def relu_bwd(dy: Tensor, y: Tensor) -> Tensor:
    dy, y = _f32(dy, "dy"), _f32(y, "y")
    st = _enter(dy)
    dz = torch.empty_like(dy)
    check(_L().step_relu_bwd_f32(dy.data_ptr(), y.data_ptr(), dy.numel(), dz.data_ptr(), st), "step_relu_bwd_f32")
    launch_counter["kernels"] += 1
    return dz


class Linear(torch.autograd.Function):
    """y = act(x W^T + b) on the split-bf16 tcgen05 GEMM, hand-written backward (dx, dW, db).  x [M,K], W [N,K]."""

    @staticmethod
    def forward(ctx, x, w, b, relu):
        y = gemm(x, w, bias=b, epilogue=GE_RELU if relu else GE_NONE)
        ctx.save_for_backward(x, w, y if relu else None)
        ctx.relu, ctx.has_bias = bool(relu), b is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w, y = ctx.saved_tensors
        dz = relu_bwd(dy, y) if ctx.relu else _f32(dy, "dy")
        dx = gemm(dz, w, transB=True) if ctx.needs_input_grad[0] else None
        dw = gemm(dz, x, transA=True, transB=True, ksplit=_ksplit(w.shape[0], w.shape[1], x.shape[0])) if ctx.needs_input_grad[1] else None
        db = colsum(dz) if (ctx.has_bias and ctx.needs_input_grad[2]) else None
        return dx, dw, db, None


class GwEpilogue(torch.autograd.Function):
    """Graph WaveNet epilogue (graphwavenet/model.py:215-220):  out = end_conv_2(relu(end_conv_1(relu(skip + fc_his(h))))),
    fc_his = Linear(96,512)-ReLU-Linear(512,256)-ReLU.  h [M,96] (no gradient: frozen TSFormer states), skip [M,256] ->
    out [M,12].  4 GEMMs forward (the skip add + both ReLUs ride on the second GEMM's epilogue), 7 GEMMs + 5 small
    kernels backward."""

    @staticmethod
    def forward(ctx, h, skip, w1, b1, w2, b2, we1, be1, we2, be2):
        h, skip = _f32(h, "h"), _f32(skip, "skip")
        h1 = gemm(h, w1, bias=b1, epilogue=GE_RELU)
        hs = torch.empty(h.shape[0], w2.shape[0], device=h.device, dtype=torch.float32)
        x2 = gemm(h1, w2, bias=b2, epilogue=GE_RELU_ADD_RELU, aux=skip, aux_out=hs)
        e1 = gemm(x2, we1, bias=be1, epilogue=GE_RELU)
        out = gemm(e1, we2, bias=be2)
        ctx.save_for_backward(h, h1, hs, x2, e1, w1, w2, we1, we2)
        return out

    @staticmethod
    def backward(ctx, dout):
        h, h1, hs, x2, e1, w1, w2, we1, we2 = ctx.saved_tensors
        dout = _f32(dout, "dout")
        M = h.shape[0]
        dwe2 = gemm(dout, e1, transA=True, transB=True, ksplit=_ksplit(we2.shape[0], we2.shape[1], M))
        dbe2 = colsum(dout)
        de1 = gemm(dout, we2, transB=True, epilogue=GE_MASK, aux=e1)
        dwe1 = gemm(de1, x2, transA=True, transB=True, ksplit=_ksplit(we1.shape[0], we1.shape[1], M))
        dbe1 = colsum(de1)
        dx2 = gemm(de1, we1, transB=True, epilogue=GE_MASK, aux=x2)          # = d skip (the add passes it through)
        dz2 = relu_bwd(dx2, hs)
        dw2 = gemm(dz2, h1, transA=True, transB=True, ksplit=_ksplit(w2.shape[0], w2.shape[1], M))
        db2 = colsum(dz2)
        dh1 = gemm(dz2, w2, transB=True, epilogue=GE_MASK, aux=h1)
        dw1 = gemm(dh1, h, transA=True, transB=True, ksplit=_ksplit(w1.shape[0], w1.shape[1], M))
        db1 = colsum(dh1)
        dh = gemm(dh1, w1, transB=True) if ctx.needs_input_grad[0] else None     # STEP: frozen TSFormer, no consumer
        return dh, dx2, dw1, db1, dw2, db2, dwe1, dbe1, dwe2, dbe2


class GwStart(torch.autograd.Function):
    """x0 [B,13,N,32] = start_conv on the left-padded history channels 0:2 (graphwavenet/model.py:145-155)."""

    @staticmethod
    def forward(ctx, history, w, b):
        history, w, b = _f32(history, "history"), _f32(w.reshape(32, 2), "start_conv.weight"), _f32(b, "start_conv.bias")
        B, T, N, Cc = history.shape
        st = _enter(history)
        x0 = torch.empty(B, T + 1, N, 32, device=history.device, dtype=torch.float32)
        check(_L().step_gw_start_fwd(history.data_ptr(), B, T, N, Cc, w.data_ptr(), b.data_ptr(), x0.data_ptr(), st), "step_gw_start_fwd")
        launch_counter["kernels"] += 1
        ctx.save_for_backward(history)
        ctx.wshape = None
        return x0

    @staticmethod
    def backward(ctx, dx0):
        (history,) = ctx.saved_tensors
        B, T, N, Cc = history.shape
        dx0 = _f32(dx0, "dx0")
        st = _enter(history)
        g = torch.empty(96, device=history.device, dtype=torch.float32)
        check(_L().step_gw_start_bwd(history.data_ptr(), B, T, N, Cc, dx0.data_ptr(), g.data_ptr(), st), "step_gw_start_bwd")
        launch_counter["kernels"] += 1
        return None, g[:64].view(32, 2, 1, 1), g[64:]


class GwSupports(torch.autograd.Function):
    """(P1, P2) = (D^-1 (A + I), D'^-1 (A^T + I)) for the sampled graph A [B,N,N] (graphwavenet/model.py:121-130,160)."""

    @staticmethod
    def forward(ctx, adj):
        adj = _f32(adj, "sampled_adj")
        B, N, _ = adj.shape
        st = _enter(adj)
        deg = torch.empty(2, B, N, device=adj.device, dtype=torch.float32)
        P1, P2 = torch.empty_like(adj), torch.empty_like(adj)
        check(_L().step_gw_supports_fwd(adj.data_ptr(), B, N, deg.data_ptr(), P1.data_ptr(), P2.data_ptr(), st), "step_gw_supports_fwd")
        launch_counter["kernels"] += 2
        ctx.save_for_backward(P1, P2, deg)
        return P1, P2

    @staticmethod
    def backward(ctx, dP1, dP2):
        P1, P2, deg = ctx.saved_tensors
        B, N, _ = P1.shape
        dP1, dP2 = _f32(dP1, "dP1"), _f32(dP2, "dP2")
        st = _enter(P1)
        dots = torch.empty(2, B, N, device=P1.device, dtype=torch.float32)
        dadj = torch.empty_like(P1)
        check(_L().step_gw_supports_bwd(dP1.data_ptr(), dP2.data_ptr(), P1.data_ptr(), P2.data_ptr(), deg.data_ptr(), B, N,
                                        dots.data_ptr(), dadj.data_ptr(), st), "step_gw_supports_bwd")
        launch_counter["kernels"] += 2
        return dadj


class GwAdaptive(torch.autograd.Function):
    """P3 [N,N] = softmax(relu(E1 E2), dim=1) (graphwavenet/model.py:165)."""

    @staticmethod
    def forward(ctx, e1, e2):
        e1, e2 = _f32(e1, "nodevec1"), _f32(e2, "nodevec2")
        N, R = e1.shape
        st = _enter(e1)
        P3 = torch.empty(N, N, device=e1.device, dtype=torch.float32)
        check(_L().step_gw_adp_fwd(e1.data_ptr(), e2.data_ptr(), N, R, P3.data_ptr(), st), "step_gw_adp_fwd")
        launch_counter["kernels"] += 1
        ctx.save_for_backward(e1, e2, P3)
        return P3

    @staticmethod
    def backward(ctx, dP3):
        e1, e2, P3 = ctx.saved_tensors
        N, R = e1.shape
        dP3 = _f32(dP3, "dP3")
        st = _enter(e1)
        scratch = torch.empty(N, N, device=e1.device, dtype=torch.float32)
        de1, de2 = torch.empty_like(e1), torch.empty_like(e2)
        check(_L().step_gw_adp_bwd(e1.data_ptr(), e2.data_ptr(), P3.data_ptr(), dP3.data_ptr(), N, R, scratch.data_ptr(),
                                   de1.data_ptr(), de2.data_ptr(), st), "step_gw_adp_bwd")
        launch_counter["kernels"] += 2
        return de1, de2


# --------------------------------------------------------------------------- #
# bf16 tensor-core encoder (tcgen05 / TMEM / TMA bulk)
# --------------------------------------------------------------------------- #
import os as _os

# STEP_B200_TS_FUSED=1: one fused token-block kernel per layer (out-proj + LN1 + FFN + LN2 + next QKV, tc_layer_kernel)
# instead of the four separate token GEMMs.  It is bit-identical and moves 2.7x fewer HBM bytes, but measured 0.84 ms vs
# 0.74 ms per layer at METR-LA (profiles/r02_fused_layer.md): its per-tile chain of 21 dependent MMA -> epilogue hops is
# latency-bound with the two co-resident CTAs the 512 TMEM columns allow, so the separate, deeply pipelined kernels stay
# the default.
TS_FUSED_LAYER = _os.environ.get("STEP_B200_TS_FUSED", "0") == "1"


def tc_pack_weight(w: Tensor) -> Tensor:
    """fp32 [Nout, K] -> bf16 weight image (uint8 tensor of Nout*K*2 bytes)."""
    w = _f32(w, "w")
    Nout, K = w.shape
    st = _enter(w)
    img = torch.empty(Nout * K * 2, device=w.device, dtype=torch.uint8)
    check(_L().step_tc_pack_weight(w.data_ptr(), Nout, K, img.data_ptr(), st), "step_tc_pack_weight")
    launch_counter["kernels"] += 1
    return img


def tc_rows_to_image(x: Tensor) -> Tensor:
    x = _f32(x, "x")
    T, K = x.shape
    st = _enter(x)
    img = torch.empty(((T + 127) // 128) * K * 256, device=x.device, dtype=torch.uint8)
    check(_L().step_tc_rows_to_image(x.data_ptr(), T, K, img.data_ptr(), st), "step_tc_rows_to_image")
    return img


def tc_image_to_rows(img: Tensor, T: int, K: int) -> Tensor:
    st = _enter(img)
    x = torch.empty(T, K, device=img.device, dtype=torch.float32)
    check(_L().step_tc_image_to_rows(img.data_ptr(), T, K, x.data_ptr(), st), "step_tc_image_to_rows")
    return x


def tc_linear(a_img: Tensor, w_img: Tensor, bias: Tensor, T: int, K: int, Nout: int, mode: int, res_img: Optional[Tensor] = None,
              ln_w: Optional[Tensor] = None, ln_b: Optional[Tensor] = None, want_f32: bool = False, drop_p: float = 0.0,
              seed: int = 0):
    """mode 0 -> fp32 [T,Nout]; mode 1 -> ReLU image; mode 2 -> residual+LayerNorm image (and fp32 rows if want_f32).
    drop_p > 0 (modes 1, 2): the epilogue's dropout site is live."""
    st = _enter(a_img)
    MT = (T + 127) // 128
    out_img = out_f32 = None
    if mode == 0 or want_f32:
        out_f32 = torch.empty(T, Nout, device=a_img.device, dtype=torch.float32)
    if mode in (1, 2):
        out_img = torch.empty(MT * Nout * 256, device=a_img.device, dtype=torch.uint8)
    if drop_p > 0.0:
        check(_L().step_tc_linear_drop(a_img.data_ptr(), w_img.data_ptr(), _f32(bias, "bias").data_ptr(), T, K, Nout, mode,
                                       _p(res_img), _p(ln_w), _p(ln_b), _p(out_img), _p(out_f32), float(drop_p),
                                       int(seed) & (2**64 - 1), st), "step_tc_linear_drop")
    else:
        check(_L().step_tc_linear(a_img.data_ptr(), w_img.data_ptr(), _f32(bias, "bias").data_ptr(), T, K, Nout, mode, _p(res_img),
                                  _p(ln_w), _p(ln_b), _p(out_img), _p(out_f32), st), "step_tc_linear")
    launch_counter["kernels"] += 1
    return out_img, out_f32


def tc_qkv_attention(x_img: Tensor, w_img: Tensor, bias: Tensor, S: int, P: int, drop_p: float = 0.0, seed: int = 0,
                     bounded_max: bool = True) -> Tensor:
    """X image [S*P,96] -> O image [S*P,96] (QKV projection + softmax(QK^T)V, both on tcgen05).  ``bounded_max``: let the
    attention kernel replace the row-maximum pass by the Cauchy-Schwarz bound of the operand norms where that is safe."""
    st = _enter(x_img)
    dev = x_img.device
    q = torch.empty(_L().step_tc_attn_image_bytes(S, P, 0), device=dev, dtype=torch.uint8)
    k = torch.empty(_L().step_tc_attn_image_bytes(S, P, 1), device=dev, dtype=torch.uint8)
    v = torch.empty(_L().step_tc_attn_image_bytes(S, P, 1), device=dev, dtype=torch.uint8)
    o = torch.empty(((S * P + 127) // 128) * 96 * 256, device=dev, dtype=torch.uint8)
    bound = None
    if bounded_max:
        bound = torch.empty(_L().step_tc_attn_image_bytes(S, P, 2) // 4, device=dev, dtype=torch.float32)
    check(_L().step_tc_qkv(x_img.data_ptr(), w_img.data_ptr(), _f32(bias, "bias").data_ptr(), S, P, q.data_ptr(), k.data_ptr(),
                           v.data_ptr(), _p(bound), st), "step_tc_qkv")
    check(_L().step_tc_attention(q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), _p(bound), S, P, float(drop_p),
                                 int(seed), st), "step_tc_attention")
    launch_counter["kernels"] += 2
    return o


def ts_pack_layer_images(layers: Sequence[Dict[str, Tensor]], fused: bool = True):
    """Pack the four weight matrices of every encoder layer into bf16 UMMA images (done once: the TSFormer is frozen).
    ``fused``: also the slice buffer of the fused token-block kernel (twelve [96 x 96] slices in program order: out_proj,
    4 x (lin1 rows, lin2 K-columns), then the NEXT layer's q / k / v projections)."""
    out = []
    for i, lw in enumerate(layers):
        im = {"in_proj": tc_pack_weight(lw["in_proj_w"]), "out_proj": tc_pack_weight(lw["out_proj_w"]),
              "lin1": tc_pack_weight(lw["lin1_w"]), "lin2": tc_pack_weight(lw["lin2_w"]), "fused": None}
        if fused:
            parts = [im["out_proj"]]
            for j in range(4):
                parts.append(tc_pack_weight(lw["lin1_w"][96 * j:96 * (j + 1)].contiguous()))
                parts.append(tc_pack_weight(lw["lin2_w"][:, 96 * j:96 * (j + 1)].contiguous()))
            if i + 1 < len(layers):
                nxt = layers[i + 1]["in_proj_w"]
                parts += [tc_pack_weight(nxt[96 * j:96 * (j + 1)].contiguous()) for j in range(3)]
            im["fused"] = torch.cat(parts)
        out.append(im)
    return out


def ts_encoder_forward_bf16(series: Tensor, patch_w: Tensor, patch_b: Tensor, pos: Tensor, layers: Sequence[Dict[str, Tensor]],
                            images, norm_w: Tensor, norm_b: Tensor, drop_p: float = 0.0, seed: int = 0, want_seq_image: bool = False):
    """series [B, P*12, N] view -> hidden [B, N, P, 96] fp32, computed on the tensor cores in bf16.
    want_seq_image: also return the bf16 sequence-major image of the hidden states (Gram operand)."""
    if not series.is_cuda or series.dtype != torch.float32:
        raise _lib.StepB200Error("ts_encoder_forward_bf16: series must be a float32 CUDA tensor")
    B, T, N = series.shape
    if T % 12 != 0:
        raise _lib.StepB200Error(f"ts_encoder_forward_bf16: history length {T} is not a multiple of the patch size 12")
    P = T // 12
    st = _enter(series)
    hidden = torch.empty(B, N, P, 96, device=series.device, dtype=torch.float32)
    ws_bytes = _L().step_ts_encoder_bf16_workspace_bytes(B, N, P)
    ws = torch.empty(ws_bytes, device=series.device, dtype=torch.uint8)
    seq_img = None
    if want_seq_image and (P * 12) % 8 == 0:
        seq_img = torch.empty(_L().step_tc_seq_image_bytes(B, N, P), device=series.device, dtype=torch.uint8)
    arr, keep = ts_layer_struct(layers)
    iarr = (_lib.TsLayerImages * len(layers))()
    for i, im in enumerate(images):
        for name in ("in_proj", "out_proj", "lin1", "lin2"):
            setattr(iarr[i], name, im[name].data_ptr())
        iarr[i].fused = None if (im.get("fused") is None or not TS_FUSED_LAYER) else im["fused"].data_ptr()
    pw, pb, ps = _f32(patch_w.reshape(96, 12), "patch_w"), _f32(patch_b, "patch_b"), _f32(pos, "pos")
    nw, nb = _f32(norm_w, "norm_w"), _f32(norm_b, "norm_b")
    sB, sT, sN = series.stride()
    check(_L().step_ts_encoder_fwd_bf16(series.data_ptr(), sB, sT, sN, B, N, P, pw.data_ptr(), pb.data_ptr(), ps.data_ptr(), arr,
                                        iarr, len(layers), nw.data_ptr(), nb.data_ptr(), hidden.data_ptr(), _p(seq_img),
                                        ws.data_ptr(), ws_bytes, float(drop_p), int(seed) & (2**64 - 1), st),
          "step_ts_encoder_fwd_bf16")
    launch_counter["kernels"] += 2 + len(layers) * 2 if TS_FUSED_LAYER else 1 + len(layers) * 5
    return (hidden, seq_img) if want_seq_image else hidden


def tc_hidden_to_seq_image(hidden: Tensor) -> Tensor:
    """fp32 hidden [B,N,P,96] -> bf16 sequence image (Gram operand)."""
    hidden = _f32(hidden, "hidden")
    B, N, P, _ = hidden.shape
    st = _enter(hidden)
    img = torch.empty(_L().step_tc_seq_image_bytes(B, N, P), device=hidden.device, dtype=torch.uint8)
    check(_L().step_tc_hidden_to_seq_image(hidden.data_ptr(), B, N, P, img.data_ptr(), st), "step_tc_hidden_to_seq_image")
    launch_counter["kernels"] += 1
    return img


def tc_cosine_gram_sharded(seq_img: Tensor, B: int, N: int, P: int, rank: int, world: int, all_reduce_sum) -> Tensor:
    """Node-parallel mode: every rank holds the full bf16 sequence image, computes the raw Gram rows of its share of the
    128-row tiles (tile t belongs to rank t mod world), one small all-reduce (B*N*N fp32) assembles the matrix, then the
    cosine normalisation runs replicated."""
    st = _enter(seq_img)
    gram = torch.zeros(B, N, N, device=seq_img.device, dtype=torch.float32)
    check(_L().step_tc_gram_rows(seq_img.data_ptr(), B, N, P, rank, world, gram.data_ptr(), st), "step_tc_gram_rows")
    all_reduce_sum(gram)
    sim = torch.empty_like(gram)
    check(_L().step_gram_normalize(gram.data_ptr(), B, N, sim.data_ptr(), st), "step_gram_normalize")
    launch_counter["kernels"] += 2
    return sim


def tc_cosine_gram(seq_img: Tensor, B: int, N: int, P: int) -> Tensor:
    """Cosine-similarity Gram matrix [B,N,N] from the encoder's bf16 sequence image (tcgen05)."""
    st = _enter(seq_img)
    scratch = torch.empty(B, N, N, device=seq_img.device, dtype=torch.float32)
    sim = torch.empty(B, N, N, device=seq_img.device, dtype=torch.float32)
    check(_L().step_tc_cosine_gram(seq_img.data_ptr(), B, N, P, scratch.data_ptr(), sim.data_ptr(), st), "step_tc_cosine_gram")
    launch_counter["kernels"] += 2
    return sim


# --------------------------------------------------------------------------- #
# discrete graph learning trunk (conv1 -> BN -> conv2 -> BN)
# --------------------------------------------------------------------------- #
class TrunkConv(torch.autograd.Function):
    """x [N, L0] -> (y2n [N, 16*(L0-18)], bn1_stats [4,8], bn2_stats [4,16]).  Parameters: conv1.w/b, bn1.w/b, conv2.w/b, bn2.w/b."""

    @staticmethod
    def forward(ctx, x, w1, b1, g1, be1, w2, b2, g2, be2, eps, training, eval_stats1, eval_stats2):
        x = _f32(x, "x")
        prm = [_f32(t, "trunk param") for t in (w1, b1, g1, be1, w2, b2, g2, be2)]
        N, L0 = x.shape
        L2 = L0 - 18
        st = _enter(x)
        dev = x.device
        if training:
            s1 = torch.empty(4, 8, device=dev, dtype=torch.float32)
            s2 = torch.empty(4, 16, device=dev, dtype=torch.float32)
        else:
            s1, s2 = _f32(eval_stats1, "eval_stats1"), _f32(eval_stats2, "eval_stats2")
        y2 = torch.empty(N, 16, L2, device=dev, dtype=torch.float32)
        y2n = torch.empty(N, 16, L2, device=dev, dtype=torch.float32)
        scratch = torch.empty(4096, device=dev, dtype=torch.uint8)
        check(_L().step_dgl_conv_fwd(x.data_ptr(), N, L0, *[t.data_ptr() for t in prm], float(eps), 1 if training else 0,
                                     s1.data_ptr(), s2.data_ptr(), y2.data_ptr(), y2n.data_ptr(), scratch.data_ptr(), st),
              "step_dgl_conv_fwd")
        launch_counter["kernels"] += 5 if training else 2
        ctx.save_for_backward(x, y2, s1, s2, *prm)
        ctx.eps, ctx.training = float(eps), bool(training)
        ctx.mark_non_differentiable(s1, s2)
        return y2n.view(N, 16 * L2), s1, s2

    @staticmethod
    def backward(ctx, dy2n, _d1, _d2):
        if not ctx.training:
            raise _lib.StepB200Error("TrunkConv: backward is only defined in training mode (batch statistics)")
        x, y2, s1, s2, w1, b1, g1, be1, w2, b2, g2, be2 = ctx.saved_tensors
        N, L0 = x.shape
        dy2n = _f32(dy2n, "dy2n")
        st = _enter(x)
        dev = x.device
        grads = [torch.empty_like(t) for t in (w1, b1, g1, be1, w2, b2, g2, be2)]
        dy1n = torch.empty(N, 8, L0 - 9, device=dev, dtype=torch.float32)
        scratch = torch.empty(4096, device=dev, dtype=torch.uint8)
        dw1, db1, dg1, dbe1, dw2, db2, dg2, dbe2 = grads
        check(_L().step_dgl_conv_bwd(dy2n.data_ptr(), x.data_ptr(), N, L0, w1.data_ptr(), b1.data_ptr(), g1.data_ptr(),
                                     w2.data_ptr(), g2.data_ptr(), ctx.eps, s1.data_ptr(), s2.data_ptr(), y2.data_ptr(),
                                     dy1n.data_ptr(), dw1.data_ptr(), db1.data_ptr(), dg1.data_ptr(), dbe1.data_ptr(),
                                     dw2.data_ptr(), db2.data_ptr(), dg2.data_ptr(), dbe2.data_ptr(), scratch.data_ptr(), st),
              "step_dgl_conv_bwd")
        launch_counter["kernels"] += 5
        return (None, *grads, None, None, None, None)


class TrunkFc(torch.autograd.Function):
    """feat [N,100] = BatchNorm1d(relu(y2n @ W^T + b)) over the N nodes (discrete_graph_learning.py:134-135): the three
    GEMMs of forward/backward run on tcgen05 with split-bf16 operands (csrc/trunk_fc.cu).  Returns (feat, stats [3,100]).
    ``shard`` = None, or (k_begin, k_end, world, all_reduce_sum): this rank owns the [k_begin, k_end) slice of the K axis
    (z and its gradient are summed over ranks; the weight gradient of the slice comes out already averaged)."""

    @staticmethod
    def forward(ctx, y2n, w, b, gamma, beta, eps, training, eval_stats, shard):
        y2n, w, b, gamma, beta = _f32(y2n, "y2n"), _f32(w, "fc.weight"), _f32(b, "fc.bias"), _f32(gamma, "bn3.weight"), _f32(beta, "bn3.bias")
        N, K = y2n.shape
        if w.shape != (100, K):
            raise _lib.StepB200Error(f"TrunkFc: fc.weight must be [100, {K}], got {tuple(w.shape)}")
        k0, k1 = (0, K) if shard is None else (int(shard[0]), int(shard[1]))
        st = _enter(y2n)
        dev = y2n.device
        splits = _L().step_dgl_fc_splits(N, k0, k1)
        partial = torch.empty(splits, N, 100, device=dev, dtype=torch.float32)
        z = torch.empty(N, 100, device=dev, dtype=torch.float32)
        check(_L().step_dgl_fc_fwd(y2n.data_ptr(), w.data_ptr(), N, K, k0, k1, partial.data_ptr(), z.data_ptr(), st), "step_dgl_fc_fwd")
        if shard is not None and shard[2] > 1:
            shard[3](z)                                   # sum of the ranks' K slices
        stats = torch.empty(3, 100, device=dev, dtype=torch.float32)
        if not training:
            stats[:2].copy_(_f32(eval_stats, "eval_stats")[:2])
        feat = torch.empty(N, 100, device=dev, dtype=torch.float32)
        check(_L().step_dgl_fc_bn_fwd(z.data_ptr(), b.data_ptr(), gamma.data_ptr(), beta.data_ptr(), N, float(eps),
                                      1 if training else 0, stats.data_ptr(), feat.data_ptr(), st), "step_dgl_fc_bn_fwd")
        launch_counter["kernels"] += 3
        ctx.save_for_backward(y2n, w, gamma, z, stats)
        ctx.training, ctx.shard = bool(training), shard
        ctx.mark_non_differentiable(stats)
        return feat, stats

    @staticmethod
    def backward(ctx, dfeat, _dstats):
        if not ctx.training:
            raise _lib.StepB200Error("TrunkFc: backward is only defined in training mode (batch statistics)")
        y2n, w, gamma, z, stats = ctx.saved_tensors
        N, K = y2n.shape
        shard = ctx.shard
        k0, k1 = (0, K) if shard is None else (int(shard[0]), int(shard[1]))
        dfeat = _f32(dfeat, "dfeat")
        st = _enter(y2n)
        dev = y2n.device
        g = torch.empty(N, 100, device=dev, dtype=torch.float32)
        dgamma, dbeta, dbias = (torch.empty(100, device=dev, dtype=torch.float32) for _ in range(3))
        check(_L().step_dgl_fc_bn_bwd(dfeat.data_ptr(), z.data_ptr(), gamma.data_ptr(), stats.data_ptr(), N, g.data_ptr(),
                                      dgamma.data_ptr(), dbeta.data_ptr(), dbias.data_ptr(), st), "step_dgl_fc_bn_bwd")
        scale = 1.0
        if shard is not None and shard[2] > 1:
            shard[3](g)                                   # every rank's loss contributes to this rank's slice
            scale = 1.0 / shard[2]
        full = (k0 == 0 and k1 == K)
        dx = torch.empty_like(y2n) if full else torch.zeros_like(y2n)
        dw = torch.empty_like(w) if full else torch.zeros_like(w)
        check(_L().step_dgl_fc_bwd(g.data_ptr(), y2n.data_ptr(), w.data_ptr(), N, K, k0, k1, scale, dx.data_ptr(), dw.data_ptr(), st),
              "step_dgl_fc_bwd")
        launch_counter["kernels"] += 3
        return dx, dw, dbias, dgamma, dbeta, None, None, None, None


# --------------------------------------------------------------------------- #
# fused STEP loss (masked MAE + graph BCE), value and gradients from one pass
# --------------------------------------------------------------------------- #
class FusedStepLoss(torch.autograd.Function):
    """(pred [..], real [..] unscaled target feature, theta [N,N], adj_knn [B,N,N]) -> scalar loss."""

    @staticmethod
    def forward(ctx, pred, real, theta, adj_knn, coeff, null_val, mean, std):
        import math
        pred, real, theta, adj_knn = _f32(pred, "pred"), _f32(real, "real"), _f32(theta, "theta"), _f32(adj_knn, "adj_knn")
        B, N, _ = adj_knn.shape
        st = _enter(pred)
        dev = pred.device
        loss = torch.empty(1, device=dev, dtype=torch.float32)
        dpred = torch.empty_like(pred)
        dtheta = torch.empty_like(theta)
        scratch = torch.empty(64, device=dev, dtype=torch.uint8)
        nan_mask = 1 if (isinstance(null_val, float) and math.isnan(null_val)) else 0
        check(_L().step_loss_fwd_bwd(pred.data_ptr(), real.data_ptr(), pred.numel(), float(mean), float(std),
                                     0.0 if nan_mask else float(null_val), nan_mask, theta.data_ptr(), adj_knn.data_ptr(), B, N,
                                     float(coeff), loss.data_ptr(), dpred.data_ptr(), dtheta.data_ptr(), scratch.data_ptr(), st),
              "step_loss_fwd_bwd")
        launch_counter["kernels"] += 2
        ctx.save_for_backward(dpred, dtheta)
        return loss[0]

    @staticmethod
    def backward(ctx, g):
        dpred, dtheta = ctx.saved_tensors
        return dpred * g, None, dtheta * g, None, None, None, None, None
