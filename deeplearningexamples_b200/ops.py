"""Autograd functions composing the sm_100a kernels into the operations the reference's modules perform.

Each Function is hand-differentiated: forward and backward call the C ABI (kernels.py) only; torch is
used for memory, streams and the autograd graph.  Activations are bf16 [tokens, features].

Saved-for-backward policy (per encoder layer, T = B*S tokens): qkv [T,3H], ctx [T,H], lse; z1 (pre-LN
sum), mean/rstd; u (pre-GELU) and g = gelu(u) [T,I]; z2.  Dropout masks are never stored: they are
regenerated from (seed, stream id) by the same counter-based RNG in forward and backward.
"""
import torch

from . import _lib as L
from . import kernels as K

bf16 = torch.bfloat16

# -------------------------------------------------------------------------------------------------
# RNG bookkeeping for dropout: one 64-bit seed per forward call site, drawn from a host counter.
# -------------------------------------------------------------------------------------------------
# Under CUDA graphs the host seeds are frozen into the captured launches, so every dropout kernel additionally mixes in a DEVICE
# step counter (one int64 per device, `step_counter`) that BertModel.forward bumps once per training forward pass
# (dle_advance_u64, itself captured): replays draw fresh masks, and the backward of a step sees the value its forward saw.
# -------------------------------------------------------------------------------------------------
_rng = {"base": None, "counter": 0}
_stream_ids = {"next": 1}
_MASK64 = (1 << 64) - 1
_step_counters = {}          # device index -> int64[1] tensor
_err_flags = {}              # device index -> int32[1] tensor (out-of-range ids seen by the gather kernels)


def manual_seed(seed):
    """Reset the dropout RNG: base seed, per-call counter, the device step counters and the call-site stream-id allocator
    (so that a model built and run after manual_seed(s) reproduces its masks exactly)."""
    _rng["base"] = int(seed) & _MASK64
    _rng["counter"] = 0
    _stream_ids["next"] = 1
    for t in _step_counters.values():
        t.zero_()


def step_counter(device):
    """The device-resident dropout step counter of `device` (created on first use)."""
    idx = torch.device(device).index
    if idx is None:
        idx = torch.cuda.current_device()
    t = _step_counters.get(idx)
    if t is None:
        t = torch.zeros(1, dtype=torch.int64, device=torch.device("cuda", idx))
        _step_counters[idx] = t
    return t


def advance_step(device):
    """Bump the device step counter (once per training forward pass; graph-capturable)."""
    K.advance_u64(step_counter(device), 1)


def err_flag(device):
    """Persistent device flag set by the embedding / row-gather kernels when they meet an out-of-range id (the kernels clamp and
    continue; the reference's nn.Embedding would device-assert).  Read it with check_device_errors() at points that already sync."""
    idx = torch.device(device).index
    if idx is None:
        idx = torch.cuda.current_device()
    t = _err_flags.get(idx)
    if t is None:
        t = torch.zeros(1, dtype=torch.int32, device=torch.device("cuda", idx))
        _err_flags[idx] = t
    return t


def check_device_errors():
    """Host sync: raise if any kernel reported an out-of-range token / type / row index since the last check."""
    for idx, t in _err_flags.items():
        if int(t.item()) != 0:
            t.zero_()
            raise L.DleError(f"cuda:{idx}: an embedding or row-gather kernel saw an out-of-range index (ids were clamped to row 0)")


def next_seed():
    if _rng["base"] is None:
        _rng["base"] = torch.initial_seed() & _MASK64
    _rng["counter"] += 1
    return (_rng["base"] * 0x9E3779B97F4A7C15 + _rng["counter"] * 0xD1B54A32D192ED03) & _MASK64


def new_stream_id():
    """Distinct RNG stream per dropout call site (module instance)."""
    _stream_ids["next"] += 1
    return _stream_ids["next"]


# -------------------------------------------------------------------------------------------------
# bf16 views of parameters (fp32-parameter / autocast-style use keeps a cached bf16 copy)
# -------------------------------------------------------------------------------------------------
_w16_cache = {}
weight_epoch = {"n": 0}          # bumped by FusedLAMBAMP.step (in-place updates through raw pointers)


def w16(p, key=None):
    """bf16 tensor holding parameter p's values (p itself when it already is bf16).  `key`: the parameter whose
    version counter governs the cache when p is a derived view (packed q|k|v block)."""
    if p is None:
        return None
    t = p.detach()
    if t.dtype == bf16:
        return t
    if t.dtype != torch.float32:
        raise L.DleError(f"parameters must be bf16 or fp32, got {t.dtype}")
    owner = p if key is None else key
    key = (id(owner), tuple(t.shape))
    ent = _w16_cache.get(key)
    sig = (t.data_ptr(), owner._version, weight_epoch["n"])
    if ent is None or ent[0] != sig:
        buf = ent[1] if (ent is not None and ent[1].shape == t.shape) else torch.empty(t.shape, device=t.device, dtype=bf16)
        K.cast_f32_to_bf16(t.contiguous(), buf)
        ent = (sig, buf)
        _w16_cache[key] = ent
    return ent[1]


def _to_param_dtype(g, p):
    return g if g.dtype == p.dtype else g.to(p.dtype)


_sm_cache = {}


def _sm_count():
    dev = torch.cuda.current_device()
    n = _sm_cache.get(dev)
    if n is None:
        n = _sm_cache[dev] = torch.cuda.get_device_properties(dev).multi_processor_count
    return n


def _split_k(tiles, slots, max_splits):
    """Split-K factor for a GEMM with `tiles` output tiles on a persistent grid of `slots` workers: the smallest factor whose work units fill
    whole waves (units / (ceil(units / slots) * slots) >= 0.93), else the best found.  Round 1 used ceil(slots / tiles), which left the
    QKV weight gradient (1.3 waves) at 1000 TFLOP/s and the attention-output one (1.08 waves) at 750."""
    best, best_eff = 1, 0.0
    for s_ in range(1, max(1, max_splits) + 1):
        units = tiles * s_
        eff = units / (-(-units // slots) * slots)
        if eff >= 0.93:
            return s_
        if eff > best_eff + 1e-9:
            best, best_eff = s_, eff
    return best


def wgrad(dy, x, out_dtype):
    """dW[N_out, K_in] = dy[T, N_out]^T @ x[T, K_in]; both operands read MN-major where they lie.
    Few output tiles => split-K over tokens with fp32 red.global.add; otherwise direct store.
    The GEMM kernel runs each 256 x 256 output tile on a pair of SMs, so work is counted in pair tiles over SMs / 2 pair slots."""
    T, n_out = dy.shape
    k_in = x.shape[1]
    tiles = ((n_out + 255) // 256) * ((k_in + 255) // 256)
    slots = _sm_count() // 2
    if tiles >= slots * 3 // 4:
        if out_dtype == torch.float32:
            return K.gemm(dy, x, a_layout=L.LAYOUT_MN, b_layout=L.LAYOUT_MN, epilogue=L.EPI_F32)
        return K.gemm(dy, x, a_layout=L.LAYOUT_MN, b_layout=L.LAYOUT_MN, epilogue=L.EPI_BIAS)
    splits = _split_k(tiles, slots, min(16, (T + 511) // 512))
    acc = K.gemm(dy, x, a_layout=L.LAYOUT_MN, b_layout=L.LAYOUT_MN, epilogue=L.EPI_ATOMIC_F32, splits=splits)
    return acc if out_dtype == torch.float32 else K.cast_f32_to_bf16(acc)


def _bias_grad(dy, p):
    return None if p is None else _to_param_dtype(K.colsum(dy), p)


# -------------------------------------------------------------------------------------------------
# y = act(x W^T + b)          act in {none, gelu_tanh, tanh}
# replaces nn.Linear / LinearActivation (modeling.py:130-160)
# -------------------------------------------------------------------------------------------------
class LinearFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, act):
        w, b = w16(weight), w16(bias)
        ctx.act = act
        if act == "gelu":
            y, u = K.gemm(x, w, bias=b, epilogue=L.EPI_BIAS_GELU)
            ctx.save_for_backward(x, weight, bias, u)
        elif act == "tanh":
            y = K.gemm(x, w, bias=b, epilogue=L.EPI_BIAS_TANH)
            ctx.save_for_backward(x, weight, bias, y)
        else:
            y = K.gemm(x, w, bias=b, epilogue=L.EPI_BIAS)
            ctx.save_for_backward(x, weight, bias, None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, weight, bias, aux = ctx.saved_tensors
        dy = dy.contiguous()
        if ctx.act == "gelu":
            dy = K.bias_gelu_bwd(dy, aux)
        elif ctx.act == "tanh":
            dy = (dy.float() * (1.0 - aux.float() ** 2)).to(bf16)      # [B,H] pooler only
        dx = K.gemm(dy, w16(weight), b_layout=L.LAYOUT_MN) if ctx.needs_input_grad[0] else None
        dw = wgrad(dy, x, weight.dtype) if ctx.needs_input_grad[1] else None
        db = _bias_grad(dy, bias) if (bias is not None and ctx.needs_input_grad[2]) else None
        return dx, dw, db, None


# -------------------------------------------------------------------------------------------------
# y = LayerNorm(dropout(x W^T + b) + residual)
# replaces BertSelfOutput.forward / BertOutput.forward (modeling.py:394-398, 430-434)
# -------------------------------------------------------------------------------------------------
class DenseDropoutAddLNFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, residual, weight, bias, gamma, beta, p_drop, eps, stream_id):
        seed = next_seed() if p_drop > 0.0 else 0
        z = K.gemm(x, w16(weight), bias=w16(bias), aux=residual, epilogue=L.EPI_BIAS_DROPOUT_RESIDUAL,
                   dropout_p=p_drop, seed=seed, dropout_stream=stream_id, seed_dev=step_counter(x.device))
        y, _, mean, rstd = K.add_ln_fwd(z, w16(gamma), w16(beta), eps=eps)
        ctx.save_for_backward(x, weight, bias, gamma, beta, z, mean, rstd)
        ctx.p_drop, ctx.seed, ctx.stream_id = p_drop, seed, stream_id
        return y

    @staticmethod
    def backward(ctx, dy):
        x, weight, bias, gamma, beta, z, mean, rstd = ctx.saved_tensors
        dz, dh, dgamma, dbeta, dbias = K.add_ln_bwd(dy.contiguous(), z, mean, rstd, w16(gamma), dropout_p=ctx.p_drop,
                                                    seed=ctx.seed, dropout_stream=ctx.stream_id, seed_dev=step_counter(z.device))
        dx = K.gemm(dh, w16(weight), b_layout=L.LAYOUT_MN)
        dw = wgrad(dh, x, weight.dtype)
        return (dx, dz, dw, _to_param_dtype(dbias, bias), _to_param_dtype(dgamma, gamma), _to_param_dtype(dbeta, beta),
                None, None, None)


# -------------------------------------------------------------------------------------------------
# packed QKV projection + fused attention
# replaces BertSelfAttention.forward (modeling.py:340-384)
# -------------------------------------------------------------------------------------------------
class SelfAttentionFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, wq, wk, wv, bq, bk, bv, w_packed, b_packed, mask, B, S, A, p_drop, stream_id, seq_first):
        """x [T,H]; wq/wk/wv, bq/bk/bv: the three nn.Linear parameters (autograd leaves) whose storage is one
        packed block; w_packed [3H,H] / b_packed [3H]: views over that block; mask fp32 [B,S] additive or None."""
        seed = next_seed() if p_drop > 0.0 else 0
        w, b = w16(w_packed, key=wq), w16(b_packed, key=bq)
        qkv = K.gemm(x, w, bias=b)
        out, lse = K.attn_fwd(qkv, mask, B, S, A, dropout_p=p_drop, seed=seed, dropout_stream=stream_id, seq_first=seq_first,
                              seed_dev=step_counter(x.device))
        ctx.save_for_backward(x, w_packed, mask, qkv, out, lse)
        ctx.cfg = (B, S, A, p_drop, seed, stream_id, seq_first)
        ctx.params = (wq, bq)
        return out

    @staticmethod
    def backward(ctx, dout):
        x, w_packed, mask, qkv, out, lse = ctx.saved_tensors
        B, S, A, p_drop, seed, stream_id, seq_first = ctx.cfg
        wq, bq = ctx.params
        dqkv = K.attn_bwd(qkv, mask, out, dout.contiguous(), lse, B, S, A, dropout_p=p_drop, seed=seed,
                          dropout_stream=stream_id, seq_first=seq_first, seed_dev=step_counter(x.device))
        dx = K.gemm(dqkv, w16(w_packed, key=wq), b_layout=L.LAYOUT_MN)
        dw = wgrad(dqkv, x, wq.dtype)                       # [3H, H]
        db = _to_param_dtype(K.colsum(dqkv), bq)            # [3H]
        H = dw.shape[1]
        return (dx, dw[0:H], dw[H:2 * H], dw[2 * H:3 * H], db[0:H], db[H:2 * H], db[2 * H:3 * H],
                None, None, None, None, None, None, None, None, None)


# -------------------------------------------------------------------------------------------------
# whole encoder layer, hand-differentiated end to end (the default path of modeling.BertLayer)
#   replaces BertLayer.forward (modeling.py:453-462) = BertAttention :407-410 + BertIntermediate :418-420 + BertOutput :430-434
# Compared with composing the per-module Functions above, backward folds two more pointwise passes into GEMM
# epilogues: gelu'(u) into the FFN2 dgrad (DLE_EPI_DGELU) and the residual-branch gradient adds into the FFN1 and
# QKV dgrads (DLE_EPI_ADD), and hands autograd one node per layer instead of five.
# -------------------------------------------------------------------------------------------------
class BertLayerFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, mask, wq, wk, wv, bq, bk, bv, wo, bo, g1, be1, w1, b1, w2, b2, g2, be2, w_qkv, b_qkv, cfg):
        B, S, A, p_attn, p_hid, eps, sid_attn, sid_h1, sid_h2, seq_first = cfg
        seed_a = next_seed() if p_attn > 0.0 else 0
        seed_1 = next_seed() if p_hid > 0.0 else 0
        seed_2 = next_seed() if p_hid > 0.0 else 0
        sdev = step_counter(x.device)
        qkv = K.gemm(x, w16(w_qkv, key=wq), bias=w16(b_qkv, key=bq))
        att, lse = K.attn_fwd(qkv, mask, B, S, A, dropout_p=p_attn, seed=seed_a, dropout_stream=sid_attn, seq_first=seq_first, seed_dev=sdev)
        z1 = K.gemm(att, w16(wo), bias=w16(bo), aux=x, epilogue=L.EPI_BIAS_DROPOUT_RESIDUAL, dropout_p=p_hid, seed=seed_1,
                    dropout_stream=sid_h1, seed_dev=sdev)
        y1, _, mean1, rstd1 = K.add_ln_fwd(z1, w16(g1), w16(be1), eps=eps)
        g, u = K.gemm(y1, w16(w1), bias=w16(b1), epilogue=L.EPI_BIAS_GELU)
        z2 = K.gemm(g, w16(w2), bias=w16(b2), aux=y1, epilogue=L.EPI_BIAS_DROPOUT_RESIDUAL, dropout_p=p_hid, seed=seed_2,
                    dropout_stream=sid_h2, seed_dev=sdev)
        y2, _, mean2, rstd2 = K.add_ln_fwd(z2, w16(g2), w16(be2), eps=eps)
        ctx.save_for_backward(x, mask, qkv, att, lse, z1, mean1, rstd1, y1, u, g, z2, mean2, rstd2, w_qkv)
        ctx.params = (wq, bq, wo, bo, g1, be1, w1, b1, w2, b2, g2, be2)
        ctx.cfg = cfg
        ctx.seeds = (seed_a, seed_1, seed_2)
        return y2

    @staticmethod
    def backward(ctx, dy2):
        x, mask, qkv, att, lse, z1, mean1, rstd1, y1, u, g, z2, mean2, rstd2, w_qkv = ctx.saved_tensors
        wq, bq, wo, bo, g1, be1, w1, b1, w2, b2, g2, be2 = ctx.params
        B, S, A, p_attn, p_hid, eps, sid_attn, sid_h1, sid_h2, seq_first = ctx.cfg
        seed_a, seed_1, seed_2 = ctx.seeds
        H_ = x.shape[1]
        sdev = step_counter(x.device)
        # bias gradients of FFN1 (4H) and q|k|v (3H) are column sums of tensors produced below: the producing kernels accumulate
        # them (warp transpose-reduce + red.add) instead of a separate pass re-reading du / dqkv from HBM
        bias_acc = torch.zeros(w1.shape[0] + 3 * H_, device=x.device, dtype=torch.float32)
        db1_acc, dbqkv_acc = bias_acc[:w1.shape[0]], bias_acc[w1.shape[0]:]
        # ---- BertOutput
        dz2, dh2, dg2, dbe2, db2 = K.add_ln_bwd(dy2.contiguous(), z2, mean2, rstd2, w16(g2), dropout_p=p_hid, seed=seed_2,
                                                dropout_stream=sid_h2, out_dtype=g2.dtype, seed_dev=sdev)
        du = K.gemm(dh2, w16(w2), b_layout=L.LAYOUT_MN, epilogue=L.EPI_DGELU, aux=u, colsum_out=db1_acc)   # dgrad * gelu'(u)
        dw2 = wgrad(dh2, g, w2.dtype)
        # ---- BertIntermediate (+ residual branch of BertOutput folded into the epilogue)
        dy1 = K.gemm(du, w16(w1), b_layout=L.LAYOUT_MN, epilogue=L.EPI_ADD, aux=dz2)
        dw1 = wgrad(du, y1, w1.dtype)
        # ---- BertSelfOutput
        dz1, dh1, dg1, dbe1, dbo = K.add_ln_bwd(dy1, z1, mean1, rstd1, w16(g1), dropout_p=p_hid, seed=seed_1, dropout_stream=sid_h1,
                                                out_dtype=g1.dtype, seed_dev=sdev)
        datt = K.gemm(dh1, w16(wo), b_layout=L.LAYOUT_MN)
        dwo = wgrad(dh1, att, wo.dtype)
        # ---- BertSelfAttention (+ residual branch of BertSelfOutput folded into the QKV dgrad epilogue)
        dqkv = K.attn_bwd(qkv, mask, att, datt, lse, B, S, A, dropout_p=p_attn, seed=seed_a, dropout_stream=sid_attn, seq_first=seq_first,
                          dbias=dbqkv_acc, seed_dev=sdev)
        dx = K.gemm(dqkv, w16(w_qkv, key=wq), b_layout=L.LAYOUT_MN, epilogue=L.EPI_ADD, aux=dz1)
        dwqkv = wgrad(dqkv, x, wq.dtype)
        bias_g = bias_acc if b1.dtype == torch.float32 else bias_acc.to(b1.dtype)
        db1, dbqkv = bias_g[:w1.shape[0]], bias_g[w1.shape[0]:]
        H = dwqkv.shape[1]
        c = _to_param_dtype
        return (dx, None, dwqkv[0:H], dwqkv[H:2 * H], dwqkv[2 * H:3 * H], dbqkv[0:H], dbqkv[H:2 * H], dbqkv[2 * H:3 * H],
                dwo, c(dbo, bo), c(dg1, g1), c(dbe1, be1), dw1, db1, dw2, c(db2, b2), c(dg2, g2), c(dbe2, be2), None, None, None)


# -------------------------------------------------------------------------------------------------
# embeddings: dropout(LayerNorm(word[ids] + pos[arange(S)] + type[tt]))
# replaces BertEmbeddings.forward (modeling.py:285-301)
# -------------------------------------------------------------------------------------------------
class EmbeddingLNFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, input_ids, token_type_ids, word, pos, typ, gamma, beta, p_drop, eps, stream_id):
        seed = next_seed() if p_drop > 0.0 else 0
        ids, tts = input_ids.contiguous(), token_type_ids.contiguous()
        y, z, mean, rstd = K.embed_ln_fwd(ids, tts, w16(word), w16(pos), w16(typ), w16(gamma), w16(beta), eps=eps,
                                          dropout_p=p_drop, seed=seed, dropout_stream=stream_id, err_flag=err_flag(word.device),
                                          seed_dev=step_counter(word.device))
        ctx.save_for_backward(ids, tts, word, pos, typ, gamma, beta, z, mean, rstd)
        ctx.cfg = (p_drop, seed, stream_id)
        return y

    @staticmethod
    def backward(ctx, dy):
        ids, tts, word, pos, typ, gamma, beta, z, mean, rstd = ctx.saved_tensors
        p_drop, seed, stream_id = ctx.cfg
        dword, dpos, dtyp, dgamma, dbeta = K.embed_ln_bwd(dy.contiguous(), z, mean, rstd, w16(gamma), ids, tts,
                                                          word.shape[0], pos.shape[0], typ.shape[0], dropout_p=p_drop,
                                                          seed=seed, dropout_stream=stream_id, seed_dev=step_counter(dy.device))
        cast = lambda g, p: g if p.dtype == torch.float32 else K.cast_f32_to_bf16(g)
        return (None, None, cast(dword, word), cast(dpos, pos), cast(dtyp, typ), _to_param_dtype(dgamma, gamma),
                _to_param_dtype(dbeta, beta), None, None, None)


# -------------------------------------------------------------------------------------------------
# plain LayerNorm (MLM transform, modeling.py:534) and masked-row gather (modeling.py:590)
# -------------------------------------------------------------------------------------------------
class LayerNormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, gamma, beta, eps):
        y, _, mean, rstd = K.add_ln_fwd(x, w16(gamma), w16(beta), eps=eps)
        ctx.save_for_backward(x, gamma, beta, mean, rstd)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, gamma, beta, mean, rstd = ctx.saved_tensors
        dz, _, dgamma, dbeta = K.add_ln_bwd(dy.contiguous(), x, mean, rstd, w16(gamma), want_dbias=False)
        return dz, _to_param_dtype(dgamma, gamma), _to_param_dtype(dbeta, beta), None


class GatherRowsFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, idx):
        ctx.save_for_backward(idx)
        ctx.n_rows = x.shape[0]
        return K.gather_rows(x, idx, err_flag=err_flag(x.device))

    @staticmethod
    def backward(ctx, dy):
        (idx,) = ctx.saved_tensors
        return K.scatter_rows(dy.contiguous(), idx, ctx.n_rows), None


# -------------------------------------------------------------------------------------------------
# mean cross-entropy over the vocabulary on bf16 logits, fp32 arithmetic, no fp32 copy of the logits
# replaces CrossEntropyLoss(ignore_index=-1) on the MLM scores (run_pretraining.py:85-95)
# -------------------------------------------------------------------------------------------------
class SoftmaxCrossEntropyFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, labels, ignore_index):
        x = logits if logits.stride(-1) == 1 else logits.contiguous()
        lse, loss_rows = K.softmax_ce_fwd(x, labels, ignore_index, err_flag=err_flag(x.device))
        count = (labels != ignore_index).sum().to(torch.float32)
        ctx.save_for_backward(x, labels, lse, count)
        ctx.ignore_index = ignore_index
        return loss_rows.sum() / count

    @staticmethod
    def backward(ctx, g):
        x, labels, lse, count = ctx.saved_tensors
        scale = (g.to(torch.float32) / count).reshape(1).contiguous()
        return K.softmax_ce_bwd(x, labels, lse, scale, ctx.ignore_index), None, None
