"""Raw (non-autograd) Python wrappers over the C ABI. Tensors are torch CUDA tensors used purely as device buffers;
every call goes to libspeecht5_b200.so on the current CUDA stream. No fallbacks."""
import ctypes as C

import torch

from . import _lib
from ._lib import ACT_IDS, BF16, F32, AttnArgs, GemmArgs


LAUNCHES = 0      # kernels of libspeecht5_b200.so launched through this module (bench.py reports it)
GEMM_RECORD = None  # when a list: every st5_gemm_bf16 argument block is appended (bench.py roofline replay)


def _count(n):
    global LAUNCHES
    LAUNCHES += n


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def dtype_id(t):
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise TypeError(f"unsupported activation dtype {t.dtype}")


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("speecht5_b200 kernels need CUDA tensors (no CPU fallback)")


def gemm(a, b, out, *, M, N, K, a_mn=False, b_mn=False, a_ld=None, b_ld=None, c_ld=None, nb1=1, nb2=1,
         a_bs=(0, 0), b_bs=(0, 0), c_bs=(0, 0), bias=None, bias2=None, bias2_rows=0, residual=None, c_pre=None,
         act=None, alpha=1.0, accumulate=False, drop_p=0.0, seed=0, offset=0, actgrad_pre=None, actgrad_act=None):
    """out[z][m][n] = epi(alpha * sum_k A[z][m][k] B[z][n][k]); see st5_gemm_bf16 in include/speecht5_b200.h."""
    _require_cuda(a, b, out)
    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16
    g = GemmArgs()
    g.M, g.N, g.K, g.nb1, g.nb2 = M, N, K, nb1, nb2
    g.a_mn, g.b_mn = int(a_mn), int(b_mn)
    g.c_fp32 = 1 if out.dtype == torch.float32 else 0
    g.act = ACT_IDS[act]
    g.accumulate = int(accumulate)
    g.bias2_rows = bias2_rows
    g.a, g.a_ld, g.a_bs1, g.a_bs2 = a.data_ptr(), (a_ld if a_ld is not None else (M if a_mn else K)), a_bs[0], a_bs[1]
    g.b, g.b_ld, g.b_bs1, g.b_bs2 = b.data_ptr(), (b_ld if b_ld is not None else (N if b_mn else K)), b_bs[0], b_bs[1]
    g.c, g.c_ld, g.c_bs1, g.c_bs2 = out.data_ptr(), (c_ld if c_ld is not None else N), c_bs[0], c_bs[1]
    g.c_pre = None if c_pre is None else c_pre.data_ptr()
    g.bias = None if bias is None else bias.data_ptr()
    g.bias2 = None if bias2 is None else bias2.data_ptr()
    g.residual = None if residual is None else residual.data_ptr()
    if bias is not None:
        assert bias.dtype == torch.float32
    if bias2 is not None:
        assert bias2.dtype == torch.float32
    if residual is not None:
        assert residual.dtype == out.dtype
    if c_pre is not None:
        assert c_pre.dtype == out.dtype
    g.alpha = alpha
    g.drop_p, g.drop_seed, g.drop_offset = drop_p, seed, offset
    if actgrad_pre is not None:
        assert actgrad_pre.dtype == out.dtype
        g.actgrad_pre, g.actgrad_act = actgrad_pre.data_ptr(), ACT_IDS[actgrad_act]
    lib = _lib.load()
    _lib.check(lib.st5_gemm_bf16(C.byref(g), _stream()), "st5_gemm_bf16")
    _count(1)
    if GEMM_RECORD is not None:
        g._keep = (a, b, out, c_pre, bias, bias2, residual, actgrad_pre)  # keep the operands alive for the replay
        GEMM_RECORD.append(g)
    return out


def gemm_replay(records):
    """Re-issue recorded GEMM launches back to back on the current stream (timing only)."""
    lib = _lib.load()
    st = _stream()
    for g in records:
        _lib.check(lib.st5_gemm_bf16(C.byref(g), st), "st5_gemm_bf16")


def cast_bf16(src, hi, lo=None):
    """2-D strided fp32 -> bf16 (hi) and optional bf16 residual (lo)."""
    _require_cuda(src, hi)
    assert src.dtype == torch.float32 and src.dim() == 2 and src.stride(1) == 1
    rows, cols = src.shape
    assert hi.stride(1) == 1 and (lo is None or lo.stride() == hi.stride())
    lib = _lib.load()
    _lib.check(lib.st5_cast_bf16(_ptr(src), src.stride(0), _ptr(hi), _ptr(lo), hi.stride(0), rows, cols, _stream()),
               "st5_cast_bf16")
    _count(1)


def posenc_fwd(tokens, emb, x, pe, alpha, y, drop_p=0.0, seed=0, offset=0):
    B, T, Cc = y.shape
    lib = _lib.load()
    _lib.check(lib.st5_posenc_fwd(_ptr(tokens), _ptr(emb), _ptr(x), _ptr(pe), _ptr(alpha), _ptr(y), dtype_id(y), B, T,
                                  Cc, drop_p, seed, offset, _stream()), "st5_posenc_fwd")
    _count(1)


def posenc_bwd(dy, tokens, padding_idx, pe, dx, demb, dalpha, drop_p=0.0, seed=0, offset=0):
    B, T, Cc = dy.shape
    lib = _lib.load()
    _lib.check(lib.st5_posenc_bwd(_ptr(dy), _ptr(tokens), padding_idx, _ptr(pe), _ptr(dx), _ptr(demb), _ptr(dalpha),
                                  dtype_id(dy), B, T, Cc, drop_p, seed, offset, _stream()), "st5_posenc_bwd")
    _count(1)


def ln_fwd(x, residual, gamma, beta, y, s_out, mean, rstd, eps, drop_p=0.0, seed=0, offset=0, residual_f32=None,
           y_f32=None):
    Cc = x.shape[-1]
    rows = x.numel() // Cc
    lib = _lib.load()
    if residual_f32 is not None or y_f32 is not None:
        assert (residual_f32 is None or residual_f32.dtype == torch.float32) and (y_f32 is None or y_f32.dtype == torch.float32)
        _lib.check(lib.st5_ln_fwd_stream(_ptr(x), _ptr(residual), _ptr(residual_f32), _ptr(gamma), _ptr(beta), _ptr(y),
                                         _ptr(y_f32), _ptr(s_out), _ptr(mean), _ptr(rstd), dtype_id(x), rows, Cc, eps,
                                         drop_p, seed, offset, _stream()), "st5_ln_fwd_stream")
    else:
        _lib.check(lib.st5_ln_fwd(_ptr(x), _ptr(residual), _ptr(gamma), _ptr(beta), _ptr(y), _ptr(s_out), _ptr(mean),
                                  _ptr(rstd), dtype_id(x), rows, Cc, eps, drop_p, seed, offset, _stream()), "st5_ln_fwd")
    _count(1)


def ln_bwd(dy, s, mean, rstd, gamma, ds, dx, dgamma, dbeta, drop_p=0.0, seed=0, offset=0, dxsum=None):
    """dxsum (optional, fp32 [C], accumulated): column sums of dx = the bias gradient of the projection that fed x."""
    Cc = dy.shape[-1]
    rows = dy.numel() // Cc
    lib = _lib.load()
    if dxsum is not None:
        assert dxsum.dtype == torch.float32 and dxsum.numel() >= Cc and dxsum.is_contiguous()
    _lib.check(lib.st5_ln_bwd(_ptr(dy), _ptr(s), _ptr(mean), _ptr(rstd), _ptr(gamma), _ptr(ds), _ptr(dx),
                              _ptr(dgamma), _ptr(dbeta), _ptr(dxsum), dtype_id(dy), rows, Cc, drop_p, seed, offset,
                              _stream()), "st5_ln_bwd")
    fused = (dgamma is not None or dbeta is not None or dxsum is not None) and (rows >= 64 or dxsum is not None)
    _count(1 if fused or (dgamma is None and dbeta is None) else 2)


def lrelu_pad(x, out, d, ph, pad, slope):
    """st5_lrelu_pad: out [B, n_in, C] <- leaky_relu(x [B, T, C]) at frames ph + d*m - pad (zeros outside [0, T))."""
    _require_cuda(x, out)
    assert x.dtype == torch.bfloat16 and out.dtype == torch.bfloat16 and x.is_contiguous() and out.is_contiguous()
    B, T, Cc = x.shape
    assert out.shape[0] == B and out.shape[2] == Cc
    _lib.check(_lib.load().st5_lrelu_pad(_ptr(x), _ptr(out), B, T, Cc, out.shape[1], int(d), int(ph), int(pad),
                                         float(slope), _stream()), "st5_lrelu_pad")
    _count(1)


def dropout(x, y, drop_p, seed, offset):
    lib = _lib.load()
    _lib.check(lib.st5_dropout(_ptr(x), _ptr(y), dtype_id(x), x.numel(), drop_p, seed, offset, _stream()),
               "st5_dropout")
    _count(1)


def act_bwd(dy, pre, dpre, act, drop_p=0.0, seed=0, offset=0):
    lib = _lib.load()
    _lib.check(lib.st5_act_bwd(_ptr(dy), _ptr(pre), _ptr(dpre), dtype_id(dy), ACT_IDS[act], dy.numel(), drop_p, seed,
                               offset, _stream()), "st5_act_bwd")
    _count(1)


def colsum(x2d, out, group_rows=0, accumulate=False, ld=None):
    rows, cols = x2d.shape
    lib = _lib.load()
    _lib.check(lib.st5_colsum(_ptr(x2d), ld if ld is not None else x2d.stride(0), _ptr(out), dtype_id(x2d), rows, cols,
                              group_rows, int(accumulate), _stream()), "st5_colsum")
    _count(1)


def attn_args(**kw):
    a = AttnArgs()
    for k, v in kw.items():
        if isinstance(v, torch.Tensor):
            v = v.data_ptr()
        setattr(a, k, v)
    return a


def attn_fwd(a):
    lib = _lib.load()
    _lib.check(lib.st5_attn_fwd(C.byref(a), _stream()), "st5_attn_fwd")
    _count(1)


def attn_bwd(a):
    lib = _lib.load()
    _lib.check(lib.st5_attn_bwd(C.byref(a), _stream()), "st5_attn_bwd")
    _count(3)


def attn_fused_fwd(a, lse, psave=None, inv_l=None, out_f32=None):
    lib = _lib.load()
    _lib.check(lib.st5_attn_fused_fwd(C.byref(a), _ptr(lse), _ptr(psave), _ptr(inv_l), _ptr(out_f32), _stream()),
               "st5_attn_fused_fwd")
    _count(1)


def attn_flash_fwd(a, lse, psave=None, inv_l=None, out_f32=None):
    lib = _lib.load()
    _lib.check(lib.st5_attn_flash_fwd(C.byref(a), _ptr(lse), _ptr(psave), _ptr(inv_l), _ptr(out_f32), _stream()),
               "st5_attn_flash_fwd")
    _count(1)


def attn_fused_bwd(a, psave, inv_l, out_f32, delta, dq_acc, ext_heads=0):
    lib = _lib.load()
    _lib.check(lib.st5_attn_fused_bwd(C.byref(a), _ptr(psave), _ptr(inv_l), _ptr(out_f32), _ptr(delta), _ptr(dq_acc),
                                      int(ext_heads), _stream()),
               "st5_attn_fused_bwd")
    _count(3 if (a.dprobs_ext and 0 < int(ext_heads) < a.H) else 2)  # (+ the guided heads' row-constant launch)



def attn_softmax_fwd(s, qp, key_pad, p, probs_f32, pdrop, B, H, Tq, Tk, p_ld, causal, maxpos, drop_p, seed, offset):
    lib = _lib.load()
    _lib.check(lib.st5_attn_softmax_fwd(_ptr(s), _ptr(qp), qp.shape[-1] if qp is not None else 0, _ptr(key_pad),
                                        _ptr(p), _ptr(probs_f32), _ptr(pdrop), B, H, Tq, Tk, p_ld, int(causal), maxpos,
                                        drop_p, seed, offset, _stream()), "st5_attn_softmax_fwd")
    _count(1)


def attn_ds(p, dp, dp_ext, ds, pdrop, B, H, Tq, Tk, p_ld, drop_p, seed, offset):
    lib = _lib.load()
    _lib.check(lib.st5_attn_ds(_ptr(p), _ptr(dp), _ptr(dp_ext), _ptr(ds), _ptr(pdrop), B, H, Tq, Tk, p_ld, drop_p, seed,
                               offset, _stream()), "st5_attn_ds")
    _count(1)


def attn_dqp_scatter(ds, dqp, B, H, Tq, Tk, p_ld, maxpos, h_major=False):
    lib = _lib.load()
    _lib.check(lib.st5_attn_dqp_scatter(_ptr(ds), _ptr(dqp), B, H, Tq, Tk, p_ld, maxpos, int(h_major), _stream()),
               "st5_attn_dqp_scatter")
    _count(1)


def bn_fwd(x, x_ld, gamma, beta, running_mean, running_var, save_mean, save_rstd, y, y_ld, y_pre, rows, Cc, training,
           momentum, eps, act, drop_p, seed, offset, scratch):
    lib = _lib.load()
    _lib.check(lib.st5_bn_fwd(_ptr(x), x_ld, _ptr(gamma), _ptr(beta), _ptr(running_mean), _ptr(running_var),
                              _ptr(save_mean), _ptr(save_rstd), _ptr(y), y_ld, _ptr(y_pre), dtype_id(x), rows, Cc,
                              int(training), momentum, eps, ACT_IDS[act], drop_p, seed, offset, _ptr(scratch),
                              _stream()), "st5_bn_fwd")
    _count(5)


def bn_bwd(dy, dy_ld, x, x_ld, y_pre, gamma, save_mean, save_rstd, dx, dx_ld, dgamma, dbeta, rows, Cc, act, drop_p,
           seed, offset, scratch):
    lib = _lib.load()
    _lib.check(lib.st5_bn_bwd(_ptr(dy), dy_ld, _ptr(x), x_ld, _ptr(y_pre), _ptr(gamma), _ptr(save_mean),
                              _ptr(save_rstd), _ptr(dx), dx_ld, _ptr(dgamma), _ptr(dbeta), dtype_id(x), rows, Cc,
                              ACT_IDS[act], drop_p, seed, offset, _ptr(scratch), _stream()), "st5_bn_bwd")
    _count(2)


def conv0_gn_gelu_fwd(wave, w, gamma, beta, y, mean, rstd, stride, eps, act):
    """st5_conv0_gn_gelu_fwd: wave [B, n] fp32, w [C, K] fp32 -> y [B, T0, C] (y.dtype)."""
    _require_cuda(wave, w, y)
    assert wave.dtype == torch.float32 and w.dtype == torch.float32 and wave.is_contiguous() and w.is_contiguous()
    B, n = wave.shape
    Cc, Kt = w.shape
    lib = _lib.load()
    ws = torch.empty(lib.st5_conv0_ws_floats(B, n, Cc, Kt, stride), device=wave.device, dtype=torch.float32)
    _lib.check(lib.st5_conv0_gn_gelu_fwd(_ptr(wave), _ptr(w), _ptr(gamma), _ptr(beta), _ptr(y), dtype_id(y), _ptr(mean),
                                         _ptr(rstd), _ptr(ws), B, n, Cc, Kt, stride, eps, ACT_IDS[act], _stream()),
               "st5_conv0_gn_gelu_fwd")
    _count(3)


def conv0_gn_gelu_bwd(dy, wave, w, gamma, beta, mean, rstd, dw, dgamma, dbeta, stride, act):
    """st5_conv0_gn_gelu_bwd: dw / dgamma / dbeta (fp32) are accumulated."""
    _require_cuda(dy, wave, w)
    assert dy.is_contiguous()
    B, n = wave.shape
    Cc, Kt = w.shape
    lib = _lib.load()
    ws = torch.empty(lib.st5_conv0_ws_floats(B, n, Cc, Kt, stride), device=wave.device, dtype=torch.float32)
    _lib.check(lib.st5_conv0_gn_gelu_bwd(_ptr(dy), _ptr(wave), _ptr(w), _ptr(gamma), _ptr(beta), _ptr(mean), _ptr(rstd),
                                         _ptr(dw), _ptr(dgamma), _ptr(dbeta), _ptr(ws), dtype_id(dy), B, n, Cc, Kt,
                                         stride, ACT_IDS[act], _stream()), "st5_conv0_gn_gelu_bwd")
    _count(4)


def conv0_ln_gelu_fwd(wave, w, gamma, beta, y, mean, rstd, stride, eps, act):
    """st5_conv0_ln_gelu_fwd: wave [B, n] fp32, w [C, K] fp32 -> y [B, T0, C] (y.dtype), mean / rstd [B * T0]."""
    _require_cuda(wave, w, y)
    assert wave.dtype == torch.float32 and w.dtype == torch.float32 and wave.is_contiguous() and w.is_contiguous()
    B, n = wave.shape
    Cc, Kt = w.shape
    lib = _lib.load()
    _lib.check(lib.st5_conv0_ln_gelu_fwd(_ptr(wave), _ptr(w), _ptr(gamma), _ptr(beta), _ptr(y), dtype_id(y), _ptr(mean),
                                         _ptr(rstd), B, n, Cc, Kt, stride, eps, ACT_IDS[act], _stream()),
               "st5_conv0_ln_gelu_fwd")
    _count(1)


def conv0_ln_gelu_bwd(dy, wave, w, gamma, beta, mean, rstd, dw, dgamma, dbeta, stride, act):
    """st5_conv0_ln_gelu_bwd: dw / dgamma / dbeta (fp32) are accumulated."""
    _require_cuda(dy, wave, w)
    assert dy.is_contiguous()
    B, n = wave.shape
    Cc, Kt = w.shape
    lib = _lib.load()
    ws = torch.empty(lib.st5_conv0_ln_ws_floats(B, n, Cc, Kt, stride), device=wave.device, dtype=torch.float32)
    _lib.check(lib.st5_conv0_ln_gelu_bwd(_ptr(dy), _ptr(wave), _ptr(w), _ptr(gamma), _ptr(beta), _ptr(mean), _ptr(rstd),
                                         _ptr(dw), _ptr(dgamma), _ptr(dbeta), _ptr(ws), dtype_id(dy), B, n, Cc, Kt,
                                         stride, ACT_IDS[act], _stream()), "st5_conv0_ln_gelu_bwd")
    _count(4)


def act_fwd(x, y, act):
    """st5_act_fwd: y = act(x), contiguous tensors of one dtype."""
    _require_cuda(x, y)
    assert x.is_contiguous() and y.is_contiguous() and x.dtype == y.dtype
    lib = _lib.load()
    _lib.check(lib.st5_act_fwd(_ptr(x), _ptr(y), dtype_id(x), ACT_IDS[act], x.numel(), _stream()), "st5_act_fwd")
    _count(1)


def ctc_loss(logits, targets, tgt_offsets, input_lengths, target_lengths, nll, grad, s_max, blank, zero_infinity):
    """logits [T, B, V] fp32 (inner stride 1); see st5_ctc_loss (rows + concurrent alpha / beta sweeps + gradient rows)."""
    _require_cuda(logits, targets, nll)
    assert logits.dtype == torch.float32 and logits.stride(2) == 1
    for t in (targets, tgt_offsets, input_lengths, target_lengths):
        assert t.dtype == torch.int64 and t.is_contiguous()
    T, B, V = logits.shape
    assert grad is None or (grad.dtype == torch.float32 and grad.stride() == logits.stride())
    lib = _lib.load()
    ws = torch.empty(lib.st5_ctc_ws_floats(T, B, s_max), device=logits.device, dtype=torch.float32)
    _lib.check(lib.st5_ctc_loss(_ptr(logits), logits.stride(0), logits.stride(1), _ptr(targets), _ptr(tgt_offsets),
                                _ptr(input_lengths), _ptr(target_lengths), _ptr(nll), _ptr(grad), _ptr(ws), T, B, V,
                                s_max, blank, int(zero_infinity), _stream()), "st5_ctc_loss")
    _count(3 if grad is not None else 2)


def ctc_prefix_init(x, t_valid, r, blank):
    """x [B, T, V] fp32 CTC log-probabilities (inner stride 1), t_valid [B] int64 -> r [B, T, 2] fp32 (st5_ctc_prefix_init)."""
    _require_cuda(x, t_valid, r)
    assert x.dtype == torch.float32 and x.stride(2) == 1 and t_valid.dtype == torch.int64 and t_valid.is_contiguous()
    B, T, V = x.shape
    assert r.shape == (B, T, 2) and r.dtype == torch.float32 and r.is_contiguous()
    lib = _lib.load()
    _lib.check(lib.st5_ctc_prefix_init(_ptr(x), x.stride(0), x.stride(1), _ptr(t_valid), _ptr(r), B, T, V, blank,
                                       _stream()), "st5_ctc_prefix_init")
    _count(1)


def ctc_prefix_score(x, t_valid, utt, r_prev, last, out_len, cs, log_psi, r, blank, eos):
    """Candidate scores log_psi [H, K] and states r [H, T, 2, K] of H hypotheses x K candidate labels cs [H, K]
    (st5_ctc_prefix_score). x [B, T, V] fp32; utt / last / out_len [H] int64; r_prev [H, T, 2] fp32."""
    _require_cuda(x, t_valid, utt, r_prev, last, out_len, cs, log_psi, r)
    assert x.dtype == torch.float32 and x.stride(2) == 1
    for t in (t_valid, utt, last, out_len, cs):
        assert t.dtype == torch.int64 and t.is_contiguous()
    B, T, V = x.shape
    H, K = cs.shape
    assert r_prev.shape == (H, T, 2) and r_prev.dtype == torch.float32 and r_prev.is_contiguous()
    assert log_psi.shape == (H, K) and log_psi.dtype == torch.float32 and log_psi.is_contiguous()
    assert r.shape == (H, T, 2, K) and r.dtype == torch.float32 and r.is_contiguous()
    lib = _lib.load()
    _lib.check(lib.st5_ctc_prefix_score(_ptr(x), x.stride(0), x.stride(1), _ptr(utt), _ptr(r_prev), _ptr(last),
                                        _ptr(out_len), _ptr(cs), _ptr(t_valid), _ptr(log_psi), _ptr(r), H, T, K, V, blank,
                                        eos, _stream()), "st5_ctc_prefix_score")
    _count(1)


def beam_gather_rows(src, dst, parent, n_rows):
    """dst[l][h, :n_rows] = src[l][parent[h], :n_rows] for every layer l (st5_beam_gather_rows): src / dst lists of
    [*, max_len, W] tensors with contiguous rows, two distinct buffer sets; parent [H] int64 on the device."""
    _require_cuda(parent, *src, *dst)
    assert len(src) == len(dst) and parent.dtype == torch.int64 and parent.is_contiguous()
    H = parent.numel()
    s0, d0 = src[0], dst[0]
    row_bytes = s0.stride(1) * s0.element_size()
    assert s0.stride(2) == 1 and s0.stride(1) == s0.shape[2] and d0.shape[0] >= H
    for s, d in zip(src, dst):
        assert s.stride() == s0.stride() and d.stride() == d0.stride() and s.dtype == d.dtype == s0.dtype
        assert d.stride(1) == s.stride(1) and d.data_ptr() != s.data_ptr()
    n = len(src)
    lib = _lib.load()
    sp = (C.c_void_p * n)(*[s.data_ptr() for s in src])
    dp = (C.c_void_p * n)(*[d.data_ptr() for d in dst])
    _lib.check(lib.st5_beam_gather_rows(sp, dp, _ptr(parent), n, H, int(n_rows), row_bytes,
                                        s0.stride(0) * s0.element_size(), d0.stride(0) * d0.element_size(), _stream()),
               "st5_beam_gather_rows")
    _count(1)


def tts_loss_ws_floats(B, L):
    return int(_lib.load().st5_tts_loss_ws_floats(B, L))


def guided_attn_ws_floats(n_layers, B, heads, T_out):
    return int(_lib.load().st5_guided_attn_ws_floats(n_layers, B, heads, T_out))


def tts_loss_fwd(after, before, logits, ys, labels, olens, r, pos_weight, sums, out):
    """st5_tts_loss_fwd: out[0..2] = l1, l2, bce of Tacotron2Loss (masked means); after / before [B, L, D] fp32."""
    _require_cuda(after, before, logits, ys, labels, olens, sums, out)
    B, L, D = after.shape
    for t in (after, before, logits):
        assert t.dtype == torch.float32 and t.is_contiguous()
    assert ys.dtype == torch.float32 and ys.stride(2) == 1 and ys.stride(1) == D and ys.shape[1] >= L
    assert labels.dtype == torch.float32 and labels.stride(1) == 1 and olens.dtype == torch.int64 and olens.is_contiguous()
    _lib.check(_lib.load().st5_tts_loss_fwd(_ptr(after), _ptr(before), _ptr(logits), _ptr(ys), ys.stride(0), _ptr(labels),
                                            labels.stride(0), _ptr(olens), B, L, D, r, pos_weight, _ptr(sums), _ptr(out),
                                            _stream()), "st5_tts_loss_fwd")
    _count(2)


def tts_loss_bwd(after, before, logits, ys, labels, olens, sums, g, r, pos_weight, d_after, d_before, d_logits):
    _require_cuda(after, g, d_after)
    B, L, D = after.shape
    assert g.dtype == torch.float32 and g.is_contiguous() and g.numel() == 3
    for t in (d_after, d_before, d_logits):
        assert t.dtype == torch.float32 and t.is_contiguous()
    _lib.check(_lib.load().st5_tts_loss_bwd(_ptr(after), _ptr(before), _ptr(logits), _ptr(ys), ys.stride(0), _ptr(labels),
                                            labels.stride(0), _ptr(olens), _ptr(sums), _ptr(g), B, L, D, r, pos_weight,
                                            _ptr(d_after), _ptr(d_before), _ptr(d_logits), _stream()), "st5_tts_loss_bwd")
    _count(1)


def _att_layout(atts):
    B, H, T_out, T_in = atts[0].shape
    p_ld = atts[0].stride(2)
    for a in atts:
        assert a.dtype == torch.float32 and a.shape == atts[0].shape and a.stride(3) == 1 and a.stride(2) == p_ld
        assert a.stride(1) == T_out * p_ld and a.stride(0) == H * T_out * p_ld, "attention probabilities: [B,H,T_out,p_ld] pitch"
    ptrs = (C.c_void_p * len(atts))(*[a.data_ptr() for a in atts])
    return B, H, T_out, T_in, p_ld, ptrs


def guided_attn_fwd(atts, heads, ilens, olens, r, sigma, alpha, gsum, out):
    """st5_guided_attn_fwd over the first `heads` heads of each tensor in `atts` ([B, H, T_out, T_in] fp32 views)."""
    _require_cuda(atts[0], ilens, olens, gsum, out)
    B, H, T_out, T_in, p_ld, ptrs = _att_layout(atts)
    assert ilens.dtype == torch.int64 and olens.dtype == torch.int64 and ilens.is_contiguous() and olens.is_contiguous()
    _lib.check(_lib.load().st5_guided_attn_fwd(ptrs, len(atts), B, H, heads, T_out, T_in, p_ld, _ptr(ilens), _ptr(olens),
                                               r, sigma, alpha, _ptr(gsum), _ptr(out), _stream()), "st5_guided_attn_fwd")
    _count(2)


def guided_attn_bwd(datts, heads, T_in, ilens, olens, r, sigma, alpha, gsum, g, zero_rest):
    """datts: [B, H, T_out, p_ld] fp32 contiguous buffers (p_ld >= T_in)."""
    _require_cuda(datts[0], gsum, g)
    B, H, T_out, p_ld = datts[0].shape
    for d in datts:
        assert d.dtype == torch.float32 and d.is_contiguous() and d.shape == datts[0].shape
    ptrs = (C.c_void_p * len(datts))(*[d.data_ptr() for d in datts])
    _lib.check(_lib.load().st5_guided_attn_bwd(ptrs, len(datts), B, H, heads, T_out, T_in, p_ld, _ptr(ilens), _ptr(olens),
                                               r, sigma, alpha, _ptr(gsum), _ptr(g), int(zero_rest), _stream()),
               "st5_guided_attn_bwd")
    _count(1)


def sumsq(x, out):
    lib = _lib.load()
    _lib.check(lib.st5_sumsq(_ptr(x), x.numel(), _ptr(out), _stream()), "st5_sumsq")
    _count(1)


def adam_step(p, g, m, v, p_bf16, lr, beta1, beta2, eps, weight_decay, step, grad_norm_sq, max_norm, grad_mul,
              lr_dev=None, step_dev=None):
    lib = _lib.load()
    _lib.check(lib.st5_adam_step(_ptr(p), _ptr(g), _ptr(m), _ptr(v), _ptr(p_bf16), p.numel(), lr, beta1, beta2, eps,
                                 weight_decay, step, _ptr(grad_norm_sq), max_norm, grad_mul, _ptr(lr_dev),
                                 _ptr(step_dev), _stream()), "st5_adam_step")
    _count(1)
