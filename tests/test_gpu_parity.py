"""GPU parity tests: every kernel of the path, called through the C-ABI (ops.* -> ctypes -> libseamless_b200.so),
against the CPU oracle / plain fp32 torch on the same seeded inputs, plus size-independent properties at the
BASELINE widths (M=1024, 16 heads).  Tolerances are stated per test; integer outputs are compared exactly, with the
documented margin audit where fp16-vs-fp32 near ties can legitimately flip an argmax (oracle/ASSUMPTIONS.md #9)."""
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle.unity_oracle import UnityOracle, VocoderOracle, fbank as o_fbank, fbank_raw as o_fbank_raw, s2st
from seamless_communication_b200 import config as C, synthetic as S

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")
dev = "cuda"


def rel(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return ((a - b).abs().max() / (b.abs().max() + 1e-9)).item()


@pytest.fixture(scope="module")
def ops():
    from seamless_communication_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def tiny():
    cfg, vc = C.tiny_v2(), C.tiny_vocoder()
    sd = S.make_unity_state_dict(cfg, 0, dec_gain=4.0, dur_gain=1.0, dur_bias=0.9)
    vsd = S.make_vocoder_state_dict(vc, 1)
    toks = S.make_tokenizers(cfg)
    from seamless_communication_b200.models.unity import load_unity_model
    from seamless_communication_b200.models.vocoder import load_vocoder_model
    model = load_unity_model("tiny_v2", state_dict=sd, tokenizers=toks)
    voc = load_vocoder_model("tiny", state_dict=vsd)
    return dict(cfg=cfg, vc=vc, sd=sd, vsd=vsd, toks=toks, model=model, voc=voc,
                uo=UnityOracle(cfg.to_dict(), sd, toks), vo=VocoderOracle(vc.to_dict(), vsd))


@pytest.fixture(scope="module")
def small():
    from seamless_communication_b200.models.unity import load_unity_model
    return load_unity_model("small_v2", synthetic=True, seed=7, dec_gain=4.0)


# ------------------------------------------------------------------------------------------------ sb_gemm
@pytest.mark.parametrize("m,n,k", [(128, 128, 64), (300, 200, 1024), (160, 3072, 1024), (1000, 1024, 4096), (513, 72, 160),
                                   (77, 10082, 128), (2000, 16, 16)])
def test_gemm_linear(ops, m, n, k):
    torch.manual_seed(m + n + k)
    a = (torch.randn(m, k, device=dev) * 0.5).half()
    w = (torch.randn(n, k, device=dev) * 0.05).half()
    bias = torch.randn(n, device=dev)
    ref = a.float() @ w.float().t() + bias
    for f32 in (False, True):
        out = ops.gemm_raw(a, w, n, bias, out_f32=f32)
        simt = ops.gemm_raw(a, w, n, bias, out_f32=f32, ref=True)
        assert rel(out, ref) < 2e-3 and rel(out, simt) < 2e-3  # fp16 inputs, fp32 accumulate; fp16 output rounding


def test_gemm_wide_tiles_256(ops):
    """gemm_tc_kernel<256> (two 48 KB stages, 2 CTAs/SM) is selected for fp16 single-output products with n % 256 == 0
    and >= 296 tiles - the encoder / T2U / vocoder shapes: every epilogue it serves against fp32 torch (bias, SiLU, GLU,
    residual + scales, conv taps over a ragged sequence batch with zeroed padding)."""
    from seamless_communication_b200.ops import Seq
    torch.manual_seed(256)
    m, k = 10000, 320  # 79 M tiles x (n / 256) >= 296 for n >= 1024
    a = (torch.randn(m, k, device=dev) * 0.5).half()
    for n in (1024, 1280):
        w = (torch.randn(n, k, device=dev) * 0.05).half()
        bias = torch.randn(n, device=dev)
        ref = a.float() @ w.float().t() + bias
        out = ops.gemm_raw(a, w, n, bias)
        assert rel(out, ref) < 2e-3 and rel(out, ops.gemm_raw(a, w, n, bias, ref=True)) < 2e-3
        assert rel(ops.gemm_raw(a, w, n, bias, act=ops.ACT_SILU), F.silu(ref)) < 2e-3
        assert rel(ops.gemm_raw(a, w, n, bias, glu=True), ref[:, 0::2] * torch.sigmoid(ref[:, 1::2])) < 2e-3
        r1 = torch.randn(m, n, device=dev).half()
        assert rel(ops.gemm_raw(a, w, n, bias, alpha=0.5, res1=r1), ref * 0.5 + r1.float()) < 2e-3
    # 3-tap conv over sequences (full, ragged, empty): halo / padded rows exactly zero
    B, T, Cc, N, taps = 40, 300, 128, 1024, 3
    lens = torch.full((B,), T, dtype=torch.int32, device=dev)
    lens[1], lens[2] = 77, 0
    x = Seq(B, T, Cc, halo=1, lens=lens)
    x.data().copy_((torch.randn(B, T, Cc, device=dev) * 0.5).half())
    w = (torch.randn(N, taps * Cc, device=dev) * 0.05).half()
    bias = torch.randn(N, device=dev)
    res = x.like(C=N, zero=True)
    res.data().copy_(torch.randn(B, T, N, device=dev).half())
    o = ops.gemm(x, w, N, bias, taps=taps, act=ops.ACT_RELU, res1=res, alpha=0.5)
    y = F.conv1d(x.data().float().transpose(1, 2), w.float().view(N, taps, Cc).permute(0, 2, 1), bias, padding=1).transpose(1, 2)
    y = (F.relu(y) * 0.5 + res.data().float()) * (torch.arange(T, device=dev)[None] < lens[:, None])[:, :, None]
    assert rel(o.data(), y) < 2e-3
    full = o.buf.float().view(B, o.Tp, N)
    assert full[:, :o.PH].abs().max() == 0 and full[:, o.PH + T:].abs().max() == 0
    assert full[1, o.PH + 77:].abs().max() == 0 and full[2].abs().max() == 0


@pytest.mark.parametrize("taps,dil", [(1, 1), (3, 1), (7, 1), (11, 5), (3, 3)])
def test_gemm_conv_mask_residual_dual_output(ops, taps, dil):
    from seamless_communication_b200.ops import Seq
    torch.manual_seed(taps * 10 + dil)
    B, T, Cc, N = 3, 150, 64, 128
    halo = (taps - 1) * dil // 2
    lens = torch.tensor([150, 33, 0], dtype=torch.int32, device=dev)  # full, ragged and EMPTY sequence
    x = Seq(B, T, Cc, halo=max(halo, 1), lens=lens)
    x.data().copy_((torch.randn(B, T, Cc, device=dev) * 0.5).half())
    w = (torch.randn(N, taps * Cc, device=dev) * 0.05).half()
    bias = torch.randn(N, device=dev)
    res, res2 = x.like(C=N, zero=True), x.like(C=N, zero=True)
    res.data().copy_(torch.randn(B, T, N, device=dev).half())
    res2.data().copy_(torch.randn(B, T, N, device=dev).half())
    o2 = x.like(C=N, zero=True)
    o = ops.gemm(x, w, N, bias, taps=taps, dil=dil, act=ops.ACT_LRELU, slope=0.1, res1=res, res2=res2, alpha=0.5, gamma=1 / 3,
                 out2=o2, out2_slope=0.01)
    xc = x.data().float().transpose(1, 2)
    wt = w.float().view(N, taps, Cc).permute(0, 2, 1)
    y = F.conv1d(xc, wt, bias, padding=halo, dilation=dil).transpose(1, 2)
    y = (F.leaky_relu(y, 0.1) * 0.5 + res.data().float() + res2.data().float()) / 3
    y = y * (torch.arange(T, device=dev)[None] < lens[:, None])[:, :, None]
    assert rel(o.data(), y) < 2e-3
    assert rel(o2.data(), F.leaky_relu(y, 0.01)) < 2e-3
    # halo rows and rows past each sequence's length are exactly zero
    full = o.buf.float().view(B, o.Tp, N)
    assert full[:, :o.PH].abs().max() == 0 and full[:, o.PH + T:].abs().max() == 0
    assert full[1, o.PH + 33:].abs().max() == 0 and full[2].abs().max() == 0


@pytest.mark.parametrize("rows,n,k,splits", [(160, 1024, 1024, 8), (160, 192, 128, 2), (37, 64, 512, 4), (1, 128, 64, 1),
                                             (150, 256, 1024, 16)])
def test_gemm_skinny_matches_simt_reference(ops, rows, n, k, splits):
    """skinny_gemm.cu (cp.async + mma.sync, the decoder-step GEMM at <= 160 rows): split-K partials sum to the product,
    and the direct mode applies bias + ReLU; both against the CUDA-core reference kernel."""
    from seamless_communication_b200.ops import Seq
    torch.manual_seed(rows + n)
    a = Seq(1, rows, k, buf=torch.randn(rows, k, device=dev).half())
    w = (torch.randn(n, k, device=dev) / math.sqrt(k)).half()
    bias = torch.randn(n, device=dev)
    want = ops.gemm_raw(a.buf, w, n, bias, act=ops.ACT_RELU, out_f32=True, ref=True)
    SR = ops.slice_rows(rows)
    part = torch.full((splits * SR, n), float("nan"), device=dev)
    ops.gemm_splitk(a, w, n, splits, part, skinny=True)
    got = part.view(splits, SR, n)[:, :rows].sum(0) + bias
    assert torch.isnan(part.view(splits, SR, n)[:, rows:]).all()  # rows past `rows` are never written
    assert (torch.relu(got) - want).abs().max() < 2e-3
    out = Seq(1, rows, n)
    out.buf.fill_(float("nan"))
    ops.gemm_skinny(a, w, n, bias, act=ops.ACT_RELU, out=out)
    assert (out.buf.float() - want).abs().max() < 4e-3  # + fp16 rounding of the output
    # same partials as the tcgen05 split-K kernel up to fp32 summation order
    part2 = torch.zeros((splits * SR, n), device=dev)
    ops.gemm_splitk(a, w, n, splits, part2)
    assert (part2.view(splits, SR, n)[:, :rows].sum(0) + bias - got).abs().max() < 1e-3


@pytest.mark.parametrize("rows,n,k,splits", [(160, 3072, 1024, 6), (160, 1024, 8192, 16), (160, 8192, 1024, 1), (40, 384, 128, 2),
                                             (5, 256, 128, 1), (256, 200, 192, 3), (33, 1126, 128, 1)])
def test_gemm_decode_transposed_matches_simt_reference(ops, rows, n, k, splits):
    """decode_gemm.cu (weights as the tcgen05 A operand, all rows as B): split-K partials sum to the product (uneven K
    slices, ragged last feature tile, rows that are not a multiple of 16), and the direct mode applies bias + ReLU; both
    against the CUDA-core reference kernel."""
    from seamless_communication_b200.ops import Seq
    torch.manual_seed(rows + n + splits)
    a = Seq(1, rows, k, buf=torch.randn(rows, k, device=dev).half())
    w = (torch.randn(n, k, device=dev) / math.sqrt(k)).half()
    bias = torch.randn(n, device=dev)
    want = ops.gemm_raw(a.buf, w, n, bias, act=ops.ACT_RELU, out_f32=True, ref=True)
    SR = ops.slice_rows(rows)
    part = torch.full((splits * SR, n), float("nan"), device=dev)
    ops.gemm_splitk(a, w, n, splits, part, transposed=True)
    got = part.view(splits, SR, n)[:, :rows].sum(0) + bias
    assert torch.isnan(part.view(splits, SR, n)[:, rows:]).all()  # rows past `rows` are never written
    assert (torch.relu(got) - want).abs().max() < 2e-3
    out = Seq(1, rows, n)
    out.buf.fill_(float("nan"))
    ops.gemm_decode(a, w, n, bias, act=ops.ACT_RELU, out=out)
    assert (out.buf.float() - want).abs().max() < 4e-3  # + fp16 rounding of the output
    lin = ops.gemm_decode(a, w, n, None)
    assert (lin.buf.float() - (a.buf.float() @ w.float().t())).abs().max() < 4e-3


@pytest.mark.parametrize("taps,Cc", [(3, 16), (7, 16), (11, 32), (11, 8)])
def test_gemm_narrow_channel_conv(ops, taps, Cc):
    """C < 64 with dilation 1 takes the overlapping-row (K-collapsed) tensor-map path."""
    from seamless_communication_b200.ops import Seq
    torch.manual_seed(taps + Cc)
    B, T, N = 2, 700, Cc
    halo = (taps - 1) // 2
    x = Seq(B, T, Cc, halo=halo + 2)
    x.data().copy_((torch.randn(B, T, Cc, device=dev) * 0.5).half())
    w = (torch.randn(N, taps * Cc, device=dev) * 0.1).half()
    bias = torch.randn(N, device=dev)
    o = ops.gemm(x, w, N, bias, taps=taps, act=ops.ACT_LRELU, slope=0.1)
    r = ops.gemm(x, w, N, bias, taps=taps, act=ops.ACT_LRELU, slope=0.1, ref=True)
    y = F.conv1d(x.data().float().transpose(1, 2), w.float().view(N, taps, Cc).permute(0, 2, 1), bias, padding=halo)
    y = F.leaky_relu(y, 0.1).transpose(1, 2)
    assert rel(o.data(), y) < 2e-3 and rel(o.data(), r.data()) < 2e-3
    full = o.buf.float().view(B, o.Tp, N)
    assert full[:, :o.PH].abs().sum() == 0 and full[:, o.PH + T:].abs().sum() == 0


def test_gemm_glu_and_splitk(ops):
    from seamless_communication_b200.ops import Seq
    torch.manual_seed(5)
    x = Seq(2, 80, 256)
    x.buf.copy_((torch.randn(160, 256, device=dev) * 0.5).half())
    w = (torch.randn(512, 256, device=dev) * 0.1).half()
    b = torch.randn(512, device=dev)
    g = ops.gemm(x, w, 512, b, glu=True)
    full = x.buf.float() @ w.float().t() + b
    assert rel(g.buf, full[:, 0::2] * torch.sigmoid(full[:, 1::2])) < 2e-3
    # split-K partials + fused reduce/LayerNorm == unsplit GEMM + residual + LayerNorm
    xk = Seq(1, 160, 2048)
    xk.buf.copy_((torch.randn(160, 2048, device=dev) * 0.3).half())
    wk = (torch.randn(1024, 2048, device=dev) * 0.03).half()
    bk, lw, lb = torch.randn(1024, device=dev) * 0.1, torch.randn(1024, device=dev), torch.randn(1024, device=dev)
    resid = Seq(1, 160, 1024)
    resid.buf.copy_(torch.randn(160, 1024, device=dev).half())
    want_x = (xk.buf.float() @ wk.float().t() + bk + resid.buf.float()).half()
    want_h = F.layer_norm(want_x.float(), (1024,), lw, lb, 1e-5)
    for splits in (1, 4, 8):
        part = torch.empty((splits * ops.slice_rows(160), 1024), dtype=torch.float32, device=dev)
        xs = Seq(1, 160, 1024, buf=resid.buf.clone())
        h = Seq(1, 160, 1024)
        ops.gemm_splitk(xk, wk, 1024, splits, part)
        ops.splitk_reduce_ln(part, splits, bk, xs, lw, lb, h)
        assert rel(xs.buf, want_x) < 2e-3 and rel(h.buf, want_h) < 3e-3


# ------------------------------------------------------------------------------------------------ a1 fbank
def test_fbank_matches_oracle_and_knf_golden(ops):
    w = S.make_waveforms(4, 32000)
    ns = torch.tensor([32000, 20000, 399, 400], dtype=torch.int32)  # full, ragged, too short (0 frames), exactly 1 frame
    fb, frames = ops.fbank(w.to(dev), ns.to(dev), 198)
    assert frames.tolist() == [198, 123, 0, 1]
    for i in range(2):
        ref = o_fbank(w[i, :ns[i]])
        # standardised log-mel ~N(0,1); fp16 output rounding + fp32 FFT order: atol 4e-3 is the reference's own
        # tolerance between its two fbank implementations (ggml/test_unity_cpp.py:584)
        assert (fb[i, :ref.shape[0]].float().cpu() - ref).abs().max() < 4e-3
        assert fb[i, ref.shape[0]:].abs().sum() == 0
    assert fb[2].abs().sum() == 0
    d = np.load(os.path.join(G, "knf_fbank.npz"))  # produced by the reference's own kaldi-native-fbank
    raw, fr = ops.fbank(torch.from_numpy(d["wave"]).to(dev), torch.full((2,), 8000, dtype=torch.int32, device=dev), 48,
                        standardize=False)
    assert fr.tolist() == [48, 48]
    assert np.abs(raw.float().cpu().numpy() - d["fbank"]).max() < 2e-2  # raw log-mel values up to ~27 stored as fp16


# ------------------------------------------------------------------------------------------------ LN / attention / dwconv
def test_layernorm_attention_dwconv(ops):
    from seamless_communication_b200.ops import Seq
    torch.manual_seed(1)
    x = Seq(3, 37, 1024, lens=torch.tensor([37, 5, 0], dtype=torch.int32, device=dev))
    x.buf.copy_(torch.randn(111, 1024, device=dev).half())
    w, b = torch.randn(1024, device=dev), torch.randn(1024, device=dev)
    y = ops.layernorm(x, w, b, mask=True)
    ref = F.layer_norm(x.buf.float(), (1024,), w, b, 1e-5).view(3, 37, 1024)
    ref = ref * (torch.arange(37, device=dev)[None] < x.lens[:, None])[:, :, None]
    assert rel(y.buf.view(3, 37, 1024), ref) < 2e-3
    B, H, Sq, M = 2, 4, 150, 256
    qkv = Seq(B, Sq, 3 * M, lens=torch.tensor([150, 97], dtype=torch.int32, device=dev))
    qkv.buf.copy_(torch.randn(B * Sq, 3 * M, device=dev).half())
    relk = (torch.randn(73, 64, device=dev) * 0.125).half()
    q, k, v = [t.float().view(B, Sq, H, 64).transpose(1, 2) for t in qkv.buf.view(B, Sq, 3 * M).split(M, dim=2)]
    for causal, rk in [(False, None), (True, None), (False, relk)]:
        out = ops.self_attention(qkv, H, causal=causal, rel_k=rk, rel_left=64, rel_right=8)
        s = q @ k.transpose(2, 3)
        if rk is not None:
            idx = (torch.arange(Sq, device=dev)[None] - torch.arange(Sq, device=dev)[:, None]).clamp(-64, 8) + 64
            s = s + torch.einsum("nhsk,stk->nhst", q, rk.float()[idx])
        s = (s * 0.125).masked_fill(~(torch.arange(Sq, device=dev)[None] < qkv.lens[:, None])[:, None, None, :], -math.inf)
        if causal:
            s = s.masked_fill(~torch.ones(Sq, Sq, dtype=torch.bool, device=dev).tril(), -math.inf)
        ref = (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(B * Sq, M)
        assert rel(out.buf, ref) < 2e-3
    xc = Seq(2, 45, 256)
    xc.buf.copy_(torch.randn(90, 256, device=dev).half())
    wd = (torch.randn(256, 31, device=dev) * 0.2).half()
    lw, lb = torch.randn(256, device=dev), torch.randn(256, device=dev)
    for kk in (31, 15):  # 31: register-resident fixed-size kernel (w2v-BERT 2.0); other sizes: generic kernel
        wk = wd[:, :kk].contiguous()
        yd = ops.dwconv_ln_silu(xc, wk, lw, lb, kk)
        c = F.conv1d(F.pad(xc.buf.float().view(2, 45, 256).transpose(1, 2), (kk - 1, 0)), wk.float().view(256, 1, kk), groups=256)
        ref = F.silu(F.layer_norm(c.transpose(1, 2), (256,), lw, lb, 1e-5)).reshape(90, 256)
        assert rel(yd.buf, ref) < 2e-3


def test_logits_topk_exact(ops):
    from seamless_communication_b200 import _lib
    lib = _lib.load()
    R, V, K = 7, 50001, 11
    ld = (V + 7) // 8 * 8
    torch.manual_seed(2)
    logits = torch.randn(R, ld, device=dev) * 4
    logits[3, 10:40] = 100.0  # massive exact ties at the top: lowest indices must win
    cv = torch.empty(R, K, device=dev); ci = torch.empty(R, K, dtype=torch.int32, device=dev); el = torch.empty(R, device=dev)
    _lib.check(lib.sb_logits_topk(logits.data_ptr(), ld, R, V, 0, 3, 1, 0.5, K, cv.data_ptr(), ci.data_ptr(), el.data_ptr(),
                                  torch.cuda.current_stream().cuda_stream))
    lp = torch.log_softmax(logits[:, :V], -1)
    assert (el - lp[:, 3]).abs().max() < 1e-4
    lp[:, 0] = -math.inf  # pad never allowed
    lp[:, 1] -= 0.5       # unk penalty
    tv, ti = torch.topk(lp, K)
    assert (tv - cv).abs().max() < 1e-4
    assert ci[3].tolist() == list(range(10, 21))
    for r in (0, 1, 2, 4, 5, 6):
        assert ci[r].tolist() == ti[r].tolist()


def test_logits_topk_from_projection_tile_statistics_exact(ops):
    """sb_gemm(tile_stats=...) + sb_logits_topk_tiles: the log-softmax statistics leave the projection's epilogue and only
    the tiles that can hold a top-K candidate are read back.  Same answers as log_softmax + topk over the produced fp32
    logits: values, indices (lowest index first on exact ties), the lprob of an arbitrary token; PAD excluded, UNK penalised;
    ragged last tile; PAD / UNK / tied tokens heading the row."""
    from seamless_communication_b200 import _lib
    from seamless_communication_b200.ops import Seq
    lib = _lib.load()
    R, V, K, D = 37, 20000 + 102, 11, 256
    torch.manual_seed(8)
    a = Seq(1, R, D, buf=torch.randn(R, D, device=dev).half())
    w = (torch.randn(V, D, device=dev) * 0.25).half()
    w[0] = a.buf[3] * 0.5            # PAD would be the best token of row 3
    w[1] = a.buf[5] * 0.5            # UNK would be the best token of row 5 (before the penalty)
    w[700:740] = a.buf[9] * 0.4      # forty exactly tied best tokens for row 9, spanning two tiles
    w[V - 1] = a.buf[11] * 0.5       # best token of row 11 sits in the ragged last tile
    ld = (V + 7) // 8 * 8
    logits = Seq(1, R, V, dtype=torch.float32, buf=torch.full((R, ld), float("nan"), device=dev))
    stats = torch.full(((V + 127) // 128, R, 2), float("nan"), device=dev)
    ops.gemm(a, w, V, None, out=logits, out_f32=True, tile_stats=stats)
    lg = logits.buf[:, :V]
    assert torch.isfinite(lg).all() and torch.isfinite(stats).all()
    # the statistics themselves
    tiles = lg.new_full((R, stats.shape[0] * 128), -math.inf)
    tiles[:, :V] = lg
    tiles = tiles.view(R, -1, 128)
    assert torch.equal(stats[:, :, 0].t(), tiles.max(-1).values)
    assert torch.allclose(stats[:, :, 1].t(), torch.exp(tiles - tiles.max(-1, keepdim=True).values).sum(-1), rtol=1e-5)
    cv = torch.empty(R, K, device=dev); ci = torch.empty(R, K, dtype=torch.int32, device=dev); el = torch.empty(R, device=dev)
    _lib.check(lib.sb_logits_topk_tiles(logits.buf.data_ptr(), ld, stats.data_ptr(), R, V, 0, 3, 1, 2.5, K, cv.data_ptr(), ci.data_ptr(),
                                        el.data_ptr(), torch.cuda.current_stream().cuda_stream))
    lp = torch.log_softmax(lg, -1)
    assert (el - lp[:, 3]).abs().max() < 1e-4
    lp[:, 0] = -math.inf
    lp[:, 1] -= 2.5
    tv, ti = torch.sort(lp, dim=-1, descending=True, stable=True)  # stable: the lowest index first among exact ties
    tv, ti = tv[:, :K], ti[:, :K]
    assert (tv - cv).abs().max() < 1e-4
    assert ci[9].tolist() == list(range(700, 711))     # exact ties: lowest indices win
    assert ci[11, 0].item() == V - 1
    assert 0 not in ci[3].tolist()                     # PAD is never a candidate
    for r in range(R):
        assert ci[r].tolist() == ti[r].tolist(), r
    # and it agrees with the two-pass kernel on the same logits
    cv2 = torch.empty_like(cv); ci2 = torch.empty_like(ci); el2 = torch.empty_like(el)
    _lib.check(lib.sb_logits_topk(logits.buf.data_ptr(), ld, R, V, 0, 3, 1, 2.5, K, cv2.data_ptr(), ci2.data_ptr(), el2.data_ptr(),
                                  torch.cuda.current_stream().cuda_stream))
    assert torch.equal(ci, ci2) and (cv - cv2).abs().max() < 1e-5


# ------------------------------------------------------------------------------------------------ encoder (a3-a6)
def test_encoder_matches_oracle_ragged(tiny, ops):
    waves = S.make_waveforms(3, 32000)
    ns = torch.tensor([32000, 23456, 16001], dtype=torch.int32)
    fb, frames = ops.fbank(waves.to(dev), ns.to(dev), 198)
    eng, uo = tiny["model"].engine, tiny["uo"]
    enc, lens, inner = eng.encode_speech(fb, frames, return_inner=True)
    ofb = torch.zeros(3, 198, 80)
    for i in range(3):
        f = o_fbank(waves[i, :ns[i]])
        ofb[i, :f.shape[0]] = f
    o_enc, o_lens, o_inner = uo.encode_speech(ofb, frames.cpu().long(), return_inner=True)
    assert lens.tolist() == o_lens.tolist()
    M = tiny["cfg"].model_dim
    for i in range(3):  # compare valid frames only; the oracle and the kernels may differ on padded garbage rows
        n_in, n_out = int(frames[i]) // 2, int(o_lens[i])
        assert rel(inner.buf.view(3, -1, M)[i, :n_in], o_inner[i, :n_in]) < 5e-3
        assert rel(enc.buf.view(3, -1, M)[i, :n_out], o_enc[i, :n_out]) < 5e-3


# ------------------------------------------------------------------------------------------------ decoder + beam search (a7-a10)
def _oracle_score(uo, enc_row, ids):
    ids = torch.tensor(ids)[None]
    h = uo.decoder(uo.embed_text(ids[:, :-1], 0), enc_row, None)
    lp = torch.log_softmax(uo.project(h).float(), -1)[0]
    return sum(float(lp[t, ids[0, t + 1]]) for t in range(ids.shape[1] - 1)) / (ids.shape[1] - 1)


def test_decoder_and_beam_search_match_oracle(tiny, ops):
    from seamless_communication_b200.ops import Seq
    cfg, uo, eng = tiny["cfg"], tiny["uo"], tiny["model"].engine
    waves = S.make_waveforms(3, 32000)
    fb = torch.stack([o_fbank(w) for w in waves])
    ref = uo.generate(fb, None, "spa", hard_max=24, output_units=False)
    M = cfg.model_dim
    enc = Seq(3, ref["enc"].shape[1], M, buf=ref["enc"].to(dev).half().reshape(-1, M).contiguous())
    prefix = [cfg.text_eos, tiny["toks"][0].lang_index("spa")]
    hyps = eng.beam_search(enc, None, prefix, beam=5, hard_max=24)
    for i in range(3):
        assert len(hyps[i]) == len(ref["hyps"][i]) == 5
        if hyps[i][0][1] != ref["text_ids"][i]:  # margin audit: a near tie under the oracle's own scoring
            assert abs(_oracle_score(uo, ref["enc"][i:i + 1], hyps[i][0][1]) - ref["hyps"][i][0][0]) < 2e-2
        assert abs(hyps[i][0][0] - ref["hyps"][i][0][0]) < 2e-2
    assert sum(h[0][1] == r for h, r in zip(hyps, ref["text_ids"])) >= 2
    # eager (no CUDA graph) and graph-replayed searches agree exactly
    hyps_eager = eng.beam_search(enc, None, prefix, beam=5, hard_max=24, use_graph=False)
    assert [h[0][1] for h in hyps_eager] == [h[0][1] for h in hyps]
    # teacher-forced pass: hidden states and logits (fp16 kernels vs fp32 oracle; logit std ~4)
    L = max(len(s) for s in ref["text_ids"])
    ts = torch.zeros(3, L, dtype=torch.int64)
    for i, s in enumerate(ref["text_ids"]):
        ts[i, :len(s)] = torch.tensor(s)
    ts = ts[:, :-1].contiguous()
    tl = torch.tensor([len(s) - 1 for s in ref["text_ids"]], dtype=torch.int32, device=dev)
    dec = eng.decode_full(ts.to(dev), tl, enc, None)
    o_dec = uo.decoder(uo.embed_text(ts, 0), ref["enc"], None, None, self_km=(torch.arange(L - 1)[None] < tl.cpu()[:, None]))
    assert rel(dec.buf.view(3, L - 1, M), o_dec) < 5e-3
    lg = ops.gemm_raw(dec.buf, eng.w["text_embed"], cfg.text_vocab, out_f32=True).view(3, L - 1, -1)
    assert (lg.float().cpu() - uo.project(o_dec)).abs().max() < 5e-2


def test_harvested_decoder_states_equal_teacher_forced_pass(tiny):
    from seamless_communication_b200.ops import Seq
    cfg, eng = tiny["cfg"], tiny["model"].engine
    torch.manual_seed(6)
    M, S_enc = cfg.model_dim, 15
    e = Seq(3, S_enc, M, buf=torch.randn(3 * S_enc, M, device=dev).half())
    lens = torch.tensor([15, 9, 15], dtype=torch.int32, device=dev)
    hyps = eng.beam_search(e, lens, [cfg.text_eos, tiny["toks"][0].lang_index("spa")], beam=5, soft_max=(1, 8))
    seqs = [h[0][1] for h in hyps]
    got = eng.harvest_decoder_states([len(s) - 1 for s in seqs])
    L = max(len(s) for s in seqs)
    ts = torch.zeros(3, L, dtype=torch.int64)
    for i, s in enumerate(seqs):
        ts[i, :len(s)] = torch.tensor(s)
    tl = torch.tensor([len(s) - 1 for s in seqs], dtype=torch.int32, device=dev)
    want = eng.decode_full(ts[:, :-1].contiguous().to(dev), tl, e, lens)
    for i, s in enumerate(seqs):
        n = len(s) - 1
        assert rel(got.buf.view(3, -1, M)[i, :n], want.buf.view(3, -1, M)[i, :n]) < 5e-3  # incremental vs full-pass fp16 order
        assert got.buf.view(3, -1, M)[i, n:].abs().sum() == 0


def test_beam_search_sentence_groups_on_streams_equal_single_group(tiny, monkeypatch):
    """beam_search cuts the batch into sentence groups stepped concurrently on separate streams; hypotheses, scores and
    harvested decoder states must not depend on the grouping."""
    from seamless_communication_b200.ops import Seq
    cfg, eng = tiny["cfg"], tiny["model"].engine
    torch.manual_seed(11)
    M, S_enc, B = cfg.model_dim, 10, 9
    e = Seq(B, S_enc, M, buf=torch.randn(B * S_enc, M, device=dev).half())
    lens = torch.tensor([10, 4, 10, 7, 10, 10, 2, 9, 10], dtype=torch.int32, device=dev)
    prefix = [cfg.text_eos, tiny["toks"][0].lang_index("spa")]
    out = {}
    for g in (1, 2, 3):
        monkeypatch.setenv("SB_SEARCH_GROUPS", str(g))
        hyps = eng.beam_search(e, lens, prefix, beam=4, soft_max=(1, 6))
        states = eng.harvest_decoder_states([len(h[0][1]) - 1 for h in hyps])
        out[g] = (hyps, states.buf.clone())
    assert len(eng._last_search_states) == 2  # 9 sentences: at most B // 4 groups
    for g in (2, 3):
        for h1, hg in zip(out[1][0], out[g][0]):
            assert [x[1] for x in h1] == [x[1] for x in hg]
            assert np.allclose([x[0] for x in h1], [x[0] for x in hg], rtol=0, atol=1e-6)
        assert torch.equal(out[1][1], out[g][1])


@pytest.mark.parametrize("which", ["tiny", "small"])
def test_persistent_decoder_step_equals_launch_chain(tiny, small, which):
    """sb_decoder_step (one persistent kernel per step: csrc/decoder_step.cu) against the per-op launch chain it
    replaces, on the same search: the final-LayerNorm state of every step within fp16 accumulation-order noise, the
    same hypotheses (or a margin-audited near tie), and the K/V cache written identically up to rounding."""
    from seamless_communication_b200.ops import Seq
    eng = (tiny["model"] if which == "tiny" else small).engine
    cfg = eng.cfg
    torch.manual_seed(21)
    M, S_enc, B, beam = cfg.model_dim, 13, (7 if which == "tiny" else 32), 5
    e = Seq(B, S_enc, M, buf=torch.randn(B * S_enc, M, device=dev).half())
    lens = torch.randint(3, S_enc + 1, (B,), dtype=torch.int32, device=dev)
    lens[0] = S_enc
    prefix = [cfg.text_eos, eng.text_tokenizer.lang_index("spa")]
    out = {}
    old = eng.decode_fused
    try:
        for fused in (False, True):
            eng.decode_fused = fused
            hyps = eng.beam_search(e, lens, prefix, beam=beam, soft_max=(1, 9), hard_max=40)
            st = eng._last_search_states[0]
            assert (st["ds_launch"] is not None) == fused
            n = min(len(h[0][1]) for h in hyps) - 1
            kc = st["kc"][cfg.dec_layers - 1]
            R = st["R"]
            # the launch chain keeps K time-major [t][slot][M], the persistent kernel head-major [slot][head][t][64]
            kc = (kc.view(R, eng.H, st["ML"], 64).permute(2, 0, 1, 3).reshape(st["ML"], R, M) if fused else kc)[:n]
            out[fused] = (hyps, st["hist"][:n].clone(), kc.clone())
    finally:
        eng.decode_fused = old
    (h0, hist0, kc0), (h1, hist1, kc1) = out[False], out[True]
    # step 0..1 see identical inputs on both paths (same prefix): states agree to accumulation-order noise
    assert rel(hist1[:2], hist0[:2]) < 4e-3 and rel(kc1[:2], kc0[:2]) < 4e-3
    same = sum(a[0][1] == b[0][1] for a, b in zip(h0, h1))
    assert same >= B - max(1, B // 8), f"only {same}/{B} best hypotheses agree"
    for a, b in zip(h0, h1):
        assert abs(a[0][0] - b[0][0]) < 2e-2
    # determinism of the persistent kernel: a second search is bit-identical
    eng.decode_fused = True
    try:
        hyps2 = eng.beam_search(e, lens, prefix, beam=beam, soft_max=(1, 9), hard_max=40)
        st = eng._last_search_states[0]
        assert [h[0][1] for h in hyps2] == [h[0][1] for h in h1]
        assert torch.equal(st["hist"][:hist1.shape[0]], hist1)
    finally:
        eng.decode_fused = old


def test_beam_search_ragged_encoder_and_early_eos(tiny):
    """Sentences with different encoder lengths, searched together, equal the same sentences searched alone."""
    from seamless_communication_b200.ops import Seq
    cfg, eng = tiny["cfg"], tiny["model"].engine
    torch.manual_seed(3)
    M, S_enc = cfg.model_dim, 12
    e = torch.randn(3, S_enc, M, device=dev).half()
    lens = torch.tensor([12, 7, 3], dtype=torch.int32, device=dev)
    prefix = [cfg.text_eos, tiny["toks"][0].lang_index("fra")]
    together = eng.beam_search(Seq(3, S_enc, M, buf=e.reshape(-1, M).contiguous()), lens, prefix, beam=3, soft_max=(1, 5))
    for i in range(3):
        alone = eng.beam_search(Seq(1, S_enc, M, buf=e[i].contiguous()), lens[i:i + 1], prefix, beam=3, soft_max=(1, 5))
        assert alone[0][0][1] == together[i][0][1]
        assert abs(alone[0][0][0] - together[i][0][0]) < 1e-4
        assert together[i][0][1][-1] == cfg.text_eos and len(together[i][0][1]) <= 17


# ------------------------------------------------------------------------------------------------ T2U (a11-a14)
def test_text_to_chars_matches_reference_fixture(tiny):
    """sb_text_to_chars (per-token tables) against char sequences / lengths produced by the reference's own
    NARDecoderFrontend.text_to_char_seqs (tests/golden/nar_frontend.npz): punctuation merge rules, unk, pad, bare space."""
    from seamless_communication_b200.ops import Seq
    cfg, eng = tiny["cfg"], tiny["model"].engine
    d = np.load(os.path.join(G, "nar_frontend.npz"))
    ts = torch.from_numpy(d["text_seqs"]).to(dev)
    B, L = ts.shape
    dec = Seq(B, L, cfg.model_dim, buf=(torch.randn(B * L, cfg.model_dim, device=dev) * 0.5).half(),
              lens=torch.tensor([L, 7, 6], dtype=torch.int32, device=dev))
    _, _, aux = eng.t2u(dec, ts)
    assert np.array_equal(aux["char_lens"].cpu().numpy(), d["char_lens"])
    assert np.array_equal(aux["char_seq_lens"].cpu().numpy(), d["char_seq_lens"])
    got = aux["char_seqs"].cpu().numpy()
    for b in range(B):
        m = int(d["char_seq_lens"][b])
        assert np.array_equal(got[b, :m], d["char_seqs"][b, :m])


def test_t2u_matches_oracle(tiny):
    from seamless_communication_b200.ops import Seq
    cfg, uo, eng = tiny["cfg"], tiny["uo"], tiny["model"].engine
    waves = S.make_waveforms(3, 32000)
    fb = torch.stack([o_fbank(w) for w in waves])
    ref = uo.generate(fb, None, "spa", hard_max=24)
    M = cfg.model_dim
    tl = torch.tensor([len(s) - 1 for s in ref["text_ids"]], dtype=torch.int32, device=dev)
    dseq = Seq(3, ref["dec_out"].shape[1], M, lens=tl, buf=ref["dec_out"].to(dev).half().reshape(-1, M).contiguous())
    ts = ref["text_seqs"].to(dev)
    units, ulens, aux = eng.t2u(dseq, ts)
    assert torch.equal(aux["char_lens"].cpu().long(), ref["chars"][2])        # integer work: exact
    assert aux["char_seq_lens"].tolist() == ref["chars"][1].tolist()
    cs = ref["chars"][0]
    assert torch.equal(aux["char_seqs"].cpu().long()[:, :cs.shape[1]], cs)
    assert rel(aux["t2u_enc"].buf.view(3, -1, M), ref["t2u_enc"]) < 5e-3
    # durations: round((exp(x)-1)) flips only where the oracle's pre-rounding value sits within 0.02 of a .5 boundary
    flips = (aux["dur"].cpu().long() != ref["dur"]).nonzero()
    assert len(flips) <= 4
    # with the oracle's durations the unit sequence is reproduced up to argmax near-ties (reference tolerance: <= 1
    # differing unit, tests/common.py:42-62)
    units2, ulens2, aux2 = eng.t2u(dseq, ts, durations=ref["dur"])
    assert ulens2.tolist() == ref["unit_lens"].tolist()
    for i in range(3):
        n = int(ref["unit_lens"][i])
        assert (units2[i, :n].cpu() != ref["units"][i, :n]).sum() <= 1
        assert (units2[i, n:] == cfg.unit_pad).all()  # pad -> 1 after UnitTokenDecoder
        z = aux2["fft_out"]
        assert rel(z.data()[i, :n], ref["fft_out"][i, :n]) < 1e-2


# ------------------------------------------------------------------------------------------------ vocoder (a15)
def test_vocoder_matches_oracle_and_reference_golden(tiny):
    vc, voc, vo = tiny["vc"], tiny["voc"], tiny["vo"]
    g = torch.Generator().manual_seed(3)
    units = torch.randint(0, vc.num_embeddings, (2, 23), generator=g)
    wav = voc(units.to(dev), "spa", -1, dur_prediction=False)
    ref = vo(units, [25, 25], [45, 45])
    assert wav.shape == (2, 1, 23 * 320)
    # waveform tolerance: 5e-3 absolute on a signal of std ~0.18 in [-1,1] (fp16 activations through 5 upsampling stages)
    assert (wav.float().cpu() - ref).abs().max() < 5e-3
    d = np.load(os.path.join(G, "codehifigan_tiny.npz"))  # produced by the reference's own CodeGenerator
    w2 = voc.code_generator(torch.from_numpy(d["units"]).to(dev), d["lang"].tolist(), d["spkr"].tolist())
    assert (w2.float().cpu().numpy() - d["wav"]).__abs__().max() < 5e-3
    with pytest.raises(KeyError):
        voc(units.to(dev), "xxx", -1, dur_prediction=False)


def test_vocoder_fused_resblocks_match_conv_by_conv_path(tiny, ops):
    """Stages with 16 / 32 channels run each ResBlock as one fused kernel (resblock.cu); the same stages conv by conv
    through sb_gemm give the same waveform up to the fp16 rounding of one extra intermediate.  Lengths around the tile
    size exercise first / interior / last tiles and the zeroed halos."""
    vc, eng = tiny["vc"], tiny["voc"].code_generator
    g = torch.Generator().manual_seed(8)
    for U in (1, 7, 23):
        units = torch.randint(0, vc.num_embeddings, (3, U), generator=g).to(dev)
        assert eng.fused_resblocks
        n0 = ops.launch_count()
        a = eng(units, [25] * 3, [45] * 3)
        n_fused = ops.launch_count() - n0
        eng.fused_resblocks = False
        try:
            n0 = ops.launch_count()
            b = eng(units, [25] * 3, [45] * 3)
            n_plain = ops.launch_count() - n0
        finally:
            eng.fused_resblocks = True
        assert n_fused < n_plain  # the fused path really ran
        assert a.shape == b.shape == (3, 1, U * 320)
        assert (a - b).abs().max() < 2e-3, (U, float((a - b).abs().max()))


# ------------------------------------------------------------------------------------------------ boundary: Translator
def test_translator_predict_s2st_and_s2tt(tiny):
    from seamless_communication_b200.inference import SequenceGeneratorOptions, Translator
    tr = Translator(tiny["model"], tiny["voc"], device="cuda")
    waves = S.make_waveforms(2, 32000)
    opts = SequenceGeneratorOptions(beam_size=5, soft_max_seq_len=(1, 200), hard_max_seq_len=20)
    src = tr.fbank_batch(waves)
    texts, speech = tr.predict(src, "s2st", "spa", text_generation_opts=opts)
    ref = s2st(tiny["uo"], tiny["vo"], waves, "spa", 25, 45, hard_max=20)
    gen = Translator._last_generator
    for i in range(2):
        hyp = gen.last_text_output.hypotheses[i][0]
        if hyp[1] != ref["text_ids"][i]:
            assert abs(_oracle_score(tiny["uo"], ref["enc"][i:i + 1], hyp[1]) - ref["hyps"][i][0][0]) < 2e-2
        else:
            assert texts[i] == ref["texts"][i]
        assert speech.audio_wavs[i].shape[:2] == (1, 1)
        # BatchedSpeechOutput trimming rule (translator.py:410-420)
        n_units = speech.audio_wavs[i].shape[-1] / 320
        assert abs(n_units - len(speech.units[i])) <= 1
    assert speech.sample_rate == 16000
    # single waveform tensor input (T,) goes through convert_to_fbank + collate like the reference
    t1, s1 = tr.predict(waves[0], "s2st", "spa", text_generation_opts=opts)
    assert t1[0] == texts[0] and s1.units[0] == speech.units[0]
    t2, none = tr.predict(src, "s2tt", "spa", text_generation_opts=opts)
    assert none is None and t2 == texts
    with pytest.raises(ValueError):
        tr.predict(src, "s2st", "not_a_lang", text_generation_opts=opts)
    with pytest.raises(ValueError):
        tr.predict("hello", "t2tt", "spa")  # src_lang missing (translator.py:295-296)


def test_lanes_concurrent_batches_equal_serial(tiny):
    """parallel.LanePool: batches in flight on separate streams / host threads, each with its own search state, return
    exactly what the same batches return one at a time (the kernels are deterministic; the lanes share only the weights)."""
    from seamless_communication_b200.inference import SequenceGeneratorOptions, Translator
    from seamless_communication_b200.parallel import LanePool
    tr = Translator(tiny["model"], tiny["voc"], device="cuda")
    eng = tiny["model"].engine
    opts = SequenceGeneratorOptions(beam_size=5, soft_max_seq_len=(1, 200), hard_max_seq_len=24)
    batches = [S.make_waveforms(3, 32000, seed=100 + i).cuda() for i in range(7)]

    def step(w):
        texts, speech = tr.predict(tr.fbank_batch(w), "s2st", "spa", text_generation_opts=opts)
        return texts, speech.units, [a.float().cpu() for a in speech.audio_wavs]

    serial = [step(w) for w in batches]
    torch.cuda.synchronize()
    pool = LanePool("cuda", 3, [eng])
    try:
        pool.warm(step, batches[0])
        for _ in range(2):  # second round: every lane's graphs exist, all three lanes run concurrently from the start
            got = pool.map(step, [(w,) for w in batches])
            for (t0, u0, a0), (t1, u1, a1) in zip(serial, got):
                assert t0 == t1 and u0 == u1
                for x, y in zip(a0, a1):
                    assert torch.equal(x, y)
        assert len({k[-1] for k in eng._graphs if k[0] == 3}) >= 3  # one search state per lane
        # a failing job surfaces through its future
        with pytest.raises(ZeroDivisionError):
            pool.submit(0, lambda: 1 // 0).result()
    finally:
        pool.close()


# ------------------------------------------------------------------------------------------------ properties at full width
def test_full_width_properties_permutation_padding_determinism(small, ops):
    """M=1024 / 16 heads / 10 s audio (the BASELINE tile shapes), too big for the CPU oracle in a unit test:
    utterances are independent, so (a) permuting the batch permutes the encoder output bit-exactly, (b) running an
    utterance alone or inside a padded batch gives the same valid frames, (c) two runs are bit-identical."""
    eng = small.engine
    waves = S.make_waveforms(4, 160000, seed=9)
    ns = torch.tensor([160000, 160000, 96000, 160000], dtype=torch.int32)
    fb, frames = ops.fbank(waves.to(dev), ns.to(dev), 998)
    enc, lens, inner = eng.encode_speech(fb, frames, return_inner=True)
    M = 1024
    e, ei = enc.buf.view(4, -1, M).clone(), inner.buf.view(4, -1, M).clone()
    enc2, _ = eng.encode_speech(fb, frames)
    assert torch.equal(e, enc2.buf.view(4, -1, M))                                # (c)
    perm = [2, 0, 3, 1]
    encp, lensp = eng.encode_speech(fb[perm].contiguous(), frames[perm].contiguous())
    assert torch.equal(encp.buf.view(4, -1, M), e[perm]) and lensp.tolist() == lens[perm].tolist()  # (a)
    # (b) on the Conformer stack output: the adaptor's strided conv deliberately reads frames past `len` (the
    # reference does not mask them either, adaptor_block.py:262-277), so only the pre-adaptor states are padding-free
    n2 = int(frames[2])
    alone, la, inner_alone = eng.encode_speech(fb[2:3, :n2 + (n2 % 2)].contiguous(), frames[2:3].contiguous(), return_inner=True)
    assert int(lens[2]) == int(la[0])
    k = n2 // 2
    assert rel(inner_alone.buf.view(1, -1, M)[0, :k], ei[2, :k]) < 2e-3           # different tiling, same values
    assert torch.isfinite(e).all() and e.float().std() > 0.1


# ------------------------------------------------------------------------------------------------ BASELINE width (config 3)
def _replay_search_on_logits(eng, trace, prefix, beam, V, len_penalty=1.0):
    """Drive the INTEGER half of the search (sb_logits_topk -> sb_beam_step -> sb_step_advance, exactly as
    engine._decoder_step_select does) with the oracle's fp32 logits, step by step, for one sentence.  Returns what the
    device decided at every step: (parent beam indices, next tokens), and the finished hypotheses."""
    import ctypes as Ct
    from seamless_communication_b200 import _lib
    from seamless_communication_b200._lib import BeamDesc, check
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    ML, P, R, c = trace["max_len"], len(prefix), beam, eng.cfg
    K = min(2 * beam + 1, 16)
    ld = (V + 7) // 8 * 8
    i32 = dict(dtype=torch.int32, device=dev)
    seqs, anc = torch.zeros((R, ML), **i32), torch.arange(R, **i32)[:, None].repeat(1, ML).contiguous()
    seqs[:, :P] = torch.tensor(prefix, **i32)
    scores = torch.zeros((R, ML), device=dev)
    scores[:, :P] = trace["prefix_scores"].to(dev)
    step = torch.full((1,), P - 1, **i32)
    logits = torch.zeros((R, ld), device=dev)
    cv, ci, el = torch.empty((R, K), device=dev), torch.empty((R, K), **i32), torch.empty((R,), device=dev)
    fin = dict(count=torch.zeros(1, **i32), score=torch.full((1, beam), -math.inf, device=dev), len=torch.zeros((1, beam), **i32),
               seqs=torch.zeros((1, beam, ML), **i32), active=torch.ones(1, **i32), n_active=torch.ones(1, **i32),
               anc=torch.zeros((1, beam, ML), **i32))
    d = BeamDesc()
    d.batch, d.beam, d.max_len, d.vocab, d.K = 1, beam, ML, V, K
    d.step_ptr, d.prefix_len, d.eos_idx, d.min_len, d.len_penalty = step.data_ptr(), P, c.text_eos, 1, len_penalty
    d.cand_val, d.cand_idx, d.eos_lprob = cv.data_ptr(), ci.data_ptr(), el.data_ptr()
    d.seqs, d.scores, d.anc = seqs.data_ptr(), scores.data_ptr(), anc.data_ptr()
    d.fin_count, d.fin_score, d.fin_len = fin["count"].data_ptr(), fin["score"].data_ptr(), fin["len"].data_ptr()
    d.fin_seqs, d.active, d.n_active, d.fin_anc = fin["seqs"].data_ptr(), fin["active"].data_ptr(), fin["n_active"].data_ptr(), fin["anc"].data_ptr()
    decisions = []
    for s, lg in enumerate(trace["logits"]):
        pos = P - 1 + s
        assert seqs[:, pos].tolist() == trace["inputs"][s].tolist(), f"step {s}: device rows feed other tokens than the oracle's"
        logits[:, :V] = lg.to(dev)
        check(lib.sb_logits_topk(logits.data_ptr(), ld, R, V, c.text_pad, c.text_eos, c.text_unk, 0.0, K, cv.data_ptr(), ci.data_ptr(),
                                 el.data_ptr(), st))
        check(lib.sb_beam_step(Ct.byref(d), st))
        check(lib.sb_step_advance(step.data_ptr(), st))
        if int(fin["active"].item()) == 0:
            break
        decisions.append((anc[:, pos].tolist(), seqs[:, pos + 1].tolist()))
    n = int(fin["count"].item())
    finished = [(float(fin["score"][0, j]), fin["seqs"][0, j, :int(fin["len"][0, j])].tolist()) for j in range(n)]
    return decisions, finished


def test_search_integer_half_is_bit_exact_on_oracle_logits(tiny):
    """Given the SAME fp32 logits, top-K selection, beam bookkeeping, EOS handling and finalisation order must be
    bit-identical to the oracle's (whose mechanics are pinned against the reference's C++ generate_sequence): parents,
    tokens, finished hypotheses and their order, at every step."""
    cfg, uo, eng = tiny["cfg"], tiny["uo"], tiny["model"].engine
    waves = S.make_waveforms(2, 32000, seed=77)
    fb = torch.stack([o_fbank(w) for w in waves])
    for sentence in (0, 1):
        trace = {"sentence": sentence}
        uo.generate(fb, None, "spa", hard_max=30, output_units=False, trace=trace)
        prefix = [cfg.text_eos, tiny["toks"][0].lang_index("spa")]
        decisions, finished = _replay_search_on_logits(eng, trace, prefix, 5, cfg.text_vocab)
        assert len(decisions) == len(trace["beam_idx"])
        for s, (parents, toks) in enumerate(decisions):
            assert parents == trace["beam_idx"][s].tolist(), f"step {s}: parent beams differ"
            if s + 1 < len(trace["inputs"]):
                assert toks == trace["inputs"][s + 1].tolist(), f"step {s}: tokens differ"
        assert [f[1] for f in finished] == [f[1] for f in trace["finished"]]
        assert np.allclose([f[0] for f in finished], [f[0] for f in trace["finished"]], rtol=0, atol=1e-5)


@pytest.fixture(scope="module")
def base():
    """seamlessM4T_v2_large + vocoder_v2 with the bench's seeded random-init weights, and the fp32 oracle on the same
    state dicts (BASELINE config 3: M=1024, 16 heads, 24+24 layers, V=256 102)."""
    from seamless_communication_b200.inference import Translator
    from seamless_communication_b200.models.unity import load_unity_model
    from seamless_communication_b200.models.vocoder import load_vocoder_model
    cfg, vc = C.base_v2(), C.base_vocoder()
    sd = S.make_unity_state_dict(cfg, seed=0, dec_gain=4.0)
    vsd = S.make_vocoder_state_dict(vc, seed=1)
    toks = S.make_tokenizers(cfg)
    model = load_unity_model("seamlessM4T_v2_large", device=dev, state_dict=sd, tokenizers=toks)
    voc = load_vocoder_model("vocoder_v2", device=dev, state_dict=vsd)
    torch.set_num_threads(min(32, os.cpu_count() or 1))
    return dict(cfg=cfg, toks=toks, model=model, voc=voc, tr=Translator(model, voc, device=dev),
                uo=UnityOracle(cfg.to_dict(), sd, toks), vo=VocoderOracle(vc.to_dict(), vsd))


def test_full_width_s2st_matches_oracle(base, ops):
    """The whole S2ST path at the BASELINE width against the fp32 CPU oracle on the bench's first utterance (seed 1234,
    10 s, beam 5, hard_max_seq_len 102): encoder output, teacher-forced decoder states and logits, the search (ids equal
    or a margin-audited near tie; the integer half bit-exact on the oracle's own logits), units from the oracle's decoder
    states, waveform from the oracle's units.  Tolerances: fp16 storage / fp32 accumulation against fp32."""
    from seamless_communication_b200.ops import Seq
    cfg, uo, vo, eng, voc, tr = base["cfg"], base["uo"], base["vo"], base["model"].engine, base["voc"], base["tr"]
    M, HARD_MAX = cfg.model_dim, 102
    waves = S.make_waveforms(1, 160000, seed=1234)
    trace = {"sentence": 0}
    with torch.inference_mode():
        ref = s2st(uo, vo, waves, "spa", 25, 45, hard_max=HARD_MAX, trace=trace)
    # --- a1-a6: fbank + encoder
    src = tr.fbank_batch(waves.to(dev))
    assert (src["seqs"][0].float().cpu() - ref["fbank"][0]).abs().max() < 2e-2  # fp16 log-mel (|x| up to ~8) vs fp32
    enc, lens = eng.encode_speech(src["seqs"], None)
    err_enc = rel(enc.buf.view(1, -1, M), ref["enc"])
    assert err_enc < 5e-3, f"encoder output rel err {err_enc}"
    # --- a8/a9: teacher-forced decoder states and logits over the oracle's best hypothesis
    ids = ref["text_ids"][0]
    assert len(ids) == HARD_MAX  # random weights: no early EOS, forced EOS at max_len - 2
    ts = torch.tensor(ids[:-1])[None]
    tl = torch.tensor([len(ids) - 1], dtype=torch.int32, device=dev)
    enc_o = Seq(1, ref["enc"].shape[1], M, buf=ref["enc"].to(dev).half().reshape(-1, M).contiguous())
    dec = eng.decode_full(ts.to(dev), tl, enc_o, None)
    err_dec = rel(dec.buf.view(1, -1, M), ref["dec_out"])
    assert err_dec < 5e-3, f"decoder states rel err {err_dec}"
    lg = ops.gemm_raw(dec.buf, eng.w["text_embed"], cfg.text_vocab, out_f32=True).float().cpu()
    with torch.inference_mode():
        lg_o = uo.project(ref["dec_out"])[0]
    err_lg = (lg - lg_o).abs().max().item()
    assert err_lg < 5e-2, f"logits abs err {err_lg} (std {lg_o.std():.2f})"
    # --- a7: the search itself (device-resident, CUDA-graph replayed) from the oracle's encoder output
    prefix = [cfg.text_eos, base["toks"][0].lang_index("spa")]
    hyps = eng.beam_search(enc_o, None, prefix, beam=5, hard_max=HARD_MAX)
    assert len(hyps[0]) == len(ref["hyps"][0]) == 5
    if hyps[0][0][1] != ids:  # margin audit under the oracle's own scoring
        with torch.inference_mode():
            assert abs(_oracle_score(uo, ref["enc"], hyps[0][0][1]) - ref["hyps"][0][0][0]) < 2e-2
    assert abs(hyps[0][0][0] - ref["hyps"][0][0][0]) < 2e-2
    same_prefix = next((i for i, (a, b) in enumerate(zip(hyps[0][0][1], ids)) if a != b), len(ids))
    assert same_prefix >= 8, f"search diverges from the oracle after {same_prefix} tokens"
    # the harvested states of the winning hypothesis equal the teacher-forced pass over it
    got = eng.harvest_decoder_states([len(hyps[0][0][1]) - 1])
    if hyps[0][0][1] == ids:
        assert rel(got.buf.view(1, -1, M), ref["dec_out"]) < 5e-3
    # --- integer half, bit-exact on the oracle's logits at V = 256 102
    decisions, finished = _replay_search_on_logits(eng, trace, prefix, 5, cfg.text_vocab)
    for s, (parents, toks) in enumerate(decisions):
        assert parents == trace["beam_idx"][s].tolist(), f"step {s}: parent beams differ"
        if s + 1 < len(trace["inputs"]):
            assert toks == trace["inputs"][s + 1].tolist(), f"step {s}: tokens differ"
    assert [f[1] for f in finished] == [f[1] for f in trace["finished"]]
    # --- a11-a14: units from the oracle's decoder states (upstream near ties cannot mask a defect).  The fp16 states come
    # from a fixture of this same oracle run (tests/golden/make_golden_full_width.py): recomputed here they move by ~1e-4
    # with the host's threads and ISA, which changes their fp16 rounding and with it units at near ties
    g = np.load(os.path.join(G, "full_width_t2u_ref.npz"))
    g_dec, g_units = torch.from_numpy(g["dec_out"]), torch.from_numpy(g["units"])
    assert rel(ref["dec_out"], g_dec) < 1e-3, "the oracle's decoder states no longer match the fixture"  # fp16 rounding
    for k in ("text_seqs", "dur", "unit_lens", "units"):
        assert torch.equal(ref[k], torch.from_numpy(g[k])), f"the oracle's {k} no longer match the fixture"
    dseq = Seq(1, g_dec.shape[1], M, lens=tl, buf=g_dec.to(dev).reshape(-1, M).contiguous())
    units, ulens, _ = eng.t2u(dseq, ref["text_seqs"].to(dev), durations=ref["dur"])
    assert ulens.tolist() == ref["unit_lens"].tolist()
    n = int(ref["unit_lens"][0])
    assert n == 495  # 99 subwords x 5 characters, duration 1 each (SURVEY 8d)
    differ = (units[0, :n].cpu() != g_units[0, :n]).nonzero().flatten().tolist()
    diff = len(differ)
    assert diff <= 1, (f"{diff} unit ids differ from the oracle at {differ} "
                       f"(oracle top-2 margins {[round(float(g['unit_margins'][i]), 5) for i in differ]})")
    # --- a15/a16: waveform from the oracle's units, and the trimming rule
    wav = voc(ref["units"].to(dev), "spa", -1, dur_prediction=False)
    err_wav = (wav.float().cpu() - ref["wav_full"]).abs().max().item()
    assert err_wav < 5e-3, f"waveform abs err {err_wav}"
    print(f"full width: enc {err_enc:.1e} dec {err_dec:.1e} logits {err_lg:.1e} units diff {diff} wav {err_wav:.1e} "
          f"search common prefix {same_prefix}/{len(ids)}")


# ------------------------------------------------------------------------------------------------ a17 monotonic decoder
def test_monotonic_decoder_pchoose_and_policy_match_oracle():
    from seamless_communication_b200.models.monotonic_decoder import load_monotonic_decoder_model
    from seamless_communication_b200.streaming import MMATextDecoderPolicy
    cfg = C.tiny_v2()
    sd = S.make_monotonic_state_dict(cfg, seed=2)
    toks = S.make_tokenizers(cfg)
    model = load_monotonic_decoder_model("tiny_v2", state_dict=sd, tokenizers=toks)
    uo = UnityOracle(cfg.to_dict(), sd, toks)
    torch.manual_seed(4)
    enc = torch.randn(1, 13, cfg.model_dim).half().float()
    ids = torch.tensor([[3, toks[0].lang_index("spa"), 20, 30, 40, 50]])
    dec, pc = model.decode(ids, enc.to(dev))
    o_dec, o_pc = uo.monotonic_decoder(ids, enc)
    assert pc.shape == o_pc.shape == (cfg.dec_layers, cfg.num_heads, 6, 7)   # ceil(13/2) pooled keys
    assert rel(dec, o_dec) < 5e-3
    assert (pc.cpu() - o_pc).abs().max() < 2e-2                               # probabilities in (0,1), sigmoid(e/0.2)
    # streaming: the same READ/WRITE decisions chunk by chunk (prob compared with a margin around the threshold)
    pol = MMATextDecoderPolicy(model, "spa", max_len_a=0, max_len_b=10)
    written, o_target = [], []
    for n, fin in ((5, False), (9, False), (13, True)):
        new, finished = pol.policy(enc[:, :n].to(dev), fin)
        o_new, o_fin = uo.emma_policy(enc[:, :n], [3, toks[0].lang_index("spa")], o_target, fin, max_len=10)
        o_target += o_new
        written += new
        assert new == o_new and finished == o_fin
        if finished:
            break
    assert written == o_target and len(written) > 0


def test_streaming_s2st_chain_runs_and_reuses_source_state(tiny):
    """The SeamlessStreaming chain on the tiny models: feature extractor residual carry (every sample is framed exactly
    once), the encoder re-encode, READ/WRITE policy, unit chunks and vocoder; the per-source decoder state (cross K/V,
    key energies) is built once per encoder output, not once per token."""
    from seamless_communication_b200.models.monotonic_decoder import load_monotonic_decoder_model
    from seamless_communication_b200.streaming.pipeline import OnlineFeatureExtractor, StreamingS2ST
    cfg = tiny["cfg"]
    sd = S.make_monotonic_state_dict(cfg, seed=2)
    mono = load_monotonic_decoder_model("tiny_v2", state_dict=sd, tokenizers=tiny["toks"])
    wave = S.make_waveforms(1, 48000, seed=5)[0]
    # feature extractor: streaming frames == offline frames of the same samples (no standardisation)
    fx = OnlineFeatureExtractor(dev)
    got = [f for s0 in range(0, 48000, 5120) if (f := fx.push(wave[s0:s0 + 5120])) is not None]
    got = torch.cat(got).float().cpu()
    ref = o_fbank_raw(wave)
    assert abs(got.shape[0] - ref.shape[0]) <= 1  # 298 frames either way (the last partial window stays in the residual)
    n = min(got.shape[0], ref.shape[0])
    assert (got[:n] - ref[:n]).abs().max() < 2e-2
    st = StreamingS2ST(tiny["model"], mono, tiny["voc"], "spa", min_starting_wait_w2vbert=40, min_unit_chunk_size=5, max_len_b=12)
    ids, chunks = st.run(wave)
    assert len(st.latencies_ms) == math.ceil(48000 / 5120)
    assert len(ids) > 0 and all(0 <= i < cfg.text_vocab for i in ids)
    assert len(chunks) > 0 and all(torch.isfinite(c).all() for c in chunks)
    calls = mono.source_state_builds
    # one build per distinct encoder output (<= number of segments), although the policy ran the decoder many more times
    assert calls <= len(st.latencies_ms)
