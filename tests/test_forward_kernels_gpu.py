"""Forward-side kernels (GPU) that the end-to-end tests reach only through code agreement, each against a plain fp64 CPU computation of
the same operation:

* the exact split-fp16 GEMM (vf_tc_gemm with torch.float16 [hi | lo] operands): the call patterns of the encoder's attention blocks,
  1x1 shortcuts and the training forward at the full VQGANConfig sizes, every accumulation-chunk choice (exact_kc 4 / 3 / 2 / 1), N
  tails, the scalar epilogue, separate lo offsets for A and B, the long-K accumulation bias, the rejected calls, and whole attention /
  residual blocks of a mixed-precision VQGAN against oracle.vqgan_oracle;
* the GroupNorm statistics the GEMM epilogue accumulates for the next GroupNorm (gn_rows_per_img);
* softmax_rows with bf16 output, ragged rows and columns, padded output rows, row0 > 0 and extreme logits;
* the metric kernels image_pair_sums / ssim_u8 and the dataset resize rule on non-square images.

Exact GEMM bounds (as test_tc_conv_exact_split_fp16 for the conv): max|got - want| / max|want| < 4e-6, and an rms error at most 1.5x
that of the fp32 CUDA-core GEMM (simt_gemm) on the same problem.  The other bounds are about 5x the largest error measured on a B200
(1000 W), given in brackets in TOL."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

# largest error measured on a B200 (1000 W) in brackets
TOL = dict(exact_max=4e-6,         # max error / max|want| of the exact GEMM, the exact conv's bound [7.3e-7]
           exact_rms_ratio=1.5,    # rms error over the CUDA-core GEMM's, the exact conv's bound [1.28]
           exact_bias=5e-6,        # |mean relative error| at K = 8192 [-1.2e-6; one accumulator for all of K: -5.2e-5]
           gn_sums=1e-5,           # rtol of the fused statistics, atol 1e-2, the conv test's bounds [3.5e-4 absolute]
           gn_apply=1e-5,          # groupnorm through fused statistics vs through the statistics kernel [1.2e-6]
           softmax=1e-6,           # fp32 P, relative [1.5e-7]
           ssim=1e-6)              # absolute, per image [8e-8]
BF16_RN = 2.0 ** -8 + 1e-5   # one round-to-nearest bf16 rounding, relative, plus the fp32 error before it


@pytest.fixture(scope="module")
def L(lib):
    from viewformer_b200 import _lib
    _lib.load(require_device=True)
    return _lib


def g(seed):
    return torch.Generator().manual_seed(seed)


def report(name, got, want, atol, rtol):
    got, want = got.double().cpu(), want.double().cpu()
    err = (got - want).abs()
    tol = atol + rtol * want.abs()
    bad = int((err > tol).sum())
    print(f"[{name}] max_abs_err={err.max():.3e} max_rel_to_scale={float(err.max()) / max(float(want.abs().max()), 1e-30):.3e} "
          f"ref_scale={want.abs().mean():.3e} bad={bad}/{err.numel()}")
    if bad:
        i = int((err - tol).argmax())
        print(f"   worst at flat index {i}: got {got.reshape(-1)[i]:.9g} want {want.reshape(-1)[i]:.9g}")
    assert bad == 0, f"{name}: {bad} elements out of tolerance (max err {err.max():.3e})"


def cu(t):
    return t.float().contiguous().cuda()


def _as_f32(v):
    return float(np.float32(v))


# ----------------------------------------------------------------------------- A. exact split-fp16 GEMM
def check_exact(tag, got, simt, want):
    """The two bounds of the exact path: max error against max|want|, rms error against the fp32 CUDA-core GEMM's."""
    got, simt, want = got.double().cpu(), simt.double().cpu(), want.double().cpu()
    assert torch.isfinite(got).all(), f"{tag}: non-finite output"
    e, e32 = (got - want).abs(), (simt - want).abs()
    rel = float(e.max()) / float(want.abs().max())
    rms, rms32 = float(e.pow(2).mean().sqrt()), float(e32.pow(2).mean().sqrt())
    print(f"[{tag}] exact: max/max|y| {rel:.2e} rms {rms:.3e} | FFMA: max/max|y| {float(e32.max()) / float(want.abs().max()):.2e} "
          f"rms {rms32:.3e} | ratio {rms / max(rms32, 1e-300):.2f}")
    assert rel < TOL["exact_max"], f"{tag}: max error {rel:.3e} of max|want|"
    assert rms <= TOL["exact_rms_ratio"] * rms32 + 1e-12 * float(want.abs().max()), f"{tag}: rms {rms:.3e} vs FFMA {rms32:.3e}"


def exact_gemm(L, A32, B32, *, M, N, K, batch=1, a_rows=0, b_rows=0, a_col=0, b_col=0, alpha=1.0, bias=None, bias_mode=None,
               residual=None, ldc=None, c_bs=None, b_lo_gap=0, tag="exact gemm"):
    """C[t, m, n] = alpha * sum_k A32[t*a_rows + m, a_col + k] * B32[t*b_rows + n, b_col + k] + bias + residual[t, m, n].

    A32 / B32 are 2-D fp32 CPU tensors; batch t advances a_rows / b_rows rows (0 = an operand shared by every batch).  The exact call
    gets their split-fp16 rows [hi(C) | lo(C)] (lo_a = lo_b = C), with ``b_lo_gap`` extra fp16 columns of noise between B's halves;
    the CUDA-core GEMM gets the fp32 rows.  Both write into NaN-filled buffers of row stride ``ldc`` / batch stride ``c_bs``: the
    elements outside the [M, N] tiles must stay NaN.  Returns (exact, simt, want) as [batch, M, N]."""
    ca, cb = A32.shape[1], B32.shape[1]
    ldc = N if ldc is None else ldc
    c_bs = M * ldc if c_bs is None else c_bs
    bias_mode = (L.BIAS_N if bias is not None else L.BIAS_NONE) if bias_mode is None else bias_mode
    size = (batch - 1) * c_bs + (M - 1) * ldc + N
    view = lambda t: t.as_strided((batch, M, N), (c_bs, ldc, 1))

    a64, b64 = A32.double(), B32.double()
    want = torch.stack([a64[t * a_rows:t * a_rows + M, a_col:a_col + K] @ b64[t * b_rows:t * b_rows + N, b_col:b_col + K].T
                        for t in range(batch)]) * _as_f32(alpha)
    if bias is not None:
        want = want + (bias.double()[None, None, :] if bias_mode == L.BIAS_N else bias.double()[None, :, None])
    res_buf = None
    if residual is not None:
        want = want + residual.double()
        res_buf = torch.zeros(size)
        view(res_buf).copy_(residual)
        res_buf = res_buf.cuda()
    bias_d = cu(bias) if bias is not None else None

    As, Bs = L.split_f16x2(cu(A32)), L.split_f16x2(cu(B32))
    lo_b = cb
    if b_lo_gap:
        noise = (torch.rand(Bs.shape[0], b_lo_gap, generator=g(7)) * 4 + 1).half().cuda()
        Bs = torch.cat([Bs[:, :cb], noise, Bs[:, cb:]], 1).contiguous()
        lo_b = cb + b_lo_gap
    out = torch.full((size,), float("nan"), device="cuda")
    L.tc_gemm(As, Bs, out, M=M, N=N, K=K, lda=2 * ca, ldb=Bs.shape[1], ldc=ldc, batch=(batch, 1), a_bs=(a_rows * 2 * ca, 0),
              b_bs=(b_rows * Bs.shape[1], 0), c_bs=(c_bs, 0), alpha=alpha, bias=bias_d, bias_mode=bias_mode, residual=res_buf,
              a_off=a_col, b_off=b_col, lo_a=ca, lo_b=lo_b)
    ref = torch.full((size,), float("nan"), device="cuda")
    L.simt_gemm(cu(A32), cu(B32), ref, M=M, N=N, K=K, a_strides=(ca, 1), b_strides=(1, cb), ldc=ldc, batch=(batch, 1),
                a_bs=(a_rows * ca, 0), b_bs=(b_rows * cb, 0), c_bs=(c_bs, 0), alpha=alpha, bias=bias_d, bias_mode=bias_mode,
                residual=res_buf, a_off=a_col, b_off=b_col)
    torch.cuda.synchronize()
    out, ref = out.cpu(), ref.cpu()
    outside = torch.ones(size, dtype=torch.bool)
    view(outside).fill_(False)
    assert torch.isnan(out[outside]).all(), f"{tag}: wrote outside the output tiles"
    return view(out), view(ref), want


# encoder call patterns at the full VQGANConfig sizes: attention at c = 256 / hw = 256 (16x16, level 3) and c = 512 / hw = 64 (mid);
# nin_shortcut 128 -> 256 (level 2, 32x32) and 256 -> 512 (level 4, 8x8)
ATTN = [(2, 256, 256), (3, 512, 64)]      # (n, c, hw)


@pytest.mark.parametrize("name,M,K,N,res", [("q|k 256", 2 * 256, 256, 512, False), ("q|k 512", 3 * 64, 512, 1024, False),
                                            ("proj_out 256", 2 * 256, 256, 256, True), ("proj_out 512", 3 * 64, 512, 512, True),
                                            ("nin_shortcut 128->256", 2 * 1024, 128, 256, False),
                                            ("nin_shortcut 256->512", 3 * 64, 256, 512, False)])
def test_exact_linear_call_patterns(L, name, M, K, N, res):
    """ops.linear with an x3 Linear: rows [hi(K) | lo(K)], lo_a = lo_b = K, ldb = 2K, BIAS_N (+ the residual of proj_out)."""
    x = torch.randn(M, K, generator=g(M + K))
    w = torch.randn(N, K, generator=g(N + 1)) / K ** 0.5
    b = torch.randn(N, generator=g(N + 2)) * 0.1
    r = torch.randn(1, M, N, generator=g(N + 3)) if res else None
    check_exact(f"linear {name}", *exact_gemm(L, x, w, M=M, N=N, K=K, bias=b, residual=r, tag=name))


@pytest.mark.parametrize("n,c,hw", ATTN)
def test_exact_attention_call_patterns(L, n, c, hw):
    """The three batched GEMMs of VQGAN._attn_exact: scores (qks [n*hw, 4c], b_off = c, lo_a = lo_b = 2c, alpha = c^-0.5),
    V^T (shared weights, a_bs = 0, BIAS_M) and P.V (K = hw; one k-block at hw = 64)."""
    qk = torch.randn(n * hw, 2 * c, generator=g(c + hw)) * 2
    got, simt, want = exact_gemm(L, qk, qk, M=hw, N=hw, K=c, batch=n, a_rows=hw, b_rows=hw, b_col=c, alpha=float(int(c) ** -0.5))
    check_exact(f"scores n{n} c{c} hw{hw}", got, simt, want)

    a = torch.randn(n * hw, c, generator=g(c + hw + 1))
    wv = torch.randn(c, c, generator=g(c + hw + 2)) / c ** 0.5
    bv = torch.randn(c, generator=g(c + hw + 3)) * 0.1
    got, simt, want = exact_gemm(L, wv, a, M=c, N=hw, K=c, batch=n, a_rows=0, b_rows=hw, bias=bv, bias_mode=L.BIAS_M)
    check_exact(f"V^T n{n} c{c} hw{hw}", got, simt, want)

    p = torch.softmax(torch.randn(n * hw, hw, generator=g(c + hw + 4)) * 3, -1)
    vt = torch.randn(n * c, hw, generator=g(c + hw + 5))
    got, simt, want = exact_gemm(L, p, vt, M=hw, N=c, K=hw, batch=n, a_rows=hw, b_rows=c)
    check_exact(f"P.V n{n} c{c} hw{hw} (K/64 = {hw // 64})", got, simt, want)


def test_exact_training_forward_pattern(L):
    """train_migt's dense forward: bias + residual, K = 768 (12 k-blocks, chunks of 4), M not a multiple of 128."""
    M, K, N = 300, 768, 768
    x = torch.randn(M, K, generator=g(11))
    w = torch.randn(N, K, generator=g(12)) * 0.02
    b = torch.randn(N, generator=g(13)) * 0.02
    r = torch.randn(1, M, N, generator=g(14))
    check_exact("training forward M300 K768", *exact_gemm(L, x, w, M=M, N=N, K=K, bias=b, residual=r))


# k-blocks per pass 1..12 cover every accumulation chunk (4: 4, 8, 12; 3: 3, 6; 2: 2; 1: 1, 5); N covers BLOCK_N 64 (40, 64) and 128,
# N tails (40, 96, 320) and the scalar epilogue they take; M cycles through one partial tile, a ragged and a multi-tile count
@pytest.mark.parametrize("kb", [1, 2, 3, 4, 5, 6, 8, 12])
@pytest.mark.parametrize("N", [40, 64, 96, 128, 320])
def test_exact_gemm_branches(L, kb, N):
    K = 64 * kb
    M = (64, 77, 300)[(kb + N) % 3]
    A = torch.randn(M, K, generator=g(kb * 1000 + N)) * 1.5
    B = torch.randn(N, K, generator=g(kb * 1000 + N + 1)) / K ** 0.5
    b = torch.randn(N, generator=g(N)) if N % 64 else None
    r = torch.randn(1, M, N, generator=g(N + 5)) if kb % 2 else None
    check_exact(f"branches M{M} K{K} N{N} bias={b is not None} res={r is not None}", *exact_gemm(L, A, B, M=M, N=N, K=K, bias=b, residual=r))


def test_exact_gemm_unaligned_ldc(L):
    """ldc % 4 != 0: the vectorised epilogue is off (vec_ok false), every element goes through the scalar path."""
    M, K, N = 77, 192, 128
    A, B = torch.randn(M, K, generator=g(21)), torch.randn(N, K, generator=g(22)) / K ** 0.5
    r = torch.randn(1, M, N, generator=g(23))
    check_exact("ldc 131", *exact_gemm(L, A, B, M=M, N=N, K=K, bias=torch.randn(N, generator=g(24)), residual=r, ldc=131))


@pytest.mark.parametrize("kb", [3, 4])
def test_exact_gemm_separate_lo_offsets(L, kb):
    """lo_a != lo_b: B's lo half starts 64 columns after its hi half ends (noise in between), A's directly after."""
    K, M, N = 64 * kb, 300, 96
    A, B = torch.randn(M, K, generator=g(31)), torch.randn(N, K, generator=g(32)) / K ** 0.5
    check_exact(f"lo_b = K + 64, K{K}", *exact_gemm(L, A, B, M=M, N=N, K=K, b_lo_gap=64))


def test_exact_gemm_long_k_accumulation_bias(L):
    """K = 8192 of positive products: a single fp32 tensor-core accumulator loses low bits at every addition and drifts to about
    -2.7e-5 relative at K = 6912 (profiles/r02_acc_rounding_probe.txt; -5.2e-5 here); the accumulation in chunks of 4 k-blocks
    (256 products, summed with RN adds) keeps the drift of each chunk small."""
    M = N = 128
    K = 8192
    A = torch.rand(M, K, generator=g(41)) * 0.75 + 0.25
    B = torch.rand(N, K, generator=g(42)) * 0.75 + 0.25
    got, simt, want = exact_gemm(L, A, B, M=M, N=N, K=K)
    bias = float(((got.double() - want) / want).mean())
    print(f"[long K] mean relative error {bias:.3e} (CUDA-core GEMM: {float(((simt.double() - want) / want).mean()):.3e})")
    assert abs(bias) < TOL["exact_bias"]
    check_exact("long K 8192", got, simt, want)


def test_exact_gemm_rejected_calls(L):
    """Calls the exact GEMM cannot serve raise before anything is launched: the output keeps its fill."""
    M, N, K = 128, 128, 128
    A = L.split_f16x2(torch.randn(M, K, generator=g(51)).cuda())
    B = L.split_f16x2(torch.randn(N, K, generator=g(52)).cuda())
    out = torch.full((M, N), float("nan"), device="cuda")
    out16 = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16)
    kw = dict(M=M, N=N, K=K, lda=2 * K, ldb=2 * K, ldc=N)
    with pytest.raises(L.LibraryError):                    # bf16 output
        L.tc_gemm(A, B, out16, **kw)
    with pytest.raises(L.LibraryError):                    # K % 64 != 0
        L.tc_gemm(A, B, out, **dict(kw, K=96), lo_a=K, lo_b=K)
    with pytest.raises(L.LibraryError):                    # lo half overlapping the hi half
        L.tc_gemm(A, B, out, **kw, lo_a=K - 64, lo_b=K)
    with pytest.raises(L.LibraryError):                    # causal mask
        L.tc_gemm(A, B, out, **kw, causal_block=64)
    torch.cuda.synchronize()
    assert torch.isnan(out.cpu()).all() and torch.isnan(out16.float().cpu()).all()


@pytest.fixture(scope="module")
def vqgan_pair(L):
    """A full-size VQGAN in the benchmarked mixed precision (exact tensor-core encoder) and in fp32, on the same synthetic weights."""
    from oracle import synth
    from viewformer_b200 import VQGAN
    from viewformer_b200.config import VQGANConfig
    cfg = VQGANConfig()
    sd = synth.make_vqgan_state_dict(cfg, 5)
    mixed = VQGAN(cfg, precision="mixed").load_state_dict(sd)
    fp32 = VQGAN(cfg, precision="fp32").load_state_dict(sd)
    return sd, mixed, fp32


@pytest.mark.parametrize("block,prefix,n,hw,c", [("mida", "encoder.mid.attn_1", 2, 8, 512),
                                                 ("level3 attn", "encoder.down.3.attn.0", 2, 16, 256),
                                                 ("level2 block0", "encoder.down.2.block.0", 2, 32, 128)])
def test_exact_encoder_blocks_against_oracle(L, vqgan_pair, block, prefix, n, hw, c):
    """VQGAN._attn / _resblock of the mixed model (every GEMM and conv on the exact path) against oracle.vqgan_oracle in fp64; the rms
    bound compares with the same block of the fp32 CUDA-core model."""
    from oracle import vqgan_oracle as vo
    sd, mixed, fp32 = vqgan_pair
    sd64 = {k: v.double() for k, v in sd.items() if k.startswith(prefix)}
    x = torch.randn(n, hw, hw, c, generator=g(hw + c)) * 2 + 0.3
    xc = x.cuda()

    def run(m):
        w = m._w["enc"]
        if block == "mida":
            return m._attn(w["mida"], xc)
        if block == "level3 attn":
            return m._attn(w["levels"][3]["attns"][0], xc)
        return m._resblock(w["levels"][2]["blocks"][0], xc)

    with torch.no_grad():
        got, ref = run(mixed), run(fp32)
        torch.cuda.synchronize()
        fn = vo.attnblock if ".attn" in prefix else vo.resblock
        want = fn(sd64, prefix, x.permute(0, 3, 1, 2).double()).permute(0, 2, 3, 1)
    assert got.shape == want.shape
    check_exact(f"block {block} ({prefix})", got, ref, want)


# ----------------------------------------------------------------------------- B. GEMM-mode fused GroupNorm statistics
@pytest.mark.parametrize("exact", [False, True])
@pytest.mark.parametrize("n,hw,c", [(3, 64, 512), (2, 256, 256), (5, 32, 128)])
def test_gemm_fused_groupnorm_statistics(L, n, hw, c, exact):
    """proj_out of an attention block: out = o @ W^T + b + x with the GroupNorm(32) statistics of `out` accumulated by the epilogue."""
    M = n * hw
    o = torch.randn(M, c, generator=g(c + hw)) * 1.5
    w = torch.randn(c, c, generator=g(c + 1)) / c ** 0.5
    b = torch.randn(c, generator=g(c + 2)) * 0.3
    x = torch.randn(M, c, generator=g(c + 3)) + 0.5
    if exact:
        A, B, kw = L.split_f16x2(cu(o)), L.split_f16x2(cu(w)), dict(lda=2 * c, ldb=2 * c, lo_a=c, lo_b=c)
    else:
        A, B, kw = cu(o).bfloat16(), cu(w).bfloat16(), dict(lda=c, ldb=c)
    out = torch.empty((M, c), device="cuda")
    L.tc_gemm(A, B, out, M=M, N=c, K=c, ldc=c, bias=cu(b), bias_mode=L.BIAS_N, residual=cu(x), gn_rows_per_img=hw, **kw)
    torch.cuda.synchronize()
    assert hasattr(out, "_gn_sums"), "fusion expected for this shape"
    tag = f"gemm gn sums n{n} hw{hw} c{c} {'exact' if exact else 'bf16'}"
    od = out.double().cpu().reshape(n, hw, 32, c // 32)
    want = torch.stack([od.sum((1, 3)), (od * od).sum((1, 3))], -1)
    report(tag, out._gn_sums[0].cpu(), want, 1e-2, TOL["gn_sums"])
    ga, be = (1 + 0.1 * torch.randn(c, generator=g(c + 4))).cuda(), (0.1 * torch.randn(c, generator=g(c + 5))).cuda()
    out4 = out.reshape(n, hw, 1, c)
    out4._gn_sums = out._gn_sums
    y_fused = L.groupnorm(out4, ga, be, swish=True, out_dtype=torch.float32)
    y_plain = L.groupnorm(out4.clone(), ga, be, swish=True, out_dtype=torch.float32)
    report(tag + " -> groupnorm", y_fused, y_plain, TOL["gn_apply"], TOL["gn_apply"])


@pytest.mark.parametrize("exact", [False, True])
def test_gemm_groupnorm_statistics_refused_shape(L, exact):
    """c = 64 (2 channels per group): gn_fusable refuses, the call attaches no statistics and writes what a plain call writes."""
    n, hw, c = 2, 64, 64
    assert not L.gn_fusable(c, 32, n * hw, hw, c)
    M = n * hw
    o, w = torch.randn(M, c, generator=g(61)), torch.randn(c, c, generator=g(62)) / 8
    x = cu(torch.randn(M, c, generator=g(63)))
    if exact:
        A, B, kw = L.split_f16x2(cu(o)), L.split_f16x2(cu(w)), dict(lda=2 * c, ldb=2 * c, lo_a=c, lo_b=c)
    else:
        A, B, kw = cu(o).bfloat16(), cu(w).bfloat16(), dict(lda=c, ldb=c)
    outs = []
    for rpi in (hw, 0):
        out = torch.empty((M, c), device="cuda")
        L.tc_gemm(A, B, out, M=M, N=c, K=c, ldc=c, residual=x, gn_rows_per_img=rpi, **kw)
        outs.append(out)
    torch.cuda.synchronize()
    assert not hasattr(outs[0], "_gn_sums")
    assert torch.equal(outs[0], outs[1])


# ----------------------------------------------------------------------------- C. softmax_rows
def _softmax64(x):
    return torch.softmax(x.double(), -1)


@pytest.mark.parametrize("rows,cols", [(37, 77), (101, 256), (13, 1024), (64 * 3 + 5, 64)])
def test_softmax_rows_bf16_output(L, rows, cols):
    """bf16 P (VQGAN bf16 attention, the unfused MIGT paths): within one bf16 rounding of the fp64 softmax."""
    x = torch.randn(rows, cols, generator=g(rows + cols)) * 4
    p = torch.empty(rows, cols, dtype=torch.bfloat16, device="cuda")
    L.softmax_rows(cu(x), p, rows_total=rows, rows_per_batch=rows, cols=cols, ld_in=cols, ld_out=cols)
    torch.cuda.synchronize()
    want = _softmax64(x)
    # round-to-nearest bf16 (8 significant bits): |got - want| <= 2^-8 |want| (half an ulp) + the fp32 error before rounding
    report(f"softmax bf16 {rows}x{cols}", p.float(), want, 1e-30, BF16_RN)


@pytest.mark.parametrize("cols", [64, 77, 256, 1024])
def test_softmax_rows_unmasked(L, cols):
    """mask 0 at the VQGAN attention widths (hw = 64 / 256) and ragged ones; rows_total not a multiple of the 8 rows of a block,
    several batches of rows."""
    rows, rpb = 3 * 29, 29
    x = torch.randn(rows, cols, generator=g(cols)) * 3
    p = torch.empty(rows, cols, device="cuda")
    L.softmax_rows(cu(x), p, rows_total=rows, rows_per_batch=rpb, cols=cols, ld_in=cols, ld_out=cols)
    torch.cuda.synchronize()
    want = _softmax64(x)
    report(f"softmax mask0 cols{cols}", p, want, TOL["softmax"] * float(want.max()), TOL["softmax"])


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_softmax_rows_padded_rows(L, dtype):
    """ld_in / ld_out > cols: the padding columns of P are left untouched (pre-filled NaN stays NaN)."""
    rows, cols, ld_in, ld_out = 45, 77, 96, 88
    x = torch.randn(rows, ld_in, generator=g(71)) * 2
    x[:, cols:] = 1e4                            # padding of the input must not enter the row maximum
    p = torch.full((rows, ld_out), float("nan"), dtype=dtype, device="cuda")
    L.softmax_rows(cu(x), p, rows_total=rows, rows_per_batch=rows, cols=cols, ld_in=ld_in, ld_out=ld_out)
    torch.cuda.synchronize()
    pc = p.float().cpu()
    assert torch.isnan(pc[:, cols:]).all(), "padding columns of P were written"
    want = _softmax64(x[:, :cols])
    rtol = TOL["softmax"] if dtype == torch.float32 else BF16_RN
    report(f"softmax padded {dtype}", pc[:, :cols], want, TOL["softmax"] * float(want.max()) if dtype == torch.float32 else 1e-30, rtol)


def test_softmax_rows_row0_matches_full_call(L):
    """row0 > 0 with the block-causal mask (the KV-cache step's query rows) == the matching rows of a row0 = 0 call."""
    S, blk, r0 = 256, 64, 100
    x = cu(torch.randn(S, S, generator=g(81)) * 3)
    full = torch.empty(S, S, device="cuda")
    L.softmax_rows(x, full, rows_total=S, rows_per_batch=S, cols=S, ld_in=S, ld_out=S, mask_mode=1, block=blk)
    part = torch.empty(S - r0, S, device="cuda")
    L.softmax_rows(x[r0:].contiguous(), part, rows_total=S - r0, rows_per_batch=S - r0, cols=S, ld_in=S, ld_out=S, mask_mode=1,
                   block=blk, row0=r0)
    torch.cuda.synchronize()
    assert torch.equal(part.cpu(), full[r0:].cpu())
    view = torch.arange(S) // blk
    m = (view[:, None] >= view[None, :]).double()
    want = _softmax64(x.cpu().double() * m - 1e4 * (1 - m))
    report("softmax row0 causal", part, want[r0:], TOL["softmax"], TOL["softmax"])


def test_softmax_rows_extreme_logits(L):
    """Logits around +-1e3: finite, rows sum to 1, equal to the fp64 softmax."""
    rows, cols = 19, 256
    x = torch.randn(rows, cols, generator=g(91)) * 5
    x[::2] += 1e3
    x[1::2] -= 1e3
    x[3, 7] = 1.02e3                             # one dominant entry
    p = torch.empty(rows, cols, device="cuda")
    L.softmax_rows(cu(x), p, rows_total=rows, rows_per_batch=rows, cols=cols, ld_in=cols, ld_out=cols)
    torch.cuda.synchronize()
    pc = p.cpu()
    assert torch.isfinite(pc).all()
    s = pc.double().sum(-1)
    print(f"[softmax +-1e3] max |row sum - 1| {float((s - 1).abs().max()):.2e}")
    assert float((s - 1).abs().max()) < 1e-5
    report("softmax +-1e3", pc, _softmax64(x), TOL["softmax"], TOL["softmax"])


# ----------------------------------------------------------------------------- D. metric kernels and resize
def _pair_sums_np(a, b):
    per = int(np.prod(a.shape[1:]))
    d = a.reshape(a.shape[0], per).astype(np.int64) - b.reshape(b.shape[0], per).astype(np.int64)
    return np.stack([np.abs(d).sum(1), (d * d).sum(1)], 1)


@pytest.mark.parametrize("shape", [(5, 7, 11, 3),          # 231 per image: less than one pass of the 256 threads
                                   (3, 33, 17, 3),         # ragged, several passes
                                   (1, 1024, 1024, 3),     # 3 Mi per image
                                   (0, 8, 8, 3)])          # empty batch
def test_image_pair_sums_exact(L, shape):
    a = torch.randint(0, 256, shape, generator=g(sum(shape)), dtype=torch.uint8)
    b = torch.randint(0, 256, shape, generator=g(sum(shape) + 1), dtype=torch.uint8)
    got = L.image_pair_sums(a.cuda(), b.cuda()).cpu().numpy()
    assert got.shape == (shape[0], 2)
    assert np.array_equal(got, _pair_sums_np(a.numpy(), b.numpy()))


def test_image_pair_sums_extreme(L):
    """0 against 255 everywhere on a large image: sum (a-b)^2 = 65025 * 3 Mi, beyond 32 bits."""
    shape = (2, 1024, 1024, 3)
    a = torch.zeros(shape, dtype=torch.uint8)
    b = torch.full(shape, 255, dtype=torch.uint8)
    got = L.image_pair_sums(a.cuda(), b.cuda()).cpu().numpy()
    n = 1024 * 1024 * 3
    assert np.array_equal(got, np.array([[255 * n, 65025 * n]] * 2, dtype=np.int64))
    assert np.array_equal(L.image_pair_sums(b.cuda(), a.cuda()).cpu().numpy(), got)


def ssim_ref_k(X, Y, k1=0.01, k2=0.03):
    """utils/metrics.py:17-73 restated in fp64 with K1 / K2 (data range 1): depthwise 7x7 box filter, VALID, sample covariance
    (49/48), C1 = K1^2, C2 = K2^2, mean over (H-6) x (W-6) x C.  X, Y uint8 NHWC."""
    X, Y = X.permute(0, 3, 1, 2).double() / 255, Y.permute(0, 3, 1, 2).double() / 255
    c = X.shape[1]
    k = torch.full((c, 1, 7, 7), 1 / 49.0, dtype=torch.float64)
    f = lambda t: F.conv2d(t, k, groups=c)
    ux, uy, uxx, uyy, uxy = f(X), f(Y), f(X * X), f(Y * Y), f(X * Y)
    cn = 49 / 48
    vx, vy, vxy = cn * (uxx - ux * ux), cn * (uyy - uy * uy), cn * (uxy - ux * uy)
    C1, C2 = k1 ** 2, k2 ** 2
    S = ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux ** 2 + uy ** 2 + C1) * (vx + vy + C2))
    return S.mean((1, 2, 3))


def _ssim_images(content, shape, seed):
    gen = g(seed)
    if content == "random":
        a = torch.randint(0, 256, shape, generator=gen, dtype=torch.uint8)
        return a, torch.randint(0, 256, shape, generator=gen, dtype=torch.uint8)
    if content == "identical":
        a = torch.randint(0, 256, shape, generator=gen, dtype=torch.uint8)
        return a, a.clone()
    if content == "bright flat":                  # 250 +- 1 against 250 +- 1
        return (torch.randint(249, 252, shape, generator=gen, dtype=torch.uint8),
                torch.randint(249, 252, shape, generator=gen, dtype=torch.uint8))
    if content == "bright flat vs 250|251":       # flat 250 against a 250 / 251 pattern
        return torch.full(shape, 250, dtype=torch.uint8), torch.randint(250, 252, shape, generator=gen, dtype=torch.uint8)
    assert content == "dark flat"
    return (torch.randint(0, 3, shape, generator=gen, dtype=torch.uint8), torch.randint(0, 3, shape, generator=gen, dtype=torch.uint8))


@pytest.mark.parametrize("k1,k2", [(0.01, 0.03), (1.0, 0.03), (0.01, 0.1), (1.0, 0.1)])
@pytest.mark.parametrize("shape", [(2, 7, 7, 3),         # a single window
                                   (2, 7, 300, 1),       # one window row
                                   (2, 300, 260, 3),     # more window positions than the 64 x 256 threads of the capped grid
                                   (9, 20, 23, 3)])
@pytest.mark.parametrize("content", ["random", "identical", "bright flat", "bright flat vs 250|251", "dark flat"])
def test_ssim_u8(L, shape, content, k1, k2):
    a, b = _ssim_images(content, shape, seed=shape[1] * 7 + shape[2] + len(content))
    got = L.ssim_u8(a.cuda(), b.cuda(), k1=k1, k2=k2).cpu()
    want = ssim_ref_k(a, b, k1, k2)
    err = float((got - want).abs().max())
    print(f"[ssim {content} {tuple(shape)} K1={k1} K2={k2}] max abs err {err:.2e} (ssim {float(want.min()):.6f}..{float(want.max()):.6f})")
    assert err < TOL["ssim"]
    if content == "identical":
        assert float((got - 1).abs().max()) < TOL["ssim"]
    if shape[0] > 1:                               # each image's value is its own: a permuted batch permutes the result
        perm = torch.randperm(shape[0], generator=g(3))
        got_p = L.ssim_u8(a[perm].contiguous().cuda(), b[perm].contiguous().cuda(), k1=k1, k2=k2).cpu()
        assert float((got_p - got[perm]).abs().max()) < 1e-12


def test_ssim_u8_rejects(L):
    a = torch.zeros(1, 6, 10, 3, dtype=torch.uint8, device="cuda")
    with pytest.raises(L.LibraryError):
        L.ssim_u8(a, a)
    a = torch.zeros(1, 10, 6, 3, dtype=torch.uint8, device="cuda")
    with pytest.raises(L.LibraryError):
        L.ssim_u8(a, a)
    a = torch.zeros(1, 8, 8, 3, dtype=torch.uint8, device="cuda")
    for k1 in (-0.1, 2e3):
        with pytest.raises(L.LibraryError):
            L.ssim_u8(a, a, k1=k1)


def resize_ref(x_u8_nhwc, size, method=None):
    """data/_common.py:19-62 restated (torch CPU): resize() returns the NHWC images unchanged when W == size, resize_th() the NCHW ones
    when H == size; otherwise the method is nearest when size > H, else bilinear (align_corners=False), to size x size."""
    if x_u8_nhwc.shape[-2] == size:
        return x_u8_nhwc
    x = x_u8_nhwc.permute(0, 3, 1, 2)
    if x.shape[-2] == size:
        return x_u8_nhwc
    x = x.to(torch.float32) / 255.0
    if method is None:
        method = "nearest" if size > x.shape[-2] else "bilinear"
    if method == "nearest":
        y = F.interpolate(x, (size, size), mode="nearest")
    else:
        y = F.interpolate(x, (size, size), mode="bilinear", align_corners=False)
    return (y.clamp_(0, 1) * 255.0).to(torch.uint8).permute(0, 2, 3, 1).contiguous()


@pytest.mark.parametrize("C", [1, 3])
@pytest.mark.parametrize("method", [None, "nearest", "bilinear"])
@pytest.mark.parametrize("H,W,size", [(200, 128, 128),     # W == size: unchanged
                                      (128, 100, 128),     # H == size: unchanged
                                      (100, 200, 128),     # growing by H (nearest), shrinking by W
                                      (200, 100, 128),     # shrinking by H (bilinear), growing by W
                                      (96, 160, 64), (50, 37, 48)])
def test_resize_u8_non_square(L, H, W, size, method, C):
    x = torch.randint(0, 256, (2, H, W, C), generator=g(H * W + C), dtype=torch.uint8)
    want = resize_ref(x, size, method)
    got = L.resize_u8(x.cuda(), size, method).cpu()
    assert got.shape == want.shape, (got.shape, want.shape)
    if size in (H, W):
        assert torch.equal(got, x)
        return
    d = (got.int() - want.int()).abs()
    print(f"[resize {H}x{W}x{C} -> {size} {method}] out {tuple(got.shape[1:3])} exact {float((d == 0).float().mean()):.5f}, "
          f"max diff {int(d.max())}")
    if (method or ("nearest" if size > H else "bilinear")) == "nearest":
        assert torch.equal(got, want)
    else:
        # bilinear weights of exactly 1/4 and 3/4 (scale 1.5 in H, 2.5 in W) put many values exactly on an integer before the
        # truncation to uint8, where the kernel's and torch's fp32 summation orders differ by one LSB: 98.7 % exact measured at
        # 96x160 -> 64, and the same on square 96x96 -> 64 images
        assert int(d.max()) <= 1 and float((d == 0).float().mean()) > 0.98


def test_generate_rejects_images_that_stay_non_square(L):
    """generate(): 32x48 images for a 32x32 codebook stay 32x48 under the dataset rule; the call says so instead of encoding them."""
    from oracle import synth
    from viewformer_b200 import VQGAN, MIGT, generate_batch_predictions
    from viewformer_b200.config import VQGANConfig, MIGTConfig
    vcfg = VQGANConfig(ch=64, ch_mult=[1, 2, 2, 2], attn_resolutions=[8], image_size=32, embed_dim=64, z_channels=64,
                       n_embed=256, num_res_blocks=1)
    tcfg = MIGTConfig(n_layer=2, n_head=4, d_model=128, sequence_size=4, n_embeddings=vcfg.n_embed, token_image_size=4)
    cb = VQGAN(vcfg, precision="fp32").load_state_dict(synth.make_vqgan_state_dict(vcfg, 1))
    tr = MIGT(tcfg, precision="fp32").load_state_dict(synth.make_migt_state_dict(tcfg, 2))
    images = torch.randint(0, 256, (2, 3, 32, 48, 3), generator=g(5), dtype=torch.uint8)
    with pytest.raises(ValueError, match="resize"):
        generate_batch_predictions(tr, cb, images, synth.make_cameras(2, 3, seed=6))
