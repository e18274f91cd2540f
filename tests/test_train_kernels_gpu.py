"""Training-step kernels (GPU), one entry point at a time: every backward / loss / optimizer kernel of libvf_b200 through its
viewformer_b200._lib wrapper against a plain fp64 CPU computation of the same operation (torch autograd for the gradient kernels), at
the shapes where the kernels change their work split: one pixel lane per block, chunked grids, grid-stride loops past the 148*16*256
launch cap, ragged rows and channel tiles.

Outputs that the kernels accumulate with atomics (norm dgamma / dbeta, conv_wgrad's dW, col_sums, migt_embed_bwd, the tensor-core weight
gradients with accumulate=True) are pre-filled with random values and compared with prefill + gradient: the trainers rely on it when a
shared parameter collects its gradient over several streams.

Tolerances: the fp32 kernels are held to atol = T * max|want| (max|gradient| for accumulated outputs), rtol = T, with T per kernel in
TOL below: about 5x the largest error measured on a B200 over all cases of the kernel, all well inside the reference project's single-layer
bound of 1e-5 (viewformer/utils/testing.py:98).  The exact split-fp16 weight-gradient GEMM is held to max error / max|dW| < 5e-6 like
test_conv_weight_gradient_on_tensor_cores; the fp64 accumulators (sumsq, the L1 loss sum) to 1e-10 relative; dropout is bit-exact."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

# largest error / max|want| measured on a B200 (1000 W) in brackets
TOL = dict(gn_bwd=5e-6,           # 8.8e-7 (dgamma at 128x128)
           ln_bwd=1.5e-6,         # 2.8e-7
           softmax_bwd=1.5e-6,    # 2.8e-7
           cross_entropy=1e-6,    # 1.3e-7 (rows, grad, row_mean)
           row_mean=1e-6,         # 1.3e-7
           pose_loss=1e-6,        # 1.5e-7
           gelu=5e-7,             # 9.4e-8
           embed_bwd=2.5e-6,      # 4.5e-7
           lincomb3=5e-7,         # 9.4e-8
           sumpool2x2=5e-7,       # 8.9e-8
           adam=2e-6,             # 3e-7 (m, v)
           conv_wgrad=3e-6,       # 5.2e-7
           conv_dgrad_s2=6e-6,    # 1.2e-6
           col_sums=7e-6,         # 1.3e-6 (3 * 2^20 rows)
           vq_commit=5e-7,        # 7e-8
           wgrad_paths=4e-6)      # 7.6e-7: dense_wgrad_tc against conv_wgrad
WGRAD_TC_TOL = 5e-6     # exact split-fp16 GEMM: max error / max|dW|
F64_TOL = 1e-10         # double-precision accumulators
GRID_CAP = 148 * 16 * 256   # elements covered by one pass of the capped elementwise grids


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


def amax(t):
    return float(t.double().abs().max())


def cu(t):
    return t.float().contiguous().cuda()


def _as_f32(v):
    """A Python float as the fp32 value a kernel argument carries (1 - 0.999f differs from 0.001 by 1.3e-5 relative)."""
    return float(np.float32(v))


# ----------------------------------------------------------------------------- normalisation backward
GN_SHAPES = [(3, 32, 8, 8),          # one channel per group
             (3, 64, 5, 7),          # a thread's channel quad spans two groups
             (1, 128, 1, 3), (3, 128, 1, 3), (3, 128, 16, 16),
             (1, 128, 128, 128),     # many pixel chunks: the ppb halving loop stops at its start value
             (3, 512, 4, 4),
             (1, 1024, 6, 6), (3, 1024, 3, 5)]      # C = 1024: one pixel lane per 256-thread block


@pytest.mark.parametrize("swish", [False, True])
@pytest.mark.parametrize("add", [False, True])
@pytest.mark.parametrize("N,C,H,W", GN_SHAPES)
def test_groupnorm_bwd(L, N, C, H, W, swish, add):
    seed = N * 7 + C + H * 31 + W
    x = torch.randn(N, H, W, C, generator=g(seed)) * 2 + 0.5
    dout = torch.randn(N, H, W, C, generator=g(seed + 1))
    ga, be = 1 + 0.2 * torch.randn(C, generator=g(seed + 2)), 0.3 * torch.randn(C, generator=g(seed + 3))
    res = torch.randn(N, H, W, C, generator=g(seed + 4)) if add else None
    pre_g, pre_b = torch.randn(C, generator=g(seed + 5)), torch.randn(C, generator=g(seed + 6))
    xd = x.permute(0, 3, 1, 2).double().requires_grad_(True)
    gd, bd = ga.double().requires_grad_(True), be.double().requires_grad_(True)
    y = F.group_norm(xd, 32, gd, bd, eps=1e-6)
    if swish:
        y = y * torch.sigmoid(y)
    y.backward(dout.permute(0, 3, 1, 2).double())
    want_dx = xd.grad.permute(0, 2, 3, 1) + (res.double() if add else 0)

    xc = cu(x)
    mr = L.gn_mean_rstd(xc)
    dgamma, dbeta = cu(pre_g), cu(pre_b)
    dx = L.groupnorm_bwd(xc, cu(dout), mr, cu(ga), cu(be), dgamma, dbeta, swish=swish, add=cu(res) if add else None)
    torch.cuda.synchronize()
    tag = f"gn_bwd N={N} C={C} {H}x{W} swish={int(swish)} add={int(add)}"
    report(tag + " dx", dx, want_dx, TOL["gn_bwd"] * amax(want_dx), TOL["gn_bwd"])
    report(tag + " dgamma", dgamma, pre_g.double() + gd.grad, TOL["gn_bwd"] * amax(gd.grad), TOL["gn_bwd"])
    report(tag + " dbeta", dbeta, pre_b.double() + bd.grad, TOL["gn_bwd"] * amax(bd.grad), TOL["gn_bwd"])


def test_groupnorm_bwd_rejects_unsupported_channels(L):
    """C = 96: the channel quads do not tile a 256-thread block; the host check refuses before any launch."""
    x = torch.zeros(1, 4, 4, 96, device="cuda")
    mr = torch.zeros(1, 32, 2, device="cuda")
    p = torch.zeros(96, device="cuda")
    with pytest.raises(L.LibraryError, match="unsupported C=96"):
        L.groupnorm_bwd(x, x, mr, p, p, p.clone(), p.clone(), swish=False)


@pytest.mark.parametrize("add", [False, True])
@pytest.mark.parametrize("rows", [1, 7, 8 * 37 + 3])
@pytest.mark.parametrize("D", [100, 128, 768, 1024, 4096])
def test_layernorm_bwd(L, D, rows, add):
    seed = D + rows
    x = torch.randn(rows, D, generator=g(seed)) * 3 + 5          # mean-shifted rows
    dy = torch.randn(rows, D, generator=g(seed + 1))
    ga, be = 1 + 0.2 * torch.randn(D, generator=g(seed + 2)), 0.1 * torch.randn(D, generator=g(seed + 3))
    res = torch.randn(rows, D, generator=g(seed + 4)) if add else None
    pre_g, pre_b = torch.randn(D, generator=g(seed + 5)), torch.randn(D, generator=g(seed + 6))
    xd = x.double().requires_grad_(True)
    gd, bd = ga.double().requires_grad_(True), be.double().requires_grad_(True)
    F.layer_norm(xd, (D,), gd, bd, eps=1e-5).backward(dy.double())
    want_dx = xd.grad + (res.double() if add else 0)

    dgamma, dbeta = cu(pre_g), cu(pre_b)
    dx = L.layernorm_bwd(cu(x), cu(dy), cu(ga), dgamma, dbeta, eps=1e-5, add=cu(res) if add else None)
    torch.cuda.synchronize()
    tag = f"ln_bwd D={D} rows={rows} add={int(add)}"
    report(tag + " dx", dx, want_dx, TOL["ln_bwd"] * amax(want_dx), TOL["ln_bwd"])
    report(tag + " dgamma", dgamma, pre_g.double() + gd.grad, TOL["ln_bwd"] * amax(gd.grad), TOL["ln_bwd"])
    report(tag + " dbeta", dbeta, pre_b.double() + bd.grad, TOL["ln_bwd"] * amax(bd.grad), TOL["ln_bwd"])


def test_layernorm_bwd_rejects_wide_rows(L):
    x = torch.zeros(2, 4097, device="cuda")
    p = torch.zeros(4097, device="cuda")
    with pytest.raises(L.LibraryError, match="vf_layernorm_bwd"):
        L.layernorm_bwd(x, x, p, p.clone(), p.clone())


# ----------------------------------------------------------------------------- softmax / losses
@pytest.mark.parametrize("cols", [64, 192, 384, 1000])
def test_softmax_bwd_rows(L, cols):
    rows = cols + 5                                              # not a multiple of the 8 rows of a block
    blk = 16
    r = torch.arange(rows).remainder(cols).reshape(-1, 1)
    allowed = torch.arange(cols).reshape(1, -1) // blk <= r // blk          # block-causal: later blocks are masked out
    s = (torch.randn(rows, cols, generator=g(cols)) * 3).double().masked_fill(~allowed, float("-inf")).requires_grad_(True)
    P = torch.softmax(s, -1)
    dP = torch.randn(rows, cols, generator=g(cols + 1))
    P.backward(dP.double())
    want = s.grad
    got = L.softmax_bwd_rows(cu(P.detach()), cu(dP))
    torch.cuda.synchronize()
    report(f"softmax_bwd cols={cols} rows={rows}", got, want, TOL["softmax_bwd"] * amax(want), TOL["softmax_bwd"])
    assert bool((got.cpu()[~allowed] == 0).all()), "masked probabilities must give exactly zero gradient"


@pytest.mark.parametrize("smoothing", [0.0, 0.1])
@pytest.mark.parametrize("cols", [33, 1000, 1024])
def test_cross_entropy_rows_grad_and_row_mean(L, cols, smoothing):
    B, S, start = 7, 11, 3
    rows = B * S
    logits = (torch.rand(rows, cols, generator=g(cols)) * 2 - 1) * 30
    labels = torch.randint(0, cols, (rows,), generator=g(cols + 1), dtype=torch.int32)
    labels[0], labels[1] = 0, cols - 1
    w = torch.rand(rows, generator=g(cols + 2)) + 0.1
    w[::5] = 0.0
    ld = logits.double().requires_grad_(True)
    ce = F.cross_entropy(ld, labels.long(), label_smoothing=smoothing, reduction="none")
    (ce * w.double()).sum().backward()

    lc, labc = cu(logits), labels.cuda()
    got_ce = L.cross_entropy_rows(lc, labc, smoothing)
    got_d = L.cross_entropy_grad(lc, labc, cu(w), smoothing)
    got_m = L.row_mean(got_ce.reshape(B, S), start)
    torch.cuda.synchronize()
    tag = f"cross_entropy cols={cols} s={smoothing}"
    report(tag + " rows", got_ce, ce.detach(), TOL["cross_entropy"] * amax(ce), TOL["cross_entropy"])
    report(tag + " grad", got_d, ld.grad, TOL["cross_entropy"] * amax(ld.grad), TOL["cross_entropy"])
    assert bool((got_d.cpu()[w == 0] == 0).all()), "rows of weight 0 must get exactly zero gradient"
    want_m = got_ce.cpu().double().reshape(B, S)[:, start:].mean(1)
    report(tag + " row_mean", got_m, want_m, TOL["cross_entropy"] * amax(want_m), TOL["cross_entropy"])


def test_row_mean_long_rows(L):
    """rows longer than the 256-thread block (strided loop), start > 0."""
    x = torch.randn(5, 1000, generator=g(3)) + 0.5
    for start in (0, 1, 250, 999):
        got = L.row_mean(cu(x), start)
        report(f"row_mean n=1000 start={start}", got, x.double()[:, start:].mean(1), TOL["row_mean"] * amax(x), TOL["row_mean"])


@pytest.mark.parametrize("mult", [1.0, 2.5])
@pytest.mark.parametrize("tpv", [1, 16, 64])
def test_pose_loss_rows_and_grad(L, tpv, mult):
    BT = 6
    rows = BT * tpv
    raw = torch.randn(rows, 7, generator=g(tpv))
    poses = torch.randn(BT, 7, generator=g(tpv + 1))
    w = torch.rand(rows, generator=g(tpv + 2)) + 0.1
    w[::3] = 0.0
    pos_scale, ori_scale = 1.5, 0.7
    rd = raw.double().requires_grad_(True)
    y = poses.double().repeat_interleave(tpv, 0)
    pos = ((y[:, :3] * mult - rd[:, :3]) ** 2).mean(1)
    ori = ((y[:, 3:] - rd[:, 3:]) ** 2).mean(1)
    (w.double() * (pos_scale * pos + ori_scale * ori)).sum().backward()

    rc, pc = cu(raw), cu(poses)
    got_pos, got_ori = L.pose_loss_rows(rc, pc, tpv, mult)
    got_d = L.pose_loss_grad(rc, pc, cu(w), tpv, mult, pos_scale, ori_scale)
    torch.cuda.synchronize()
    tag = f"pose_loss tpv={tpv} mult={mult}"
    report(tag + " pos", got_pos, pos.detach(), TOL["pose_loss"] * amax(pos), TOL["pose_loss"])
    report(tag + " ori", got_ori, ori.detach(), TOL["pose_loss"] * amax(ori), TOL["pose_loss"])
    report(tag + " grad", got_d, rd.grad, TOL["pose_loss"] * amax(rd.grad), TOL["pose_loss"])


# ----------------------------------------------------------------------------- elementwise
def test_gelu_and_gelu_bwd(L):
    x = torch.cat([torch.linspace(-12, 12, 100001), torch.randn(GRID_CAP + 777, generator=g(1)) * 3])      # n odd, above the grid cap
    dy = torch.randn(x.numel(), generator=g(2))
    xd = x.double().requires_grad_(True)
    y = F.gelu(xd)
    y.backward(dy.double())
    got_y = L.gelu(cu(x))
    got_d = L.gelu_bwd(cu(x), cu(dy))
    torch.cuda.synchronize()
    report(f"gelu n={x.numel()}", got_y, y.detach(), TOL["gelu"] * amax(y), TOL["gelu"])
    report(f"gelu_bwd n={x.numel()}", got_d, xd.grad, TOL["gelu"] * amax(xd.grad), TOL["gelu"])


@pytest.mark.parametrize("mode", ["random_ids", "one_id", "fixed_token_no_pose"])
def test_migt_embed_bwd(L, mode):
    BT, Lt, d, V = 6, 16, 128, 50
    dh = torch.randn(BT * Lt, d, generator=g(1))
    if mode == "random_ids":
        ids = torch.randint(0, V, (BT, Lt), generator=g(2), dtype=torch.int32)
    elif mode == "one_id":
        ids = torch.full((BT, Lt), 7, dtype=torch.int32)            # every token of the batch lands in the same row
    else:
        ids = None
    fixed = V - 1
    wte, wpe, pose = (torch.randn(V, d, generator=g(3)).double().requires_grad_(True),
                      torch.randn(Lt + 3, d, generator=g(4)).double().requires_grad_(True),
                      torch.randn(BT, d, generator=g(5)).double().requires_grad_(True))
    tok = (ids.long() if ids is not None else torch.full((BT, Lt), fixed)).reshape(-1)
    h = wte[tok] + wpe[:Lt].repeat(BT, 1)
    if mode != "fixed_token_no_pose":
        h = h + pose.repeat_interleave(Lt, 0)
    h.backward(dh.double())
    pre = [torch.randn(t.shape, generator=g(10 + i)) for i, t in enumerate((wte, wpe, pose))]
    dwte, dwpe, dpose = cu(pre[0]), cu(pre[1]), cu(pre[2])
    L.migt_embed_bwd(cu(dh), ids.cuda() if ids is not None else None, fixed, BT, Lt, dwte, dwpe,
                     dpose if mode != "fixed_token_no_pose" else None)
    torch.cuda.synchronize()
    for name, got, p, leaf in (("dwte", dwte, pre[0], wte), ("dwpe", dwpe, pre[1], wpe), ("dpose", dpose, pre[2], pose)):
        gr = leaf.grad if leaf.grad is not None else torch.zeros_like(leaf)
        report(f"embed_bwd {mode} {name}", got, p.double() + gr, TOL["embed_bwd"] * max(amax(gr), 1.0), TOL["embed_bwd"])
    assert torch.equal(dwpe.cpu()[Lt:], pre[1][Lt:]), "rows of wpe past L must stay untouched"


def test_l1_grad(L):
    n = 2 * GRID_CAP + 13
    x = torch.randn(n, generator=g(1))
    y = torch.randn(n, generator=g(2))
    y[::7] = x[::7]                                             # exact ties: torch.abs backward gives 0 there
    scale = 1.0 / n
    dy, ls = L.l1_grad(cu(x), cu(y), scale)
    torch.cuda.synchronize()
    d = y - x                                                   # fp32 difference, as the kernel forms it
    want_dy = torch.sign(d) * torch.tensor(scale, dtype=torch.float32)
    assert torch.equal(dy.cpu(), want_dy)
    assert bool((dy.cpu()[::7] == 0).all())
    want_ls = float(d.abs().double().sum())
    print(f"[l1_grad] loss sum {float(ls):.12e} want {want_ls:.12e} rel err {abs(float(ls) - want_ls) / want_ls:.2e}")
    assert abs(float(ls) - want_ls) <= F64_TOL * want_ls


@pytest.mark.parametrize("pattern", ["x", "xy", "xz", "xyz", "xyz_out_is_x"])
def test_lincomb3(L, pattern):
    n = GRID_CAP + 1001
    x, y, z = (torch.randn(n, generator=g(i)) for i in range(3))
    a, b, c = 0.7, -1.3, 2.1
    want = a * x.double()
    if "y" in pattern:
        want = want + b * y.double()
    if "z" in pattern:
        want = want + c * z.double()
    xc = cu(x)
    out = L.lincomb3(a, xc, b, cu(y) if "y" in pattern else None, c, cu(z) if "z" in pattern else None,
                     out=xc if pattern.endswith("out_is_x") else None)
    torch.cuda.synchronize()
    if pattern.endswith("out_is_x"):
        assert out.data_ptr() == xc.data_ptr()
    report(f"lincomb3 {pattern}", out, want, TOL["lincomb3"] * amax(want), TOL["lincomb3"])


@pytest.mark.parametrize("N,H,W,C", [(2, 5, 7, 48), (3, 64, 40, 128)])
def test_sumpool2x2(L, N, H, W, C):
    u = torch.zeros(N, C, H, W, dtype=torch.float64, requires_grad=True)
    dx = torch.randn(N, 2 * H, 2 * W, C, generator=g(H))
    F.interpolate(u, scale_factor=2.0, mode="nearest").backward(dx.permute(0, 3, 1, 2).double())
    got = L.sumpool2x2(cu(dx))
    torch.cuda.synchronize()
    want = u.grad.permute(0, 2, 3, 1)
    report(f"sumpool2x2 {N}x{H}x{W}x{C}", got, want, TOL["sumpool2x2"] * amax(want), TOL["sumpool2x2"])


def test_sumsq(L):
    n = 10_000_019
    x = torch.randn(n, generator=g(1)) * 1e3
    got = float(L.sumsq(cu(x)))
    want = float((x.double() ** 2).sum())
    print(f"[sumsq n={n}] got {got:.15e} want {want:.15e} rel err {abs(got - want) / want:.2e}")
    assert abs(got - want) <= F64_TOL * want


# ----------------------------------------------------------------------------- optimizers
def test_adam(L):
    n, lr, betas, eps, gs = 1_000_003, 1e-3, (0.5, 0.9), 1e-8, 0.5
    f32 = _as_f32                                                # the kernel receives lr / betas / eps as fp32
    p0 = torch.randn(n, generator=g(1))
    grads = [torch.randn(n, generator=g(10 + t)) for t in range(5)]
    ref = p0.double().clone().requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=f32(lr), betas=(f32(betas[0]), f32(betas[1])), eps=f32(eps), foreach=False)
    p, m, v = cu(p0), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    for t, gr in enumerate(grads):
        ref.grad = gr.double() * gs
        opt.step()
        L.adam(p, cu(gr), m, v, lr=lr, beta1=betas[0], beta2=betas[1], eps=eps, step=t + 1, grad_scale=gs)
    torch.cuda.synchronize()
    st = opt.state[ref]
    # p is stored in fp32 after every step: up to half an ulp of |p| per step on top of the update itself
    ulp_p = 5 * 2.0 ** -24 * amax(p0) * 2
    T = TOL["adam"]
    report("adam update", p.cpu().double() - p0.double(), ref.detach() - p0.double(), ulp_p, T)
    report("adam m", m, st["exp_avg"], T * amax(st["exp_avg"]), T)
    report("adam v", v, st["exp_avg_sq"], T * amax(st["exp_avg_sq"]), T)


@pytest.mark.parametrize("wd", [0.0, 0.01])
def test_adamw_keras(L, wd):
    from oracle.make_golden import keras_adamw_reference
    n, lr, betas, eps, gs, cs = 300_007, 1e-2, (0.9, 0.999), 1e-8, 0.5, 0.8
    p0 = torch.randn(n, generator=g(1))
    grads = [torch.randn(n, generator=g(20 + t)) for t in range(5)]
    P, M, Vv = {"w": p0.double().clone()}, {"w": torch.zeros(n, dtype=torch.float64)}, {"w": torch.zeros(n, dtype=torch.float64)}
    p, m, v = cu(p0), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    for t, gr in enumerate(grads):
        keras_adamw_reference(P, {"w": gr.double() * gs * _as_f32(cs)}, M, Vv, t + 1, _as_f32(lr), _as_f32(wd),
                              betas=(_as_f32(betas[0]), _as_f32(betas[1])), eps=_as_f32(eps))
        L.adamw_keras(p, cu(gr), m, v, lr=lr, beta1=betas[0], beta2=betas[1], eps=eps, weight_decay=wd, step=t + 1, grad_scale=gs,
                      clip_scale=cs)
    torch.cuda.synchronize()
    ulp_p = 5 * 2.0 ** -24 * amax(p0) * 2
    T = TOL["adam"]
    report(f"adamw_keras wd={wd} update", p.cpu().double() - p0.double(), P["w"] - p0.double(), ulp_p, T)
    report(f"adamw_keras wd={wd} m", m, M["w"], T * amax(M["w"]), T)
    report(f"adamw_keras wd={wd} v", v, Vv["w"], T * amax(Vv["w"]), T)


# ----------------------------------------------------------------------------- weight / data gradients of the convolutions
def _conv_wgrad_case(L, x, dy, w_shape, fwd, kh, **kw):
    """x NHWC, dy NHWC; fwd(x_nchw, w) is the forward conv.  Returns (got dW incl. prefill, want)."""
    cout, cin = w_shape[0], w_shape[1]
    xd = x.permute(0, 3, 1, 2).double()
    wd = torch.zeros(w_shape, dtype=torch.float64, requires_grad=True)
    fwd(xd, wd).backward(dy.permute(0, 3, 1, 2).double())
    grad = wd.grad.permute(2, 3, 1, 0).reshape(kh * kh * cin, cout)           # [tap * Cin + ci, co]
    pre = torch.randn(grad.shape, generator=g(cin + cout))
    dw = cu(pre)
    L.conv_wgrad(cu(x), cu(dy), dw, kh=kh, **kw)
    torch.cuda.synchronize()
    return dw, pre.double() + grad, grad


@pytest.mark.parametrize("cin,cout,hw", [(3, 128, 16), (128, 3, 16), (96, 80, 9)])
def test_conv_wgrad_3x3(L, cin, cout, hw):
    x = torch.randn(2, hw, hw - 2, cin, generator=g(cin))
    dy = torch.randn(2, hw, hw - 2, cout, generator=g(cout))
    got, want, grad = _conv_wgrad_case(L, x, dy, (cout, cin, 3, 3), lambda a, w: F.conv2d(a, w, padding=1), 3)
    report(f"conv_wgrad 3x3 {cin}->{cout}", got, want, TOL["conv_wgrad"] * amax(grad), TOL["conv_wgrad"])


def test_conv_wgrad_stride2(L):
    x = torch.randn(2, 12, 10, 64, generator=g(1))
    dy = torch.randn(2, 6, 5, 32, generator=g(2))
    got, want, grad = _conv_wgrad_case(L, x, dy, (32, 64, 3, 3), lambda a, w: F.conv2d(F.pad(a, (0, 1, 0, 1)), w, stride=2), 3,
                                       stride=2, pad=(0, 0))
    report("conv_wgrad 3x3 stride 2", got, want, TOL["conv_wgrad"] * amax(grad), TOL["conv_wgrad"])


def test_conv_wgrad_upsample(L):
    x = torch.randn(2, 6, 5, 64, generator=g(3))
    dy = torch.randn(2, 12, 10, 48, generator=g(4))
    got, want, grad = _conv_wgrad_case(L, x, dy, (48, 64, 3, 3),
                                       lambda a, w: F.conv2d(F.interpolate(a, scale_factor=2.0, mode="nearest"), w, padding=1), 3,
                                       upsample=True)
    report("conv_wgrad 3x3 nearest-x2", got, want, TOL["conv_wgrad"] * amax(grad), TOL["conv_wgrad"])


@pytest.mark.parametrize("rows", [77, 4097])
def test_conv_wgrad_linear_layouts(L, rows):
    """1x1 'conv' over rows = the Linear weight gradient, written [out, in] (so=(1, k)) and [in, out] (so=(n, 1))."""
    k, n = 128, 96
    x = torch.randn(rows, k, generator=g(rows))
    dy = torch.randn(rows, n, generator=g(rows + 1))
    grad = x.double().t() @ dy.double()                          # [in, out]
    for so, want_g in (((1, k), grad.t()), ((n, 1), grad)):
        pre = torch.randn(want_g.shape, generator=g(so[0]))
        dw = cu(pre)
        L.conv_wgrad(cu(x).reshape(1, rows, 1, k), cu(dy).reshape(1, rows, 1, n), dw, kh=1, pad=(0, 0), so=so)
        torch.cuda.synchronize()
        report(f"conv_wgrad linear rows={rows} so={so}", dw, pre.double() + want_g, TOL["conv_wgrad"] * amax(want_g), TOL["conv_wgrad"])


@pytest.mark.parametrize("cin,cout,hw", [(128, 128, 32), (256, 256, 8), (96, 64, 6)])
def test_simt_conv_dgrad_s2(L, cin, cout, hw):
    n = 3
    w = torch.randn(cout, cin, 3, 3, generator=g(cin)) / (3 * cin ** 0.5)
    dy = torch.randn(n, hw // 2, hw // 2, cout, generator=g(cout))
    xd = torch.zeros(n, cin, hw, hw, dtype=torch.float64, requires_grad=True)
    F.conv2d(F.pad(xd, (0, 1, 0, 1)), w.double(), stride=2).backward(dy.permute(0, 3, 1, 2).double())
    want = xd.grad.permute(0, 2, 3, 1)
    w_dgrad = w.permute(2, 3, 0, 1).reshape(9 * cout, cin)       # [tap * Cout + co, ci], taps not flipped
    got = L.simt_conv_dgrad_s2(cu(dy), cu(w_dgrad), (hw, hw))
    torch.cuda.synchronize()
    report(f"simt_conv_dgrad_s2 {cin}->{cout} hw={hw}", got, want, TOL["conv_dgrad_s2"] * amax(want), TOL["conv_dgrad_s2"])


def _wgrad_err(got, want, grad):
    return amax(got.cpu().double() - want) / amax(grad)


@pytest.mark.parametrize("m,k,n", [(77, 128, 128), (1000, 128, 384), (4099, 768, 3072), (320, 128, 1024)])
def test_dense_wgrad_tc(L, m, k, n):
    x = torch.randn(m, k, generator=g(m))
    dy = torch.randn(m, n, generator=g(m + 1))
    grad = x.double().t() @ dy.double()
    pre = torch.randn(k, n, generator=g(m + 2))
    dw = cu(pre)
    L.dense_wgrad_tc(cu(x), cu(dy), dw)                          # accumulate=True
    torch.cuda.synchronize()
    e_acc = _wgrad_err(dw, pre.double() + grad, grad)
    # accumulate=False overwrites whatever the buffer held
    dw2 = cu(torch.randn(k, n, generator=g(m + 3)))
    L.dense_wgrad_tc(cu(x), cu(dy), dw2, accumulate=False)
    torch.cuda.synchronize()
    e_ovw = _wgrad_err(dw2, grad, grad)
    # the same shape again with new data: the cached operand buffers must hold the new operands only
    x2, dy2 = torch.randn(m, k, generator=g(m + 4)), torch.randn(m, n, generator=g(m + 5))
    grad2 = x2.double().t() @ dy2.double()
    dw3 = torch.zeros(k, n, device="cuda")
    L.dense_wgrad_tc(cu(x2), cu(dy2), dw3, accumulate=False)
    torch.cuda.synchronize()
    e_new = _wgrad_err(dw3, grad2, grad2)
    # the CUDA-core Linear weight gradient ([in, out] layout) computes the same thing
    dwc = torch.zeros(k, n, device="cuda")
    L.conv_wgrad(cu(x2).reshape(1, m, 1, k), cu(dy2).reshape(1, m, 1, n), dwc, kh=1, pad=(0, 0), so=(n, 1))
    torch.cuda.synchronize()
    e_cc = amax(dwc.cpu().double() - dw3.cpu().double()) / amax(grad2)
    print(f"[dense_wgrad_tc m={m} k={k} n={n}] max err / max|dW|: accumulate {e_acc:.2e} overwrite {e_ovw:.2e} second call {e_new:.2e}; "
          f"vs conv_wgrad {e_cc:.2e}")
    assert max(e_acc, e_ovw, e_new) < WGRAD_TC_TOL
    assert e_cc < TOL["wgrad_paths"]


def test_dense_wgrad_tc_into_leading_rows(L):
    """The tied LM head: dW of the first V rows of the [V + 2, d] embedding table; the two extra rows stay bit-identical."""
    m, V, d = 320, 1024, 128
    x = torch.randn(m, V, generator=g(1))
    dy = torch.randn(m, d, generator=g(2))
    grad = x.double().t() @ dy.double()
    pre = torch.randn(V + 2, d, generator=g(3))
    big = cu(pre)
    L.dense_wgrad_tc(cu(x), cu(dy), big[:V])
    torch.cuda.synchronize()
    e = _wgrad_err(big[:V], pre[:V].double() + grad, grad)
    print(f"[dense_wgrad_tc into big[:V]] max err / max|dW| {e:.2e}")
    assert e < WGRAD_TC_TOL
    assert torch.equal(big[V:].cpu(), pre[V:])


@pytest.mark.parametrize("rows,C", [(r, c) for r in (1, 7, 1024, 1025) for c in (3, 33, 768)] + [(3 * 2 ** 20 + 5, 3), (3 * 2 ** 20 + 5, 33)])
def test_col_sums(L, rows, C):
    x = torch.randn(rows, C, generator=g(rows + C)) + 0.25
    want = x.double().sum(0)
    pre = torch.randn(C, generator=g(C))
    out = cu(pre)
    L.col_sums(cu(x), out)
    torch.cuda.synchronize()
    scale = max(amax(want), float(rows) ** 0.5)
    report(f"col_sums rows={rows} C={C}", out, pre.double() + want, TOL["col_sums"] * scale, TOL["col_sums"])


@pytest.mark.parametrize("K", [64, 1024])
def test_vq_commit_grad(L, K):
    D, M, coef = 16, 500, 0.37
    emb = torch.randn(D, K, generator=g(K))
    z = torch.randn(M, D, generator=g(K + 1))
    idx = torch.randint(0, K // 2, (M,), generator=g(K + 2))     # codes K/2 .. K-1 are never used (zero count)
    e = emb.t().double().requires_grad_(True)
    (coef / 2 * ((e[idx] - z.double()) ** 2).sum()).backward()
    want = e.grad.t()
    counts, esum = L.vq_ema_stats(cu(z), idx.cuda(), K)
    grad = torch.full((D, K), float("nan"), device="cuda")
    L.vq_commit_grad(cu(emb), counts, esum, coef, grad)
    torch.cuda.synchronize()
    report(f"vq_commit_grad K={K}", grad, want, TOL["vq_commit"] * amax(want), TOL["vq_commit"])
    assert bool((grad.cpu()[:, K // 2:] == 0).all())


# ----------------------------------------------------------------------------- dropout
_M64 = (1 << 64) - 1


def _mix32(k):
    with np.errstate(over="ignore"):
        k = k ^ (k >> np.uint64(33))
        k = k * np.uint64(0xFF51AFD7ED558CCD)
        k = k ^ (k >> np.uint64(33))
        k = k * np.uint64(0xC4CEB9FE1A85EC53)
        k = k ^ (k >> np.uint64(33))
    return (k & np.uint64(0xFFFFFFFF)).astype(np.uint32)


def _dropout_ref(x, rate, seed):
    """Restatement of dropout_kernel (vf_backward.cu): keep element i iff mix32(seed * 0x9E3779B97F4A7C15 + i) >= rate * 2^32 (uint64
    wraparound, threshold formed in fp32), kept values x * float32(1 / (1 - rate)) with the division in fp32."""
    n = x.size
    base = np.uint64(((seed & _M64) * 0x9E3779B97F4A7C15) & _M64)
    with np.errstate(over="ignore"):
        keys = base + np.arange(n, dtype=np.uint64)
    thr = int(np.float32(rate) * np.float32(4294967296.0))
    keep = _mix32(keys) >= np.uint32(min(thr, 0xFFFFFFFF))
    sc = np.float32(1.0) / (np.float32(1.0) - np.float32(rate))
    return keep, np.where(keep, x * sc, np.float32(0.0)).astype(np.float32)


TRAINER_SEEDS = [(s * 1000003 + it) * 4096 + site for s, it, site in ((0, 0, 10), (0, 3, 104), (7, 1, 128), (12345, 999, 131))]


@pytest.mark.parametrize("seed", [0, 1, 12345, 2 ** 63, 2 ** 63 + 977, 2 ** 64 - 1] + TRAINER_SEEDS)
@pytest.mark.parametrize("rate", [0.1, 0.5])
def test_dropout_mask_bit_exact(L, rate, seed):
    n = GRID_CAP + 4099                                          # past the grid cap: the grid-stride loop runs twice
    x = (torch.randn(n, generator=g(seed % 1000)) + 0.1).numpy()
    got = L.dropout(torch.from_numpy(x).cuda(), rate, seed).cpu().numpy()
    keep, want = _dropout_ref(x, rate, seed)
    kept = int(keep.sum())
    sigma = (n * rate * (1 - rate)) ** 0.5
    print(f"[dropout rate={rate} seed={seed}] kept {kept}/{n} (expected {n * (1 - rate):.0f} +- {sigma:.0f}); "
          f"bit mismatches {int((got.view(np.uint32) != want.view(np.uint32)).sum())}")
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert np.array_equal(got != 0, keep)
    assert abs(kept - n * (1 - rate)) < 6 * sigma


def test_dropout_rate_zero_is_identity(L):
    x = torch.randn(GRID_CAP + 3, generator=g(1)).cuda()
    assert torch.equal(L.dropout(x, 0.0, 123), x)


@pytest.mark.parametrize("rate", [0.1, 0.5])
def test_dropout_adjacent_sites_uncorrelated(L, rate):
    """The trainer gives every site its own seed (base * 4096 + site): masks of neighbouring sites agree on (1-r)^2 + r^2 of the elements."""
    n = GRID_CAP + 17
    ones = torch.ones(n, device="cuda")
    base = (3 * 1000003 + 5) * 4096
    q = (1 - rate) ** 2 + rate ** 2
    sigma = (n * q * (1 - q)) ** 0.5
    for site in (10, 100, 104, 108):
        a = L.dropout(ones, rate, base + site) != 0
        b = L.dropout(ones, rate, base + site + 1) != 0
        agree = int((a == b).sum())
        print(f"[dropout sites {site}/{site + 1} rate={rate}] agree {agree}/{n} (expected {n * q:.0f} +- {sigma:.0f})")
        assert abs(agree - n * q) < 6 * sigma
