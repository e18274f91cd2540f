"""ctypes binding of libvf_b200.so (include/vf_b200.h) + thin tensor-level helpers.

torch is used here only as the device-memory / stream plumbing: every helper passes raw
``data_ptr()`` values and the current CUDA stream handle across the C-ABI.  There is no CPU or
PyTorch fallback: if the shared library is missing or the device is not sm_100, calls raise.
"""
import ctypes as C
import os

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VF_B200_LIB") or os.path.join(HERE, "libvf_b200.so")

F32, BF16, F16X2 = 0, 1, 2     # F16X2: an fp32 value as two fp16 (hi | lo*2^11) along the channel axis — torch.float16 tensors with 2C channels
ACT_NONE, ACT_GELU = 0, 1
BIAS_NONE, BIAS_N, BIAS_M = 0, 1, 2

EXPORTS = [
    "vf_last_error", "vf_version", "vf_sizeof_simt_gemm", "vf_sizeof_tc_gemm", "vf_device_check", "vf_u8_to_unit_f32", "vf_unit_f32_to_u8",
    "vf_nchw_to_nhwc_f32", "vf_nhwc_to_nchw_f32", "vf_groupnorm_stats", "vf_groupnorm_apply", "vf_layernorm",
    "vf_simt_gemm", "vf_tc_gemm", "vf_vq_lookup", "vf_gather_rows", "vf_vq_ema_stats", "vf_vq_ema_update", "vf_vq_commit_grad",
    "vf_vq_prepare_codebook", "vf_migt_embed", "vf_softmax_rows", "vf_argmax_rows", "vf_pose_postprocess",
    "vf_cameras_prepare", "vf_cameras_from_relative",
    "vf_conv3x3_small_cin", "vf_conv3x3_small_cout", "vf_groupnorm_finalize", "vf_split_f16x2", "vf_attn_block_causal", "vf_attn_block_causal_tail", "vf_attn_block_causal_decode", "vf_attn_block_multiend",
    "vf_vq_split3", "vf_vq_select", "vf_cross_entropy_rows", "vf_pose_loss_rows", "vf_row_mean",
    "vf_vq_prepare_codebook_f16", "vf_vq_lookup_fused", "vf_resize_u8", "vf_image_pair_sums", "vf_ssim_u8", "vf_ssim_u8_k",
    "vf_conv_wgrad", "vf_pad_transpose_split", "vf_sum_splits", "vf_col_sums", "vf_groupnorm_bwd", "vf_softmax_bwd_rows", "vf_l1_grad", "vf_lincomb3", "vf_sumpool2x2", "vf_adam",
    "vf_layernorm_bwd", "vf_gelu_fwd", "vf_gelu_bwd", "vf_migt_embed_bwd", "vf_cross_entropy_grad", "vf_pose_loss_grad", "vf_adamw_keras", "vf_sumsq", "vf_dropout",
]


class SimtGemm(C.Structure):
    _fields_ = [
        ("A", C.c_void_p), ("a_dtype", C.c_int), ("conv", C.c_int),
        ("N", C.c_int), ("H", C.c_int), ("W", C.c_int), ("Cin", C.c_int),
        ("OH", C.c_int), ("OW", C.c_int), ("KH", C.c_int), ("KW", C.c_int), ("stride", C.c_int),
        ("pad_t", C.c_int), ("pad_l", C.c_int), ("upsample2x", C.c_int),
        ("a_sm", C.c_int64), ("a_sk", C.c_int64),
        ("B", C.c_void_p), ("b_dtype", C.c_int), ("b_sk", C.c_int64), ("b_sn", C.c_int64),
        ("M", C.c_int), ("Ncols", C.c_int), ("K", C.c_int), ("batch1", C.c_int), ("batch2", C.c_int),
        ("a_sb1", C.c_int64), ("a_sb2", C.c_int64), ("b_sb1", C.c_int64), ("b_sb2", C.c_int64),
        ("c_sb1", C.c_int64), ("c_sb2", C.c_int64),
        ("alpha", C.c_float), ("bias", C.c_void_p), ("bias_mode", C.c_int), ("act", C.c_int),
        ("residual", C.c_void_p), ("C_f32", C.c_void_p), ("C_bf16", C.c_void_p), ("ldc", C.c_int64),
    ]


class TcGemm(C.Structure):
    _fields_ = [
        ("conv", C.c_int), ("ab_dtype", C.c_int), ("A", C.c_void_p), ("B", C.c_void_p),
        ("M", C.c_int), ("Ncols", C.c_int), ("K", C.c_int), ("batch1", C.c_int), ("batch2", C.c_int),
        ("lda", C.c_int64), ("ldb", C.c_int64),
        ("a_sb1", C.c_int64), ("a_sb2", C.c_int64), ("b_sb1", C.c_int64), ("b_sb2", C.c_int64),
        ("N", C.c_int), ("H", C.c_int), ("W", C.c_int), ("Ctot", C.c_int), ("Cin", C.c_int),
        ("OH", C.c_int), ("OW", C.c_int), ("ntaps", C.c_int),
        ("tap_dy", C.c_int * 9), ("tap_dx", C.c_int * 9), ("tap_coff", C.c_int * 9),
        ("causal_block", C.c_int), ("causal_skip_n", C.c_int),
        ("alpha", C.c_float), ("bias", C.c_void_p), ("bias_mode", C.c_int), ("act", C.c_int),
        ("residual", C.c_void_p), ("C_f32", C.c_void_p), ("C_bf16", C.c_void_p),
        ("ldc", C.c_int64), ("c_sb1", C.c_int64), ("c_sb2", C.c_int64),
        ("gn_sums", C.c_void_p), ("gn_groups", C.c_int), ("gn_rows_per_img", C.c_int),
        ("norm_mean_rstd", C.c_void_p), ("norm_gamma", C.c_void_p), ("norm_beta", C.c_void_p),
        ("norm_groups", C.c_int), ("norm_swish", C.c_int),
        ("exact_lo_a", C.c_int64), ("exact_lo_b", C.c_int64),
    ]


_lib = None
_device_ok = []


class LibraryError(RuntimeError):
    pass


def load(require_device=False):
    """dlopen the in-tree library.  Fails loudly — there is no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LibraryError(f"{LIB_PATH} not found — run `python -m viewformer_b200.build` (no CPU/PyTorch fallback exists)")
        lib = C.CDLL(LIB_PATH)
        lib.vf_last_error.restype = C.c_char_p
        for name in EXPORTS:
            if not hasattr(lib, name):
                raise LibraryError(f"{LIB_PATH} does not export {name}")
            if name != "vf_last_error":
                getattr(lib, name).restype = C.c_int
        if lib.vf_sizeof_simt_gemm() != C.sizeof(SimtGemm) or lib.vf_sizeof_tc_gemm() != C.sizeof(TcGemm):
            raise LibraryError("parameter struct layout mismatch between _lib.py and include/vf_b200.h")
        _lib = lib
    if require_device and not _device_ok:
        if not torch.cuda.is_available():
            raise LibraryError("viewformer_b200 needs a CUDA device (sm_100a); no CPU fallback exists")
        rc = _lib.vf_device_check()
        if rc != 0:
            raise LibraryError(_lib.vf_last_error().decode())
        _device_ok.append(True)          # checked once per process (cudaGetDeviceProperties is slow)
    return _lib


_launches = 0


def reset_launch_count():
    global _launches
    _launches = 0


def launch_count():
    """Number of libvf_b200 kernel-launching C-ABI calls since the last reset (bench.py's gpu_launches)."""
    return _launches


def _check(rc):
    global _launches
    _launches += 1
    if rc != 0:
        raise LibraryError(f"libvf_b200 error {rc}: {_lib.vf_last_error().decode()}")


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def on_model_device(fn):
    """Method decorator for the model classes: run with the model's device as the CURRENT CUDA device.  Every wrapper below launches on
    ``torch.cuda.current_stream()`` of the current device and the library caches per-device attributes, so a model built with
    ``device='cuda:1'`` must not run while device 0 is current."""
    import functools

    @functools.wraps(fn)
    def wrap(self, *a, **k):
        dev = getattr(self, "device", None)
        if dev is None or dev.type != "cuda" or dev.index is None or dev.index == torch.cuda.current_device():
            return fn(self, *a, **k)
        with torch.cuda.device(dev):
            return fn(self, *a, **k)
    return wrap


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _dt(t):
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    if t.dtype == torch.float16:
        return F16X2
    raise TypeError(f"unsupported dtype {t.dtype}")


def _dev(t, dtype=None):
    assert t.is_cuda and t.is_contiguous(), "device-contiguous tensor expected"
    if t.device.index != torch.cuda.current_device():
        raise LibraryError(f"tensor on cuda:{t.device.index} but the current device is cuda:{torch.cuda.current_device()}: kernels launch on the "
                           "current device's stream (the model classes switch devices themselves; raw _lib callers must use torch.cuda.device)")
    if dtype is not None:
        assert t.dtype == dtype, f"expected {dtype}, got {t.dtype}"
    return t


# ----------------------------------------------------------------------------------------------- pixels / layout
def u8_to_unit(x_u8, first_views=None):
    """uint8 -> f32 x*(1/255)*2-1.  ``first_views=n`` on a [B,T,H,W,3] tensor converts views 0..n-1 of every scene
    into a contiguous [B*n,H,W,3] tensor (strided read, no gather copy)."""
    lib = load(True)
    _dev(x_u8, torch.uint8)
    if first_views is None:
        out = torch.empty(x_u8.shape, dtype=torch.float32, device=x_u8.device)
        _check(lib.vf_u8_to_unit_f32(_p(x_u8), _p(out), C.c_int64(1), C.c_int64(x_u8.numel()), C.c_int64(0), _stream()))
        return out
    b, t = x_u8.shape[:2]
    per_view = x_u8[0, 0].numel()
    out = torch.empty((b * first_views,) + tuple(x_u8.shape[2:]), dtype=torch.float32, device=x_u8.device)
    _check(lib.vf_u8_to_unit_f32(_p(x_u8), _p(out), C.c_int64(b), C.c_int64(first_views * per_view), C.c_int64(t * per_view), _stream()))
    return out


def unit_to_u8(x):
    lib = load(True)
    _dev(x, torch.float32)
    out = torch.empty(x.shape, dtype=torch.uint8, device=x.device)
    _check(lib.vf_unit_f32_to_u8(_p(x), _p(out), C.c_int64(x.numel()), _stream()))
    return out


def nchw_to_nhwc(x):
    lib = load(True)
    _dev(x, torch.float32)
    n, c, h, w = x.shape
    out = torch.empty((n, h, w, c), dtype=torch.float32, device=x.device)
    _check(lib.vf_nchw_to_nhwc_f32(_p(x), _p(out), n, c, h, w, _stream()))
    return out


def nhwc_to_nchw(x):
    lib = load(True)
    _dev(x, torch.float32)
    n, h, w, c = x.shape
    out = torch.empty((n, c, h, w), dtype=torch.float32, device=x.device)
    _check(lib.vf_nhwc_to_nchw_f32(_p(x), _p(out), n, c, h, w, _stream()))
    return out


def resize_u8(x_u8, size, method=None):
    """data/_common.py:19-62 (resize -> resize_th) for uint8 NHWC images [N,H,W,C] -> [N,size,size,C]: bilinear (align_corners=False)
    when shrinking, nearest when growing (or the explicit ``method``).  As in the reference, the images come back unchanged when
    either side already equals ``size`` (resize tests W, resize_th tests H), and the method is chosen by H: a non-square input
    can stay non-square."""
    lib = load(True)
    _dev(x_u8, torch.uint8)
    n, h, w, c = x_u8.shape
    if w == size or h == size:
        return x_u8
    if method is None:
        method = "nearest" if size > h else "bilinear"
    assert method in ("nearest", "bilinear")
    out = torch.empty((n, size, size, c), dtype=torch.uint8, device=x_u8.device)
    _check(lib.vf_resize_u8(_p(x_u8), n, h, w, c, size, size, int(method == "bilinear"), _p(out), _stream()))
    return out


def image_pair_sums(a_u8, b_u8):
    """uint8 images [N,...] x2 -> int64 [N,2] = (sum |a-b|, sum (a-b)^2) per image (exact)."""
    lib = load(True)
    _dev(a_u8, torch.uint8)
    _dev(b_u8, torch.uint8)
    assert a_u8.shape == b_u8.shape
    n = a_u8.shape[0]
    out = torch.empty((n, 2), dtype=torch.int64, device=a_u8.device)
    _check(lib.vf_image_pair_sums(_p(a_u8), _p(b_u8), n, C.c_int64(a_u8[0].numel() if n else 1), _p(out), _stream()))
    return out


def ssim_u8(a_u8, b_u8, k1=None, k2=None):
    """utils/metrics.py:17-73 on uint8 NHWC images -> float64 [N] mean SSIM per image.  ``k1`` / ``k2``: the K1 / K2 of ``ssim()``
    (defaults 0.01 / 0.03); the reference's SSIMMetric passes K1 = 1 (metrics.py:183)."""
    lib = load(True)
    _dev(a_u8, torch.uint8)
    _dev(b_u8, torch.uint8)
    n, h, w, c = a_u8.shape
    out = torch.empty((n,), dtype=torch.float64, device=a_u8.device)
    if k1 is None and k2 is None:
        _check(lib.vf_ssim_u8(_p(a_u8), _p(b_u8), n, h, w, c, _p(out), _stream()))
    else:
        _check(lib.vf_ssim_u8_k(_p(a_u8), _p(b_u8), n, h, w, c, C.c_double(0.01 if k1 is None else float(k1)),
                                C.c_double(0.03 if k2 is None else float(k2)), _p(out), _stream()))
    return out


# ----------------------------------------------------------------------------------------------- norms
def groupnorm(x, gamma, beta, *, swish, out_dtype, eps=1e-6, groups=32, upsample=False, normalize=True, s2d=False):
    """x f32|bf16 [N,H,W,C] -> GroupNorm(32) [+swish] [+nearest x2] as out_dtype (vqgan_th.py:11-17,29-30).
    A bf16 x must carry the statistics its producing conv accumulated (from the fp32 accumulators) in ``_gn_sums``."""
    lib = load(True)
    _dev(x)
    n, h, w, c = x.shape
    stats = None
    if normalize:
        stats = torch.empty((n, groups, 2), dtype=torch.float32, device=x.device)      # (mean, rstd)
        fused = getattr(x, "_gn_sums", None)        # statistics already accumulated by the producing conv's epilogue
        if fused is not None and fused[1] == groups:
            _check(lib.vf_groupnorm_finalize(_p(fused[0]), n * groups, C.c_double(float(h * w * (c // groups))), C.c_float(eps),
                                             _p(stats), _stream()))
        else:
            if x.dtype != torch.float32:
                raise LibraryError("groupnorm: a bf16 input needs fused statistics from its producer")
            sums = torch.empty((n, groups, 2), dtype=torch.float64, device=x.device)
            _check(lib.vf_groupnorm_stats(_p(x), n, h * w, c, groups, C.c_float(eps), _p(sums), _p(stats), _stream()))
    oshape = (n, 2 * h, 2 * w, c) if upsample else ((n, h // 2, w // 2, 4 * c) if s2d else (n, h, w, c))
    if out_dtype == torch.float16:          # split-fp16 pair [hi | lo] (exact tensor-core operand): twice the channels
        oshape = oshape[:3] + (2 * oshape[3],)
    y = torch.empty(oshape, dtype=out_dtype, device=x.device)
    _check(lib.vf_groupnorm_apply(_p(x), _dt(x), _p(stats), _p(gamma), _p(beta), n, h, w, c, groups, C.c_float(eps),
                                  int(normalize), int(swish), 1 if upsample else (2 if s2d else 0), _p(y), _dt(y), _stream()))
    return y


def layernorm(x, gamma, beta, out_dtype, eps=1e-5):
    lib = load(True)
    _dev(x, torch.float32)
    d = x.shape[-1]
    rows = x.numel() // d
    y = torch.empty(x.shape, dtype=out_dtype, device=x.device)
    _check(lib.vf_layernorm(_p(x), _p(gamma), _p(beta), C.c_int64(rows), d, C.c_float(eps), _p(y), _dt(y), _stream()))
    return y


# ----------------------------------------------------------------------------------------------- GEMM / conv
def _outs(out):
    f32 = out if (out is not None and out.dtype == torch.float32) else None
    b16 = out if (out is not None and out.dtype == torch.bfloat16) else None
    return f32, b16


def simt_conv(x, w_kn, bias, *, kh, stride=1, pad=(1, 1), upsample=False, residual=None, out_dtype=torch.float32, out=None):
    """fp32 CUDA-core convolution.  x [N,H,W,Cin] f32|bf16, w_kn [kh*kh*Cin, Cout] f32."""
    lib = load(True)
    _dev(x)
    n, h, w, cin = x.shape
    cout = w_kn.shape[1]
    vh, vw = (2 * h, 2 * w) if upsample else (h, w)
    if stride == 1:
        oh, ow = vh, vw
    else:
        oh, ow = vh // 2, vw // 2
    if out is None:
        out = torch.empty((n, oh, ow, cout), dtype=out_dtype, device=x.device)
    p = SimtGemm()
    p.A, p.a_dtype, p.conv = x.data_ptr(), _dt(x), 1
    p.N, p.H, p.W, p.Cin = n, h, w, cin
    p.OH, p.OW, p.KH, p.KW, p.stride = oh, ow, kh, kh, stride
    p.pad_t, p.pad_l, p.upsample2x = pad[0], pad[1], int(upsample)
    p.B, p.b_dtype, p.b_sk, p.b_sn = w_kn.data_ptr(), _dt(w_kn), cout, 1
    p.M, p.Ncols, p.K, p.batch1, p.batch2 = n * oh * ow, cout, kh * kh * cin, 1, 1
    p.alpha = 1.0
    p.bias, p.bias_mode = (bias.data_ptr(), BIAS_N) if bias is not None else (None, BIAS_NONE)
    p.act = ACT_NONE
    p.residual = residual.data_ptr() if residual is not None else None
    f32, b16 = _outs(out)
    p.C_f32 = f32.data_ptr() if f32 is not None else None
    p.C_bf16 = b16.data_ptr() if b16 is not None else None
    p.ldc = cout
    _check(lib.vf_simt_gemm(C.byref(p), _stream()))
    return out


def simt_gemm(A, B, out, *, M, N, K, a_strides, b_strides, ldc, batch=(1, 1), a_bs=(0, 0), b_bs=(0, 0), c_bs=(0, 0),
              alpha=1.0, bias=None, bias_mode=BIAS_NONE, act=ACT_NONE, residual=None, a_off=0, b_off=0, c_off=0):
    """Dense strided fp32 GEMM: C[m,n] = act(alpha*sum_k A(m,k) B(k,n) + bias) + residual.
    a_strides = (stride_m, stride_k), b_strides = (stride_k, stride_n) in elements; *_off element offsets."""
    lib = load(True)
    p = SimtGemm()
    p.A, p.a_dtype, p.conv = A.data_ptr() + a_off * A.element_size(), _dt(A), 0
    p.a_sm, p.a_sk = a_strides
    p.B, p.b_dtype = B.data_ptr() + b_off * B.element_size(), _dt(B)
    p.b_sk, p.b_sn = b_strides
    p.M, p.Ncols, p.K, p.batch1, p.batch2 = M, N, K, batch[0], batch[1]
    p.a_sb1, p.a_sb2 = a_bs
    p.b_sb1, p.b_sb2 = b_bs
    p.c_sb1, p.c_sb2 = c_bs
    p.alpha = alpha
    p.bias, p.bias_mode = (bias.data_ptr(), bias_mode) if bias is not None else (None, BIAS_NONE)
    p.act = act
    p.residual = (residual.data_ptr() + c_off * 4) if residual is not None else None
    f32, b16 = _outs(out)
    p.C_f32 = (f32.data_ptr() + c_off * 4) if f32 is not None else None
    p.C_bf16 = (b16.data_ptr() + c_off * 2) if b16 is not None else None
    p.ldc = ldc
    _check(lib.vf_simt_gemm(C.byref(p), _stream()))
    return out


def tc_gemm(A, B, out, *, M, N, K, lda, ldb, ldc, batch=(1, 1), a_bs=(0, 0), b_bs=(0, 0), c_bs=(0, 0), alpha=1.0,
            bias=None, bias_mode=BIAS_NONE, act=ACT_NONE, residual=None, a_off=0, b_off=0, c_off=0, causal_block=0,
            causal_skip_n=False, out2=None, gn_rows_per_img=0, gn_groups=32, lo_a=None, lo_b=None, k_offsets=None):
    """tcgen05 GEMM: C[m,n] = act(alpha*sum_k A[m,k] B[n,k] + bias) + residual; A,B K-major bf16 (or f32 -> TF32).
    ``out2`` optionally receives a second copy in the other dtype (f32 + bf16 from one epilogue).
    float16 operands = split-fp16 pairs (exact mode): a row holds hi(K) at column 0 and lo(K) at column ``lo_a`` / ``lo_b``."""
    lib = load(True)
    assert A.dtype == B.dtype
    p = TcGemm()
    if A.dtype == torch.float16:
        p.exact_lo_a, p.exact_lo_b = (K if lo_a is None else lo_a), (K if lo_b is None else lo_b)
    p.conv, p.ab_dtype = 0, _dt(A)
    p.A = A.data_ptr() + a_off * A.element_size()
    p.B = B.data_ptr() + b_off * B.element_size()
    p.M, p.Ncols, p.K, p.batch1, p.batch2 = M, N, K, batch[0], batch[1]
    p.lda, p.ldb = lda, ldb
    p.a_sb1, p.a_sb2 = a_bs
    p.b_sb1, p.b_sb2 = b_bs
    p.c_sb1, p.c_sb2 = c_bs
    p.causal_block, p.causal_skip_n = causal_block, int(causal_skip_n)
    if k_offsets is not None:            # batch1 index b reads A shifted by k_offsets[b] elements along K (vf_tc_gemm_t.ntaps in gemm mode)
        assert len(k_offsets) == batch[0] <= 9
        p.ntaps = len(k_offsets)
        for i, o in enumerate(k_offsets):
            p.tap_coff[i] = int(o)
    p.alpha = alpha
    p.bias, p.bias_mode = (bias.data_ptr(), bias_mode) if bias is not None else (None, BIAS_NONE)
    p.act = act
    p.residual = (residual.data_ptr() + c_off * 4) if residual is not None else None
    for o in (out, out2):
        if o is None:
            continue
        if o.dtype == torch.float32:
            p.C_f32 = o.data_ptr() + c_off * 4
        else:
            p.C_bf16 = o.data_ptr() + c_off * 2
    p.ldc = ldc
    sums = None
    if gn_rows_per_img and batch == (1, 1) and gn_fusable(N, gn_groups, M, gn_rows_per_img, ldc):
        sums = torch.empty((M // gn_rows_per_img, gn_groups, 2), dtype=torch.float64, device=out.device)
        p.gn_sums, p.gn_groups, p.gn_rows_per_img = sums.data_ptr(), gn_groups, gn_rows_per_img
    _check(lib.vf_tc_gemm(C.byref(p), _stream()))
    if sums is not None:
        out._gn_sums = (sums, gn_groups)
    return out


def gn_fusable(channels, groups, rows, rows_per_img, ldc):
    """Shapes for which the tcgen05 epilogue can accumulate GroupNorm statistics (see vf_tc_gemm_t.gn_sums)."""
    if channels % groups:
        return False
    cpg = channels // groups
    return (cpg % 4 == 0 and cpg <= 32 and 32 % cpg == 0 and channels % 128 == 0 and rows_per_img >= 32 and rows_per_img % 32 == 0
            and rows % rows_per_img == 0 and ldc % 4 == 0)


TAPS_3x3 = [(dy, dx) for dy in (-1, 0, 1) for dx in (-1, 0, 1)]
# stride-2 conv over a space-to-depth operand: filter tap (dy,dx) in 0..2 reads phase (dy%2, dx%2) at offset (dy//2, dx//2)
TAPS_S2D = [(dy // 2, dx // 2) for dy in (0, 1, 2) for dx in (0, 1, 2)]


def s2d_coffs(c):
    return [((dy % 2) * 2 + (dx % 2)) * c for dy in (0, 1, 2) for dx in (0, 1, 2)]


def conv3x3_small_cin(x, w_kn, bias, gn_groups=0):
    """exact fp32 conv_in (Cin=3): x f32 [N,H,W,3], w_kn [27, Cout].  ``gn_groups=32`` (Cout = 128) also accumulates the
    GroupNorm statistics of the output and attaches them as ``_gn_sums`` (consumed by ``groupnorm``)."""
    lib = load(True)
    _dev(x, torch.float32)
    n, h, w, cin = x.shape
    cout = w_kn.shape[1]
    y = torch.empty((n, h, w, cout), dtype=torch.float32, device=x.device)
    sums = None
    if gn_groups == 32 and cout == 128:
        sums = torch.empty((n, 32, 2), dtype=torch.float64, device=x.device)
    _check(lib.vf_conv3x3_small_cin(_p(x), _p(w_kn), _p(bias), n, h, w, cin, cout, _p(y), _p(sums), _stream()))
    if sums is not None:
        y._gn_sums = (sums, 32)
    return y


def conv3x3_small_cout(x, w_kn, bias):
    """exact fp32-accumulate conv_out (128 -> 3): x f32|bf16 [N,H,W,128], w_kn [1152, 3]."""
    lib = load(True)
    _dev(x)
    n, h, w, cin = x.shape
    cout = w_kn.shape[1]
    y = torch.empty((n, h, w, cout), dtype=torch.float32, device=x.device)
    _check(lib.vf_conv3x3_small_cout(_p(x), _dt(x), _p(w_kn), _p(bias), n, h, w, cin, cout, _p(y), _stream()))
    return y


def conv_norm_fusable(x, cout):
    """Shapes for which vf_tc_gemm can apply GroupNorm+swish to the conv INPUT on the fly (vf_tc_gemm_t.norm_*)."""
    n, h, w, c = x.shape
    return (os.environ.get("VF_TC_WIDE", "1") != "0" and x.dtype == torch.bfloat16
            and c % 64 == 0 and cout % 128 == 0 and h >= 32 and w >= 8 and n * h * w * cout < 2 ** 31)


def gn_mean_rstd(x, groups=32, eps=1e-6):
    """(mean, rstd) float [N, groups, 2] of x [N,H,W,C] — from the statistics its producer fused, else one statistics pass."""
    lib = load(True)
    n, h, w, c = x.shape
    stats = torch.empty((n, groups, 2), dtype=torch.float32, device=x.device)
    fused = getattr(x, "_gn_sums", None)
    if fused is not None and fused[1] == groups:
        _check(lib.vf_groupnorm_finalize(_p(fused[0]), n * groups, C.c_double(float(h * w * (c // groups))), C.c_float(eps),
                                         _p(stats), _stream()))
    else:
        if x.dtype != torch.float32:
            raise LibraryError("gn_mean_rstd: a bf16 input needs fused statistics from its producer")
        sums = torch.empty((n, groups, 2), dtype=torch.float64, device=x.device)
        _check(lib.vf_groupnorm_stats(_p(x), n, h * w, c, groups, C.c_float(eps), _p(sums), _p(stats), _stream()))
    return stats


def tc_conv(x, w_nk, bias, *, taps=TAPS_3x3, coffs=None, cin=None, out_hw=None, residual=None, out=None,
            out_dtype=torch.float32, out2=None, gn_groups=0, norm=None):
    """tcgen05 implicit-GEMM conv.  x [N,H,W,Ctot] bf16|f32 NHWC; w_nk [Cout, ntaps*Cin] (K-major, same dtype).
    ``norm=(mean_rstd, gamma, beta, groups, swish)``: x is the RAW activation and GroupNorm(+swish) is applied to it inside the
    kernel (only for ``conv_norm_fusable`` shapes)."""
    lib = load(True)
    _dev(x)
    n, h, w, ctot = x.shape
    split = 2 if x.dtype == torch.float16 else 1            # exact mode: x = [hi | lo] halves, weights [Cout][tap][hi(Cin) | lo(Cin)]
    cin = ctot // split if cin is None else cin
    cout = w_nk.shape[0]
    oh, ow = (h, w) if out_hw is None else out_hw
    if out is None:
        out = torch.empty((n, oh, ow, cout), dtype=out_dtype, device=x.device)
    p = TcGemm()
    p.conv, p.ab_dtype = 1, _dt(x)
    assert w_nk.dtype == x.dtype and w_nk.shape[1] == len(taps) * cin * split
    p.A, p.B = x.data_ptr(), w_nk.data_ptr()
    p.Ncols = cout
    p.N, p.H, p.W, p.Ctot, p.Cin, p.OH, p.OW, p.ntaps = n, h, w, ctot, cin, oh, ow, len(taps)
    for i, (dy, dx) in enumerate(taps):
        p.tap_dy[i], p.tap_dx[i] = dy, dx
        p.tap_coff[i] = 0 if coffs is None else coffs[i]
    p.alpha = 1.0
    p.bias, p.bias_mode = (bias.data_ptr(), BIAS_N) if bias is not None else (None, BIAS_NONE)
    p.act = ACT_NONE
    p.residual = residual.data_ptr() if residual is not None else None
    for o in (out, out2):
        if o is None:
            continue
        if o.dtype == torch.float32:
            p.C_f32 = o.data_ptr()
        else:
            p.C_bf16 = o.data_ptr()
    p.ldc = cout
    sums = None
    if gn_groups and gn_fusable(cout, gn_groups, n * oh * ow, oh * ow, cout):
        sums = torch.empty((n, gn_groups, 2), dtype=torch.float64, device=out.device)
        p.gn_sums, p.gn_groups = sums.data_ptr(), gn_groups
    if norm is not None:
        mr, gamma, beta, ngroups, swish = norm
        _dev(mr, torch.float32); _dev(gamma, torch.float32); _dev(beta, torch.float32)
        p.norm_mean_rstd, p.norm_gamma, p.norm_beta = mr.data_ptr(), gamma.data_ptr(), beta.data_ptr()
        p.norm_groups, p.norm_swish = ngroups, int(swish)      # 0 none, 1 = ex2/rcp fp32 (as vf_groupnorm_apply), 2 = packed bf16 tanh
    _check(lib.vf_tc_gemm(C.byref(p), _stream()))
    if sums is not None:
        out._gn_sums = (sums, gn_groups)
    return out


# ----------------------------------------------------------------------------------------------- codebook
def vq_prepare_codebook(emb_dk):
    lib = load(True)
    _dev(emb_dk, torch.float32)
    d, k = emb_dk.shape
    et = torch.empty((k, d), dtype=torch.float32, device=emb_dk.device)
    esq = torch.empty((k,), dtype=torch.float32, device=emb_dk.device)
    _check(lib.vf_vq_prepare_codebook(_p(emb_dk), d, k, _p(et), _p(esq), _stream()))
    return et, esq


def vq_lookup(z_rows, et, esq, want_quant=True, want_diff=True):
    """z_rows f32 [M,D] -> (idx int64 [M], quant f32 [M,D] | None, diff_sum f64[1] | None)."""
    lib = load(True)
    _dev(z_rows, torch.float32)
    m, d = z_rows.shape
    k = et.shape[0]
    idx = torch.empty((m,), dtype=torch.int64, device=z_rows.device)
    quant = torch.empty((m, d), dtype=torch.float32, device=z_rows.device) if want_quant else None
    dsum = torch.zeros((1,), dtype=torch.float64, device=z_rows.device) if want_diff else None
    _check(lib.vf_vq_lookup(_p(z_rows), _p(et), _p(esq), C.c_int64(m), d, k, _p(idx), _p(quant), _p(dsum), _stream()))
    return idx, quant, dsum


def split_f16x2(x_rows):
    """f32 [rows, C] -> f16 [rows, 2C] = [hi | lo], hi = fp16(v), lo = fp16((v - hi) * 2^11) (weights of the exact convolution)."""
    lib = load(True)
    _dev(x_rows, torch.float32)
    rows, c = x_rows.shape
    out = torch.empty((rows, 2 * c), dtype=torch.float16, device=x_rows.device)
    _check(lib.vf_split_f16x2(_p(x_rows), C.c_int64(rows), c, _p(out), _stream()))
    return out


def vq_split3(x, codebook):
    """f32 [rows,D] -> bf16 [rows,3D] two-term split ([hi|hi|lo] for queries, [hi|lo|hi] for the codebook)."""
    lib = load(True)
    _dev(x, torch.float32)
    rows, d = x.shape
    out = torch.empty((rows, 3 * d), dtype=torch.bfloat16, device=x.device)
    _check(lib.vf_vq_split3(_p(x), C.c_int64(rows), d, int(codebook), _p(out), _stream()))
    return out


def vq_lookup_tc(z_rows, et, esq, et3, want_quant=True, want_diff=True, tol=1e-4, count_rescored=False):
    """Tensor-core lookup: bf16x3 distance GEMM on tcgen05 + exact fp64 re-score of near-ties.  Same outputs as vq_lookup."""
    lib = load(True)
    _dev(z_rows, torch.float32)
    m, d = z_rows.shape
    k = et.shape[0]
    a3 = vq_split3(z_rows, False)
    scores = torch.empty((m, k), dtype=torch.float32, device=z_rows.device)
    tc_gemm(a3, et3, scores, M=m, N=k, K=3 * d, lda=3 * d, ldb=3 * d, ldc=k, alpha=-2.0, bias=esq, bias_mode=BIAS_N)
    idx = torch.empty((m,), dtype=torch.int64, device=z_rows.device)
    quant = torch.empty((m, d), dtype=torch.float32, device=z_rows.device) if want_quant else None
    dsum = torch.zeros((1,), dtype=torch.float64, device=z_rows.device) if want_diff else None
    nres = torch.zeros((1,), dtype=torch.int32, device=z_rows.device) if count_rescored else None
    _check(lib.vf_vq_select(_p(scores), _p(z_rows), _p(et), _p(esq), C.c_int64(m), d, k, C.c_float(tol), _p(idx), _p(quant), _p(dsum),
                            _p(nres), _stream()))
    return (idx, quant, dsum, nres) if count_rescored else (idx, quant, dsum)


def vq_prepare_codebook_f16(et):
    """Et f32 [K,D] -> fp16(-2 e) [K,D], the B operand of the fused lookup."""
    lib = load(True)
    _dev(et, torch.float32)
    k, d = et.shape
    eh = torch.empty((k, d), dtype=torch.float16, device=et.device)
    _check(lib.vf_vq_prepare_codebook_f16(_p(et), k, d, _p(eh), _stream()))
    return eh


def vq_fused_ok(d, k):
    return d % 64 == 0 and d <= 256 and k % 256 == 0 and k <= 1024


def vq_lookup_fused(z_rows, et, esq, eh, emb_dk=None, want_quant=True, want_diff=True, tol_factor=0.25, return_counts=False):
    """Fused tcgen05 lookup (vf_vq_fused.cu): z read once, top-2 from TMEM, exact fp64 settlement of near-ties.  Same outputs as
    vq_lookup; ``return_counts`` adds the int32[2] tensor (rows settled between two candidates, rows settled over all codes)."""
    lib = load(True)
    _dev(z_rows, torch.float32)
    m, d = z_rows.shape
    k = et.shape[0]
    if emb_dk is None:
        emb_dk = et.t().contiguous()                         # callers that hold the reference's [D,K] layout pass it instead
    idx = torch.empty((m,), dtype=torch.int64, device=z_rows.device)
    work = torch.empty((max(m, 1), 4), dtype=torch.int32, device=z_rows.device)
    counter = torch.empty((2,), dtype=torch.int32, device=z_rows.device)
    quant = torch.empty((m, d), dtype=torch.float32, device=z_rows.device) if want_quant else None
    dsum = torch.zeros((1,), dtype=torch.float64, device=z_rows.device) if want_diff else None
    _check(lib.vf_vq_lookup_fused(_p(z_rows), _p(eh), _p(et), _p(emb_dk), _p(esq), C.c_int64(m), d, k, C.c_float(tol_factor), _p(idx), _p(work),
                                  _p(counter), _p(quant), _p(dsum), _stream()))
    return (idx, quant, dsum, counter) if return_counts else (idx, quant, dsum)


def gather_rows(table, idx):
    lib = load(True)
    _dev(table, torch.float32)
    _dev(idx, torch.int64)
    m = idx.numel()
    d = table.shape[1]
    out = torch.empty((m, d), dtype=torch.float32, device=table.device)
    _check(lib.vf_gather_rows(_p(table), _p(idx), C.c_int64(m), d, C.c_int64(table.shape[0]), _p(out), _stream()))
    return out


def vq_ema_stats(z_rows, idx, k):
    lib = load(True)
    m, d = z_rows.shape
    counts = torch.zeros((k,), dtype=torch.float32, device=z_rows.device)
    esum = torch.zeros((d, k), dtype=torch.float32, device=z_rows.device)
    _check(lib.vf_vq_ema_stats(_p(z_rows), _p(idx), C.c_int64(m), d, k, _p(counts), _p(esum), _stream()))
    return counts, esum


def vq_commit_grad(emb_dk, counts, esum, coef, grad_dk):
    lib = load(True)
    d, k = emb_dk.shape
    _check(lib.vf_vq_commit_grad(_p(emb_dk), _p(counts), _p(esum), d, k, C.c_float(coef), _p(grad_dk), _stream()))
    return grad_dk


def vq_ema_update(counts, esum, alpha, corr, eps, cs_hidden, dw_hidden, emb_dk, et, esq):
    lib = load(True)
    d, k = emb_dk.shape
    _check(lib.vf_vq_ema_update(_p(counts), _p(esum), d, k, C.c_float(alpha), C.c_float(corr), C.c_float(eps),
                                _p(cs_hidden), _p(dw_hidden), _p(emb_dk), _p(et), _p(esq), _stream()))


# ----------------------------------------------------------------------------------------------- transformer glue
def migt_embed(ids_i32, fixed_token, wte, wpe, pose_rows, BT, L):
    lib = load(True)
    d = wte.shape[1]
    out = torch.empty((BT * L, d), dtype=torch.float32, device=wte.device)
    _check(lib.vf_migt_embed(_p(ids_i32), int(fixed_token), _p(wte), _p(wpe), _p(pose_rows), C.c_int64(BT), L, d, _p(out),
                             _stream()))
    return out


def attn_block_causal(qk, vt, B, S, H, d, block, first_query=0, out=None, skip_view=-1):
    """Fused tcgen05 block-causal attention: qk bf16 [B,S,2d] (q|k), vt bf16 [B,d,S] -> bf16 [B*S, d].
    ``first_query`` > 0 computes only the query rows from that row's 128-row tile on (KV-cache decode); ``skip_view`` >= 0 leaves the
    keys of that view out (an unused slot of the cache)."""
    lib = load(True)
    _dev(qk, torch.bfloat16)
    _dev(vt, torch.bfloat16)
    if out is None:
        out = torch.empty((B * S, d), dtype=torch.bfloat16, device=qk.device)
    _check(lib.vf_attn_block_causal_decode(_p(qk), _p(vt), B, S, H, d, block, int(first_query), int(skip_view), _p(out), _stream()))
    return out


def attn_block_multiend(qk, vt, B, S, n_streams, stream, H, d, block, out=None):
    """Fused branching attention of stream ``stream`` (0 = block-causal over stream 0; s >= 1 = stream-0 keys of earlier views + own
    view of stream s): qk bf16 [B, n_streams*S, 2d], vt bf16 [B, d, n_streams*S] -> bf16 [B*S, d]."""
    lib = load(True)
    _dev(qk, torch.bfloat16)
    _dev(vt, torch.bfloat16)
    if out is None:
        out = torch.empty((B * S, d), dtype=torch.bfloat16, device=qk.device)
    _check(lib.vf_attn_block_multiend(_p(qk), _p(vt), B, S, n_streams, stream, H, d, block, _p(out), _stream()))
    return out


def softmax_rows(scores, P, *, rows_total, rows_per_batch, cols, ld_in, ld_out, mask_mode=0, block=0, row0=0):
    lib = load(True)
    _check(lib.vf_softmax_rows(_p(scores), C.c_int64(rows_total), rows_per_batch, cols, C.c_int64(ld_in), mask_mode, block,
                               row0, _p(P), _dt(P), C.c_int64(ld_out), _stream()))
    return P


def argmax_rows(x_rows):
    lib = load(True)
    _dev(x_rows, torch.float32)
    rows, cols = x_rows.shape
    out = torch.empty((rows,), dtype=torch.int64, device=x_rows.device)
    _check(lib.vf_argmax_rows(_p(x_rows), C.c_int64(rows), cols, C.c_int64(cols), _p(out), _stream()))
    return out


def pose_postprocess(raw_rows, mult):
    lib = load(True)
    _dev(raw_rows, torch.float32)
    out = torch.empty_like(raw_rows)
    _check(lib.vf_pose_postprocess(_p(raw_rows), C.c_int64(raw_rows.shape[0]), C.c_float(mult), _p(out), _stream()))
    return out


def cameras_prepare(cams, relative):
    """cams f32 [B,T,7] (device) -> (relative+normalised cams [B,T,7], transform [B,7]) in one launch."""
    lib = load(True)
    _dev(cams, torch.float32)
    b, t, _ = cams.shape
    out = torch.empty_like(cams)
    tr = torch.empty((b, 7), dtype=torch.float32, device=cams.device)
    _check(lib.vf_cameras_prepare(_p(cams), b, t, int(relative), _p(out), _p(tr), _stream()))
    return out, tr


def cameras_from_relative(cams, transform):
    lib = load(True)
    _dev(cams, torch.float32)
    b, n, _ = cams.shape
    out = torch.empty_like(cams)
    _check(lib.vf_cameras_from_relative(_p(cams), _p(transform), b, n, _p(out), _stream()))
    return out


def cross_entropy_rows(logits_rows, labels_i32, smoothing=0.0):
    lib = load(True)
    _dev(logits_rows, torch.float32)
    _dev(labels_i32, torch.int32)
    rows, cols = logits_rows.shape
    out = torch.empty((rows,), dtype=torch.float32, device=logits_rows.device)
    _check(lib.vf_cross_entropy_rows(_p(logits_rows), _p(labels_i32), C.c_int64(rows), cols, C.c_float(smoothing), _p(out), _stream()))
    return out


def pose_loss_rows(raw_rows, poses_bt7, tokens_per_view, mult):
    lib = load(True)
    rows = raw_rows.shape[0]
    pos = torch.empty((rows,), dtype=torch.float32, device=raw_rows.device)
    ori = torch.empty((rows,), dtype=torch.float32, device=raw_rows.device)
    _check(lib.vf_pose_loss_rows(_p(raw_rows), _p(poses_bt7), C.c_int64(rows), tokens_per_view, C.c_float(mult), _p(pos), _p(ori), _stream()))
    return pos, ori


def row_mean(x_rows, start=0):
    """x [rows, n] -> [rows] mean over columns start..n-1."""
    lib = load(True)
    _dev(x_rows, torch.float32)
    rows, n = x_rows.shape
    out = torch.empty((rows,), dtype=torch.float32, device=x_rows.device)
    _check(lib.vf_row_mean(_p(x_rows), C.c_int64(rows), n, start, _p(out), _stream()))
    return out


# ----------------------------------------------------------------------------------------------- backward pass (training step)
def simt_conv_dgrad_s2(dy, w_dgrad_kn, in_hw):
    """Data gradient of the stride-2 Downsample conv: dy f32 [N,OH,OW,Cout], w_dgrad_kn [9*Cout, Cin] (tap-major, NOT flipped)
    -> dx f32 [N,H,W,Cin]."""
    lib = load(True)
    _dev(dy, torch.float32)
    n, oh, ow, cout = dy.shape
    h, w = in_hw
    cin = w_dgrad_kn.shape[1]
    out = torch.empty((n, h, w, cin), dtype=torch.float32, device=dy.device)
    p = SimtGemm()
    p.A, p.a_dtype, p.conv = dy.data_ptr(), F32, 2
    p.N, p.H, p.W, p.Cin = n, oh, ow, cout
    p.OH, p.OW, p.KH, p.KW, p.stride = h, w, 3, 3, 1
    p.pad_t, p.pad_l, p.upsample2x = 0, 0, 0
    p.B, p.b_dtype, p.b_sk, p.b_sn = w_dgrad_kn.data_ptr(), F32, cin, 1
    p.M, p.Ncols, p.K, p.batch1, p.batch2 = n * h * w, cin, 9 * cout, 1, 1
    p.alpha, p.act, p.bias_mode = 1.0, ACT_NONE, BIAS_NONE
    p.C_f32, p.ldc = out.data_ptr(), cin
    _check(lib.vf_simt_gemm(C.byref(p), _stream()))
    return out


def conv_wgrad(x, dy, dw, *, kh, stride=1, pad=(1, 1), upsample=False, so=None):
    """dw (zeroed by the caller, accumulated here) [kh*kh*Cin, Cout] (or any layout via ``so`` = (stride of k, stride of co))."""
    lib = load(True)
    _dev(x, torch.float32); _dev(dy, torch.float32); _dev(dw, torch.float32)
    n, h, w, cin = x.shape
    _, oh, ow, cout = dy.shape
    so_k, so_n = (cout, 1) if so is None else so
    _check(lib.vf_conv_wgrad(_p(x), _p(dy), n, h, w, cin, oh, ow, cout, kh, kh, stride, pad[0], pad[1], int(upsample), C.c_int64(so_k),
                             C.c_int64(so_n), _p(dw), _stream()))
    return dw


_wgrad_bufs = {}


def conv_wgrad_tc_ok(x, dy, kh, stride, upsample):
    n, h, w, cin = x.shape
    return kh == 3 and stride == 1 and not upsample and cin % 128 == 0 and dy.shape[-1] % 128 == 0 and dy.shape[1:3] == x.shape[1:3]


def conv_wgrad_tc(x, dy, dw, *, accumulate=True):
    """Weight gradient of a 3x3 stride-1 pad-1 convolution on the exact split-fp16 tensor-core GEMM.  x [N,H,W,Cin], dy [N,H,W,Cout] fp32;
    dw [9*Cin, Cout] (k = (ky*3 + kx)*Cin + c).  dW[ky,kx][c, co] = sum_q xpad[c, q + (ky-1) pitch + (kx-1)] * dypad[co, q] over the
    zero-padded pixel grid: both operands are transposed to K-major split form, the horizontal shifts are three row blocks of the activation
    operand (M = 3 Cin), the vertical ones are K offsets of whole (8-aligned) rows, the pixel axis is split over the SMs and the partial
    products are folded by vf_sum_splits."""
    lib = load(True)
    _dev(x, torch.float32); _dev(dy, torch.float32); _dev(dw, torch.float32)
    n, h, w, cin = x.shape
    cout = dy.shape[-1]
    pitch = (w + 2 + 7) // 8 * 8
    ppad = n * (h + 2) * pitch
    tiles = (3 * cin // 128) * (cout // 128)
    splits = max(1, min(64, (148 + 3 * tiles - 1) // (3 * tiles)))
    kc = (ppad + splits - 1) // splits
    kc = (kc + 63) // 64 * 64                                  # the exact GEMM walks K in blocks of 64
    kpad = kc * splits
    margin = pitch + 8                                          # multiple of 8, >= pitch + 1
    la = kpad + 2 * margin
    lb = kpad
    # operand buffers are cached per shape: the transposer rewrites every interior position on each call and never touches the zero
    # borders / pitch padding / margins, so they are cleared once
    key = (x.device, n, h, w, cin, cout)
    bufs = _wgrad_bufs.get(key)
    if bufs is None:
        if len(_wgrad_bufs) >= 32:
            _wgrad_bufs.clear()
        bufs = (torch.zeros((3 * cin, 2, la), dtype=torch.float16, device=x.device), torch.zeros((cout, 2, lb), dtype=torch.float16, device=x.device),
                torch.empty((3, splits, 3 * cin, cout), dtype=torch.float32, device=x.device))
        _wgrad_bufs[key] = bufs
    at, bt, partial = bufs
    _check(lib.vf_pad_transpose_split(_p(x), n, h, w, cin, pitch, 3, C.c_int64(margin), C.c_int64(la), _p(at), _stream()))
    _check(lib.vf_pad_transpose_split(_p(dy), n, h, w, cout, pitch, 1, C.c_int64(0), C.c_int64(lb), _p(bt), _stream()))
    offs = [margin - pitch, margin, margin + pitch]
    tc_gemm(at, bt, partial, M=3 * cin, N=cout, K=kc, lda=2 * la, ldb=2 * lb, ldc=cout, batch=(3, splits), a_bs=(0, kc), b_bs=(0, kc),
            c_bs=(splits * 3 * cin * cout, 3 * cin * cout), lo_a=la, lo_b=lb, k_offsets=offs)
    _check(lib.vf_sum_splits(_p(partial), 3, splits, C.c_int64(3 * cin * cout), int(accumulate), _p(dw), _stream()))
    return dw


def dense_wgrad_tc(x_rows, dy_rows, dw_kn, *, accumulate=True):
    """dW[k, n] (+)= sum_m x[m, k] dy[m, n] on the exact split-fp16 tensor-core GEMM (K = rows): both operands are transposed to K-major
    split form (vf_pad_transpose_split, plain mode), the row axis is split over the SMs, vf_sum_splits folds the partial products."""
    lib = load(True)
    _dev(x_rows, torch.float32); _dev(dy_rows, torch.float32); _dev(dw_kn, torch.float32)
    m, k = x_rows.shape
    n = dy_rows.shape[1]
    tiles = (k // 128) * (n // 128)
    splits = max(1, min(32, (148 + tiles - 1) // tiles))
    kc = ((m + splits - 1) // splits + 63) // 64 * 64
    lm = kc * splits
    key = ("dense", x_rows.device, m, k, n)
    bufs = _wgrad_bufs.get(key)
    if bufs is None:
        if len(_wgrad_bufs) >= 32:
            _wgrad_bufs.clear()
        bufs = (torch.zeros((k, 2, lm), dtype=torch.float16, device=x_rows.device), torch.zeros((n, 2, lm), dtype=torch.float16, device=x_rows.device),
                torch.empty((splits, k, n), dtype=torch.float32, device=x_rows.device))
        _wgrad_bufs[key] = bufs
    at, bt, partial = bufs
    _check(lib.vf_pad_transpose_split(_p(x_rows), 1, 1, m, k, 0, 1, C.c_int64(0), C.c_int64(lm), _p(at), _stream()))
    _check(lib.vf_pad_transpose_split(_p(dy_rows), 1, 1, m, n, 0, 1, C.c_int64(0), C.c_int64(lm), _p(bt), _stream()))
    tc_gemm(at, bt, partial, M=k, N=n, K=kc, lda=2 * lm, ldb=2 * lm, ldc=n, batch=(1, splits), a_bs=(0, kc), b_bs=(0, kc),
            c_bs=(0, k * n), lo_a=lm, lo_b=lm)
    _check(lib.vf_sum_splits(_p(partial), 1, splits, C.c_int64(k * n), int(accumulate), _p(dw_kn), _stream()))
    return dw_kn


def col_sums(x_rows, out):
    lib = load(True)
    _dev(x_rows, torch.float32)
    _check(lib.vf_col_sums(_p(x_rows), C.c_int64(x_rows.numel() // x_rows.shape[-1]), x_rows.shape[-1], _p(out), _stream()))
    return out


def groupnorm_bwd(x, dout, mean_rstd, gamma, beta, dgamma, dbeta, *, swish, groups=32, add=None):
    lib = load(True)
    _dev(x, torch.float32); _dev(dout, torch.float32)
    n, h, w, c = x.shape
    dx = torch.empty_like(x)
    gs = torch.empty((n, groups, 2), dtype=torch.float64, device=x.device)
    _check(lib.vf_groupnorm_bwd(_p(x), _p(dout), _p(mean_rstd), _p(gamma), _p(beta), n, h * w, c, groups, int(swish), _p(add), _p(gs),
                                _p(dgamma), _p(dbeta), _p(dx), _stream()))
    return dx


def softmax_bwd_rows(P, dP):
    lib = load(True)
    dS = torch.empty_like(P)
    _check(lib.vf_softmax_bwd_rows(_p(P), _p(dP), C.c_int64(P.numel() // P.shape[-1]), P.shape[-1], _p(dS), _stream()))
    return dS


def l1_grad(x, y, scale):
    """(dy = scale * sign(y - x), loss_sum f64[1] = sum |y - x|)"""
    lib = load(True)
    dy = torch.empty_like(y)
    ls = torch.zeros((1,), dtype=torch.float64, device=y.device)
    _check(lib.vf_l1_grad(_p(x), _p(y), C.c_int64(y.numel()), C.c_float(scale), _p(dy), _p(ls), _stream()))
    return dy, ls


def lincomb3(a, x, b=0.0, y=None, c=0.0, z=None, out=None):
    lib = load(True)
    if out is None:
        out = torch.empty_like(x)
    _check(lib.vf_lincomb3(C.c_float(a), _p(x), C.c_float(b), _p(y), C.c_float(c), _p(z), C.c_int64(x.numel()), _p(out), _stream()))
    return out


def sumpool2x2(x):
    lib = load(True)
    n, h2, w2, c = x.shape
    y = torch.empty((n, h2 // 2, w2 // 2, c), dtype=torch.float32, device=x.device)
    _check(lib.vf_sumpool2x2(_p(x), n, h2 // 2, w2 // 2, c, _p(y), _stream()))
    return y


def adam(p, g, m, v, *, lr, beta1, beta2, eps, step, grad_scale=1.0):
    lib = load(True)
    _check(lib.vf_adam(_p(p), _p(g), _p(m), _p(v), C.c_int64(p.numel()), C.c_float(lr), C.c_float(beta1), C.c_float(beta2), C.c_float(eps),
                       int(step), C.c_float(grad_scale), _stream()))


def layernorm_bwd(x, dy, gamma, dgamma, dbeta, eps=1e-5, add=None):
    lib = load(True)
    d = x.shape[-1]
    dx = torch.empty_like(x)
    _check(lib.vf_layernorm_bwd(_p(x), _p(dy), _p(gamma), _p(add), C.c_int64(x.numel() // d), d, C.c_float(eps), _p(dgamma), _p(dbeta), _p(dx), _stream()))
    return dx


def gelu(x):
    lib = load(True)
    y = torch.empty_like(x)
    _check(lib.vf_gelu_fwd(_p(x), C.c_int64(x.numel()), _p(y), _stream()))
    return y


def gelu_bwd(pre, dy):
    lib = load(True)
    out = torch.empty_like(pre)
    _check(lib.vf_gelu_bwd(_p(pre), _p(dy), C.c_int64(pre.numel()), _p(out), _stream()))
    return out


def migt_embed_bwd(dh, ids_i32, fixed_token, BT, L, dwte, dwpe, dpose):
    lib = load(True)
    _check(lib.vf_migt_embed_bwd(_p(dh), _p(ids_i32), int(fixed_token), C.c_int64(BT), L, dh.shape[-1], _p(dwte), _p(dwpe), _p(dpose), _stream()))


def cross_entropy_grad(logits_rows, labels_i32, row_weight, smoothing=0.0):
    lib = load(True)
    rows, cols = logits_rows.shape
    out = torch.empty_like(logits_rows)
    _check(lib.vf_cross_entropy_grad(_p(logits_rows), _p(labels_i32), _p(row_weight), C.c_int64(rows), cols, C.c_float(smoothing), _p(out), _stream()))
    return out


def pose_loss_grad(raw_rows, poses_bt7, row_weight, tokens_per_view, mult, pos_scale=1.0, ori_scale=1.0):
    lib = load(True)
    out = torch.empty_like(raw_rows)
    _check(lib.vf_pose_loss_grad(_p(raw_rows), _p(poses_bt7), _p(row_weight), C.c_int64(raw_rows.shape[0]), tokens_per_view, C.c_float(mult),
                                 C.c_float(pos_scale), C.c_float(ori_scale), _p(out), _stream()))
    return out


def adamw_keras(p, g, m, v, *, lr, beta1, beta2, eps, weight_decay, step, grad_scale=1.0, clip_scale=1.0):
    lib = load(True)
    _check(lib.vf_adamw_keras(_p(p), _p(g), _p(m), _p(v), C.c_int64(p.numel()), C.c_float(lr), C.c_float(beta1), C.c_float(beta2), C.c_float(eps),
                              C.c_float(weight_decay), int(step), C.c_float(grad_scale), C.c_float(clip_scale), _stream()))


def sumsq(x):
    lib = load(True)
    out = torch.zeros((1,), dtype=torch.float64, device=x.device)
    _check(lib.vf_sumsq(_p(x), C.c_int64(x.numel()), _p(out), _stream()))
    return out


def dropout(x, rate, seed):
    lib = load(True)
    y = torch.empty_like(x)
    _check(lib.vf_dropout(_p(x), C.c_int64(x.numel()), C.c_float(rate), C.c_uint64(int(seed) & ((1 << 64) - 1)), _p(y), _stream()))
    return y
