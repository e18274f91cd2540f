// Evaluation-side kernels around the hot path (SURVEY.md §8 f2 / f3): the dataset resize rule and the image metrics.
//   vf_resize_u8        viewformer/data/_common.py:19-44 (resize_th): uint8 -> float /255 -> torch.nn.functional.interpolate
//                       (bilinear align_corners=False when shrinking, nearest when growing) -> clamp -> * 255 -> uint8 (truncation)
//   vf_image_pair_sums  per-image sum |a-b| and sum (a-b)^2 over uint8 images: MSE / MAE / RMSE / PSNR follow exactly on the host
//                       (viewformer/utils/metrics.py:173-205, tf.image.psnr)
//   vf_ssim_u8[_k]      viewformer/utils/metrics.py:17-73: 7x7 uniform window, VALID, sample covariance, K1 = 0.01, K2 = 0.03 (or the caller's),
//                       data range 1, mean over (H-6) x (W-6) x C
#include "vf_common.cuh"

namespace {

// torch's area_pixel_compute_source_index(scale, dst, align_corners=false, cubic=false): scale * (dst + 0.5) - 0.5, clamped at 0
__device__ __forceinline__ float src_index(float scale, int dst) {
    const float s = __fsub_rn(__fmul_rn(scale, __fadd_rn((float)dst, 0.5f)), 0.5f);
    return s < 0.f ? 0.f : s;
}

__global__ void resize_u8_kernel(const uint8_t* __restrict__ x, int N, int H, int W, int C, int OH, int OW, int bilinear,
                                 uint8_t* __restrict__ y) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)N * OH * OW * C;
    if (i >= total) return;
    const int c = (int)(i % C);
    long long r = i / C;
    const int ox = (int)(r % OW);
    r /= OW;
    const int oy = (int)(r % OH);
    const int n = (int)(r / OH);
    const uint8_t* img = x + (long long)n * H * W * C;
    auto px = [&](int yy, int xx) { return __fdiv_rn((float)img[((long long)yy * W + xx) * C + c], 255.f); };
    float v;
    if (!bilinear) {
        // torch 'nearest': src = min(floor(dst * scale), in - 1), scale = (float)in / out
        const float sh = (float)H / (float)OH, sw = (float)W / (float)OW;
        int sy = (int)floorf(__fmul_rn((float)oy, sh)), sx = (int)floorf(__fmul_rn((float)ox, sw));
        sy = sy < H - 1 ? sy : H - 1;
        sx = sx < W - 1 ? sx : W - 1;
        v = px(sy, sx);
    } else {
        const float sh = (float)H / (float)OH, sw = (float)W / (float)OW;
        const float fy = src_index(sh, oy), fx = src_index(sw, ox);
        const int y0 = (int)fy, x0 = (int)fx;
        const int y1 = y0 + (y0 < H - 1 ? 1 : 0), x1 = x0 + (x0 < W - 1 ? 1 : 0);
        const float ly1 = __fsub_rn(fy, (float)y0), lx1 = __fsub_rn(fx, (float)x0);
        const float ly0 = __fsub_rn(1.f, ly1), lx0 = __fsub_rn(1.f, lx1);
        // h0lambda * (w0lambda * p00 + w1lambda * p01) + h1lambda * (w0lambda * p10 + w1lambda * p11)   (UpSampleKernel.cpp)
        const float top = __fadd_rn(__fmul_rn(lx0, px(y0, x0)), __fmul_rn(lx1, px(y0, x1)));
        const float bot = __fadd_rn(__fmul_rn(lx0, px(y1, x0)), __fmul_rn(lx1, px(y1, x1)));
        v = __fadd_rn(__fmul_rn(ly0, top), __fmul_rn(ly1, bot));
    }
    v = fminf(fmaxf(v, 0.f), 1.f);
    y[i] = (uint8_t)(__fmul_rn(v, 255.f));          // .to(torch.uint8): truncation toward zero
}

// one block per image: exact integer sums
__global__ void __launch_bounds__(256) pair_sums_kernel(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, long long per_image,
                                                        unsigned long long* __restrict__ out) {
    __shared__ unsigned long long s1[8], s2[8];
    const uint8_t* pa = a + (long long)blockIdx.x * per_image;
    const uint8_t* pb = b + (long long)blockIdx.x * per_image;
    unsigned long long l1 = 0, l2 = 0;
    for (long long i = threadIdx.x; i < per_image; i += 256) {
        const int d = (int)pa[i] - (int)pb[i];
        l1 += (unsigned)(d < 0 ? -d : d);
        l2 += (unsigned)(d * d);
    }
    for (int o = 16; o > 0; o >>= 1) { l1 += __shfl_xor_sync(0xffffffffu, l1, o); l2 += __shfl_xor_sync(0xffffffffu, l2, o); }
    if ((threadIdx.x & 31) == 0) { s1[threadIdx.x >> 5] = l1; s2[threadIdx.x >> 5] = l2; }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t1 = 0, t2 = 0;
        for (int w = 0; w < 8; ++w) { t1 += s1[w]; t2 += s2[w]; }
        out[2 * blockIdx.x] = t1;
        out[2 * blockIdx.x + 1] = t2;
    }
}

// grid (chunks, N): every thread strides over the (H-6)(W-6)C window positions of one image; integer window sums are exact
__global__ void __launch_bounds__(256) ssim_u8_kernel(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, int H, int W, int C,
                                                      float C1, float C2, double* __restrict__ out) {
    __shared__ double sh[8];
    const int OH = H - 6, OW = W - 6;
    const long long total = (long long)OH * OW * C;
    const uint8_t* pa = a + (long long)blockIdx.y * H * W * C;
    const uint8_t* pb = b + (long long)blockIdx.y * H * W * C;
    const float cov_norm = 49.f / 48.f;                   // C1 = (K1 R)^2, C2 = (K2 R)^2 with data range R = 1 come from the caller
    double acc = 0.0;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
        const int c = (int)(i % C);
        const long long r = i / C;
        const int ox = (int)(r % OW), oy = (int)(r / OW);
        unsigned sx = 0, sy = 0, sxx = 0, syy = 0, sxy = 0;
        for (int dy = 0; dy < 7; ++dy)
            for (int dx = 0; dx < 7; ++dx) {
                const long long o = ((long long)(oy + dy) * W + ox + dx) * C + c;
                const unsigned xv = pa[o], yv = pb[o];
                sx += xv; sy += yv; sxx += xv * xv; syy += yv * yv; sxy += xv * yv;
            }
        // window means of X = x/255 etc. (the reference filters with 1/49 weights in fp32; the integer sums here are exact)
        const float ux = (float)sx / (49.f * 255.f), uy = (float)sy / (49.f * 255.f);
        // uxx - ux*ux = (49 sxx - sx^2) / (49^2 255^2): the numerators are formed exactly (|.| < 2^28) and converted once, since
        // the fp32 difference of the two means cancels on bright, nearly flat windows (an SSIM error of 2e-5 at 250 vs 250|251)
        const long long nx = 49ll * sxx - (long long)sx * sx, ny = 49ll * syy - (long long)sy * sy, nxy = 49ll * sxy - (long long)sx * sy;
        const float vscale = 1.f / (2401.f * 65025.f);
        const float vx = cov_norm * ((float)nx * vscale), vy = cov_norm * ((float)ny * vscale), vxy = cov_norm * ((float)nxy * vscale);
        const float A1 = 2.f * ux * uy + C1, A2 = 2.f * vxy + C2, B1 = ux * ux + uy * uy + C1, B2 = vx + vy + C2;
        acc += (double)((A1 * A2) / (B1 * B2));
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0;
        for (int w = 0; w < 8; ++w) t += sh[w];
        atomicAdd(out + blockIdx.y, t / (double)total);
    }
}

}  // namespace

extern "C" int vf_resize_u8(const void* x, int N, int H, int W, int C, int OH, int OW, int bilinear, void* y, vf_stream_t s) {
    VF_CHECK_ARG(x && y && N >= 0 && H > 0 && W > 0 && C > 0 && OH > 0 && OW > 0, "vf_resize_u8: bad args");
    const long long total = (long long)N * OH * OW * C;
    if (total == 0) return VF_OK;
    resize_u8_kernel<<<(unsigned)((total + 255) / 256), 256, 0, vf_s(s)>>>(reinterpret_cast<const uint8_t*>(x), N, H, W, C, OH, OW, bilinear,
                                                                            reinterpret_cast<uint8_t*>(y));
    VF_CHECK_LAUNCH("vf_resize_u8");
    return VF_OK;
}

extern "C" int vf_image_pair_sums(const void* a, const void* b, int N, int64_t per_image, uint64_t* out, vf_stream_t s) {
    VF_CHECK_ARG(N >= 0 && per_image > 0, "vf_image_pair_sums: bad args");
    if (N == 0) return VF_OK;                      // empty tensors may carry null pointers
    VF_CHECK_ARG(a && b && out, "vf_image_pair_sums: null pointer");
    pair_sums_kernel<<<N, 256, 0, vf_s(s)>>>(reinterpret_cast<const uint8_t*>(a), reinterpret_cast<const uint8_t*>(b), per_image,
                                              reinterpret_cast<unsigned long long*>(out));
    VF_CHECK_LAUNCH("vf_image_pair_sums");
    return VF_OK;
}

extern "C" int vf_ssim_u8_k(const void* a, const void* b, int N, int H, int W, int C, double K1, double K2, double* out, vf_stream_t s) {
    VF_CHECK_ARG(N >= 0 && H >= 7 && W >= 7 && C > 0 && N <= 65535, "vf_ssim_u8: bad args (images must be at least 7x7)");
    VF_CHECK_ARG(K1 >= 0.0 && K1 <= 1e3, "vf_ssim_u8: K1 out of range");
    VF_CHECK_ARG(K2 >= 0.0 && K2 <= 1e3, "vf_ssim_u8: K2 out of range");
    if (N == 0) return VF_OK;                      // empty tensors may carry null pointers
    VF_CHECK_ARG(a && b && out, "vf_ssim_u8: null pointer");
    cudaError_t e = cudaMemsetAsync(out, 0, sizeof(double) * N, vf_s(s));
    if (e != cudaSuccess) { vf_set_error("vf_ssim_u8: memset: %s", cudaGetErrorString(e)); return VF_ERR_CUDA; }
    const long long total = (long long)(H - 6) * (W - 6) * C;
    int chunks = (int)((total + 255) / 256);
    if (chunks > 64) chunks = 64;
    const float k1 = (float)K1, k2 = (float)K2;
    ssim_u8_kernel<<<dim3(chunks, N), 256, 0, vf_s(s)>>>(reinterpret_cast<const uint8_t*>(a), reinterpret_cast<const uint8_t*>(b), H, W, C,
                                                         k1 * k1, k2 * k2, out);
    VF_CHECK_LAUNCH("vf_ssim_u8");
    return VF_OK;
}

extern "C" int vf_ssim_u8(const void* a, const void* b, int N, int H, int W, int C, double* out, vf_stream_t s) {
    return vf_ssim_u8_k(a, b, N, H, W, C, 0.01, 0.03, out, s);          // the defaults of ssim() (metrics.py:17)
}
