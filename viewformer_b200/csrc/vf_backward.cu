// Backward-pass kernels of the codebook training step (viewformer/models/vqgan_th.py:395-423, 443-445; fp32 as the reference
// requires, vqgan_th.py:326).  Data gradients of the convolutions and all dense layers reuse the forward GEMM / conv kernels
// (a data gradient IS a convolution with flipped taps); this file holds what has no forward twin:
//   vf_conv_wgrad          dW[ky,kx,ci,co] = sum_pixels X(gathered as in the forward conv) * dY       (+ strides: also Linear dW)
//   vf_col_sums            bias gradients
//   vf_groupnorm_bwd       GroupNorm(32) [+ swish] backward: per-(image, group) sums, then dx; accumulates dgamma / dbeta
//   vf_softmax_bwd_rows    dS = P * (dP - sum_j dP_j P_j)
//   vf_l1_grad             d mean|x - y| / dy, and the loss sum
//   vf_lincomb3            out = a x + b y + c z   (gradient merges, straight-through + commitment term of the quantizer)
//   vf_sumpool2x2          backward of the nearest x2 upsampling
//   vf_adam                torch.optim.Adam step (betas (0.5, 0.9) at the call site) over a flat parameter / gradient buffer
#include "vf_common.cuh"
#include <cuda_fp16.h>

namespace {

constexpr int WT = 64;          // wgrad tile: 64 input channels x 64 output channels per block
constexpr int WP = 16;          // pixels per smem stage

// grid = (pixel chunks, taps, ci tiles * co tiles); every block reduces its pixel chunk and adds the tile to dW with fp32 atomics
__global__ void __launch_bounds__(256) conv_wgrad_kernel(const float* __restrict__ x, const float* __restrict__ dy, int N, int H, int W,
                                                         int Cin, int OH, int OW, int Cout, int KH, int KW, int stride, int pad_t,
                                                         int pad_l, int upsample2x, long long pix_per_block, long long so_k, long long so_n,
                                                         float* __restrict__ dw) {
    __shared__ float Xs[WP][WT + 4];
    __shared__ float Ys[WP][WT + 4];
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    const int tap = blockIdx.y, kh = tap / KW, kw = tap % KW;
    const int co_tiles = (Cout + WT - 1) / WT;
    const int ci0 = (blockIdx.z / co_tiles) * WT, co0 = (blockIdx.z % co_tiles) * WT;
    const long long total = (long long)N * OH * OW;
    const long long p0 = (long long)blockIdx.x * pix_per_block;
    const long long p1 = p0 + pix_per_block < total ? p0 + pix_per_block : total;
    const int VH = upsample2x ? 2 * H : H, VW = upsample2x ? 2 * W : W;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    // loader: thread -> (pixel lp of the stage, 4 consecutive channels lc)
    const int lp = tid >> 4, lc = (tid & 15) * 4;
    for (long long pb = p0; pb < p1; pb += WP) {
        const long long p = pb + lp;
        float xv[4] = {0.f, 0.f, 0.f, 0.f}, yv[4] = {0.f, 0.f, 0.f, 0.f};
        if (p < p1) {
            const int ox = (int)(p % OW);
            const long long t = p / OW;
            const int oy = (int)(t % OH), n = (int)(t / OH);
            const int iy = oy * stride + kh - pad_t, ix = ox * stride + kw - pad_l;
            if (iy >= 0 && iy < VH && ix >= 0 && ix < VW) {
                const int sy = upsample2x ? iy >> 1 : iy, sx = upsample2x ? ix >> 1 : ix;
                const float* xr = x + (((long long)n * H + sy) * W + sx) * Cin;
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (ci0 + lc + q < Cin) xv[q] = __ldg(xr + ci0 + lc + q);
                const float* yr = dy + p * Cout;
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (co0 + lc + q < Cout) yv[q] = __ldg(yr + co0 + lc + q);
            }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) { Xs[lp][lc + q] = xv[q]; Ys[lp][lc + q] = yv[q]; }
        __syncthreads();
#pragma unroll
        for (int pp = 0; pp < WP; ++pp) {
            const float4 a4 = *reinterpret_cast<const float4*>(&Xs[pp][ty * 4]);
            const float4 b4 = *reinterpret_cast<const float4*>(&Ys[pp][tx * 4]);
            const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int ci = ci0 + ty * 4 + i;
        if (ci >= Cin) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int co = co0 + tx * 4 + j;
            if (co < Cout) atomicAdd(dw + ((long long)tap * Cin + ci) * so_k + (long long)co * so_n, acc[i][j]);
        }
    }
}

// out[c] += sum over rows of x[row][c]; grid (column blocks of 32, row chunks)
__global__ void __launch_bounds__(256) col_sums_kernel(const float* __restrict__ x, long long rows, int C, long long rows_per_block,
                                                       float* __restrict__ out) {
    __shared__ float sh[8][33];
    const int c = blockIdx.x * 32 + (threadIdx.x & 31), rl = threadIdx.x >> 5;
    const long long r0 = (long long)blockIdx.y * rows_per_block, r1 = r0 + rows_per_block < rows ? r0 + rows_per_block : rows;
    float s = 0.f;
    if (c < C)
        for (long long r = r0 + rl; r < r1; r += 8) s += __ldg(x + r * C + c);
    sh[rl][threadIdx.x & 31] = s;
    __syncthreads();
    if (rl == 0 && c < C) {
        float t = 0.f;
        for (int w = 0; w < 8; ++w) t += sh[w][threadIdx.x & 31];
        atomicAdd(out + c, t);
    }
}

__device__ __forceinline__ float swish_grad(float g) {      // d/dg [g sigmoid(g)]
    const float sg = 1.0f / (1.0f + expf(-g));
    return sg * (1.0f + g * (1.0f - sg));
}

// pass 1: grid (pixel chunks, N), 256 threads, thread = one channel quad of the image (as gn_apply_kernel)
__global__ void __launch_bounds__(256) gn_bwd_stats_kernel(const float* __restrict__ x, const float* __restrict__ dout, const float* __restrict__ mr,
                                                           const float* __restrict__ gamma, const float* __restrict__ beta, int HW, int C,
                                                           int groups, int swish, int pix_per_block, double* __restrict__ gsums,
                                                           float* __restrict__ dgamma, float* __restrict__ dbeta) {
    extern __shared__ double shg[];           // [groups][2] doubles, then [2][C] floats (per-channel dbeta / dgamma of this block)
    float* shc = reinterpret_cast<float*>(shg + 2 * groups);
    const int quads = C >> 2, lanes = 256 / quads;
    const int cq = threadIdx.x % quads, pl = threadIdx.x / quads, n = blockIdx.y, cpg = C / groups;
    for (int i = threadIdx.x; i < groups * 2; i += 256) shg[i] = 0.0;
    for (int i = threadIdx.x; i < 2 * C; i += 256) shc[i] = 0.f;
    __syncthreads();
    float mu[4], rs[4], ga[4], be[4], s1[4] = {0, 0, 0, 0}, s2[4] = {0, 0, 0, 0};
    if (pl < lanes) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = cq * 4 + j;
            const float2 m = __ldg(reinterpret_cast<const float2*>(mr) + (long long)n * groups + c / cpg);
            mu[j] = m.x; rs[j] = m.y; ga[j] = __ldg(gamma + c); be[j] = __ldg(beta + c);
        }
        const int p0 = blockIdx.x * pix_per_block, p1 = min(HW, p0 + pix_per_block);
        for (int p = p0 + pl; p < p1; p += lanes) {
            const long long o = ((long long)n * HW + p) * C + cq * 4;
            const float4 xv = __ldg(reinterpret_cast<const float4*>(x + o)), dv = __ldg(reinterpret_cast<const float4*>(dout + o));
            const float xe[4] = {xv.x, xv.y, xv.z, xv.w}, de[4] = {dv.x, dv.y, dv.z, dv.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float xh = (xe[j] - mu[j]) * rs[j];
                float dg = de[j];
                if (swish) dg *= swish_grad(xh * ga[j] + be[j]);
                s1[j] += dg;
                s2[j] = fmaf(dg, xh, s2[j]);
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = cq * 4 + j;
            // the block's pixel lanes meet in shared memory first: one global atomic per (block, channel) instead of one per thread
            atomicAdd(shc + c, s1[j]);
            atomicAdd(shc + C + c, s2[j]);
            atomicAdd(&shg[(c / cpg) * 2 + 0], (double)(s1[j] * ga[j]));
            atomicAdd(&shg[(c / cpg) * 2 + 1], (double)(s2[j] * ga[j]));
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < groups * 2; i += 256) atomicAdd(gsums + (long long)n * groups * 2 + i, shg[i]);
    for (int c = threadIdx.x; c < C; c += 256) {
        atomicAdd(dbeta + c, shc[c]);
        atomicAdd(dgamma + c, shc[C + c]);
    }
}

// pass 2: dx = rstd * (dg*gamma - mean(dg*gamma) - xhat * mean(dg*gamma*xhat)) [+ add]
__global__ void __launch_bounds__(256) gn_bwd_apply_kernel(const float* __restrict__ x, const float* __restrict__ dout, const float* __restrict__ mr,
                                                           const float* __restrict__ gamma, const float* __restrict__ beta,
                                                           const double* __restrict__ gsums, const float* __restrict__ add, int HW, int C,
                                                           int groups, int swish, int pix_per_block, float* __restrict__ dx) {
    const int quads = C >> 2, lanes = 256 / quads;
    const int cq = threadIdx.x % quads, pl = threadIdx.x / quads, n = blockIdx.y, cpg = C / groups;
    if (pl >= lanes) return;
    const float inv_cnt = 1.0f / ((float)HW * (float)cpg);
    float mu[4], rs[4], ga[4], be[4], m1[4], m2[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int c = cq * 4 + j, g = c / cpg;
        const float2 m = __ldg(reinterpret_cast<const float2*>(mr) + (long long)n * groups + g);
        mu[j] = m.x; rs[j] = m.y; ga[j] = __ldg(gamma + c); be[j] = __ldg(beta + c);
        m1[j] = (float)(gsums[((long long)n * groups + g) * 2] * (double)inv_cnt);
        m2[j] = (float)(gsums[((long long)n * groups + g) * 2 + 1] * (double)inv_cnt);
    }
    const int p0 = blockIdx.x * pix_per_block, p1 = min(HW, p0 + pix_per_block);
    for (int p = p0 + pl; p < p1; p += lanes) {
        const long long o = ((long long)n * HW + p) * C + cq * 4;
        const float4 xv = __ldg(reinterpret_cast<const float4*>(x + o)), dv = __ldg(reinterpret_cast<const float4*>(dout + o));
        float4 av = make_float4(0.f, 0.f, 0.f, 0.f);
        if (add) av = __ldg(reinterpret_cast<const float4*>(add + o));
        const float xe[4] = {xv.x, xv.y, xv.z, xv.w}, de[4] = {dv.x, dv.y, dv.z, dv.w}, ae[4] = {av.x, av.y, av.z, av.w};
        float r[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float xh = (xe[j] - mu[j]) * rs[j];
            float dg = de[j];
            if (swish) dg *= swish_grad(xh * ga[j] + be[j]);
            r[j] = rs[j] * (dg * ga[j] - m1[j] - xh * m2[j]) + ae[j];
        }
        *reinterpret_cast<float4*>(dx + o) = make_float4(r[0], r[1], r[2], r[3]);
    }
}

// one warp per row
__global__ void __launch_bounds__(256) softmax_bwd_rows_kernel(const float* __restrict__ P, const float* __restrict__ dP, long long rows, int cols,
                                                               float* __restrict__ dS) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * 8 + warp;
    if (row >= rows) return;
    const float* p = P + row * cols;
    const float* d = dP + row * cols;
    float s = 0.f;
    for (int c = lane; c < cols; c += 32) s = fmaf(p[c], d[c], s);
    s = warp_sum(s);
    for (int c = lane; c < cols; c += 32) dS[row * cols + c] = p[c] * (d[c] - s);
}

__global__ void l1_grad_kernel(const float* __restrict__ x, const float* __restrict__ y, long long n, float scale, float* __restrict__ dy,
                               double* __restrict__ loss_sum) {
    __shared__ double sh[8];
    double ls = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float d = y[i] - x[i];
        ls += (double)fabsf(d);
        dy[i] = d > 0.f ? scale : (d < 0.f ? -scale : 0.f);       // torch.abs backward: sign(d), 0 at 0
    }
    for (int o = 16; o > 0; o >>= 1) ls += __shfl_xor_sync(0xffffffffu, ls, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = ls;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sh[w];
        atomicAdd(loss_sum, t);
    }
}

__global__ void lincomb3_kernel(float a, const float* __restrict__ x, float b, const float* __restrict__ y, float c, const float* __restrict__ z,
                                long long n, float* __restrict__ out) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        float v = a * x[i];
        if (y) v = fmaf(b, y[i], v);
        if (z) v = fmaf(c, z[i], v);
        out[i] = v;
    }
}

__global__ void sumpool2x2_kernel(const float* __restrict__ x, int N, int H, int W, int C, float* __restrict__ y) {      // x [N,2H,2W,C] -> y [N,H,W,C]
    const long long total = (long long)N * H * W * C;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        long long r = i / C;
        const int xx = (int)(r % W);
        r /= W;
        const int yy = (int)(r % H), n = (int)(r / H);
        const long long W2 = 2 * (long long)W;
        const long long o = (((long long)n * 2 * H + 2 * yy) * W2 + 2 * xx) * C + c;
        y[i] = (x[o] + x[o + C]) + (x[o + W2 * C] + x[o + W2 * C + C]);
    }
}

// torch.optim.Adam (no weight decay, no amsgrad): m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2; p -= lr / bc1 * m / (sqrt(v) / sqrt(bc2) + eps)
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n,
                            float lr, float b1, float b2, float eps, float bc1, float bc2_sqrt, float grad_scale) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float gi = g[i] * grad_scale;
        const float mi = m[i] + (1.0f - b1) * (gi - m[i]);          // lerp form used by torch (exp_avg.lerp_(grad, 1 - beta1))
        const float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
        m[i] = mi;
        v[i] = vi;
        const float denom = sqrtf(vi) / bc2_sqrt + eps;
        p[i] -= (lr / bc1) * (mi / denom);
    }
}


// ---- transformer training step (models/migt.py:464-505): LayerNorm / GELU / embedding / loss backward, AdamWeightDecay --------------

// LayerNorm backward, one warp per row (any D <= 4096: the [2][D] shared partial sums fit the default 48 KB), columns strided over
// the warp's lanes: dx = rstd (dy g - mean(dy g) - xhat mean(dy g xhat)) + add;
// dgamma / dbeta partial sums per block in shared memory, then one atomic per column and block
__global__ void __launch_bounds__(256) layernorm_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dy, const float* __restrict__ gamma,
                                                            const float* __restrict__ add, long long rows, int D, float eps,
                                                            float* __restrict__ dgamma, float* __restrict__ dbeta, float* __restrict__ dx) {
    extern __shared__ float shs[];            // [2][D]
    float* sg = shs;
    float* sb = shs + D;
    for (int i = threadIdx.x; i < 2 * D; i += 256) shs[i] = 0.f;
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * 8 + warp;
    if (row < rows) {
        const float* xr = x + row * D;
        const float* dr = dy + row * D;
        float s = 0.f;
        for (int c = lane; c < D; c += 32) s += xr[c];
        const float mean = warp_sum(s) / (float)D;
        float ss = 0.f;
        for (int c = lane; c < D; c += 32) { const float t = xr[c] - mean; ss = fmaf(t, t, ss); }
        const float rstd = rsqrtf(warp_sum(ss) / (float)D + eps);
        float m1 = 0.f, m2 = 0.f;
        for (int c = lane; c < D; c += 32) {
            const float xh = (xr[c] - mean) * rstd, dg = dr[c] * __ldg(gamma + c);
            m1 += dg;
            m2 = fmaf(dg, xh, m2);
            atomicAdd(sb + c, dr[c]);
            atomicAdd(sg + c, dr[c] * xh);
        }
        m1 = warp_sum(m1) / (float)D;
        m2 = warp_sum(m2) / (float)D;
        for (int c = lane; c < D; c += 32) {
            const float xh = (xr[c] - mean) * rstd, dg = dr[c] * __ldg(gamma + c);
            float v = rstd * (dg - m1 - xh * m2);
            if (add) v += add[row * D + c];
            dx[row * D + c] = v;
        }
    }
    __syncthreads();
    for (int c = threadIdx.x; c < D; c += 256) {
        atomicAdd(dgamma + c, sg[c]);
        atomicAdd(dbeta + c, sb[c]);
    }
}

__global__ void gelu_fwd_kernel(const float* __restrict__ x, long long n, float* __restrict__ y) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) y[i] = vf_gelu_erf(x[i]);
}

__global__ void gelu_bwd_kernel(const float* __restrict__ pre, const float* __restrict__ dy, long long n, float* __restrict__ out) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float xv = pre[i];
        const float cdf = 0.5f * (1.0f + erff(xv * 0.70710678118654752440f));
        const float pdf = 0.39894228040143267794f * expf(-0.5f * xv * xv);
        out[i] = dy[i] * (cdf + xv * pdf);
    }
}

// backward of migt_embed_kernel: dh [BT*L, d] -> dwte[id] += dh (atomic scatter), dwpe[l] += dh, dpose[bt] += dh
__global__ void embed_bwd_kernel(const float* __restrict__ dh, const int32_t* __restrict__ ids, int fixed_token, long long BT, int L, int d,
                                 float* __restrict__ dwte, float* __restrict__ dwpe, float* __restrict__ dpose) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= BT * L * d) return;
    const int c = (int)(i % d);
    const long long tok = i / d;
    const int l = (int)(tok % L);
    const long long bt = tok / L;
    int id = ids ? ids[tok] : -1;
    if (id < 0) id = fixed_token;
    const float g = dh[i];
    atomicAdd(dwte + (long long)id * d + c, g);
    atomicAdd(dwpe + (long long)l * d + c, g);
    if (dpose) atomicAdd(dpose + bt * d + c, g);
}

// d/dlogits of sum_rows w[row] * CE_smooth(logits[row], label[row]): w (softmax - (1-s) onehot - s/cols); one warp per row
__global__ void __launch_bounds__(256) ce_grad_kernel(const float* __restrict__ logits, const int32_t* __restrict__ labels, const float* __restrict__ w,
                                                      long long rows, int cols, float smoothing, float* __restrict__ dlogits) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * 8 + warp;
    if (row >= rows) return;
    const float* x = logits + row * cols;
    const float wr = w[row];
    float mx = -INFINITY;
    for (int c = lane; c < cols; c += 32) mx = fmaxf(mx, x[c]);
    mx = warp_max(mx);
    float se = 0.f;
    for (int c = lane; c < cols; c += 32) se += expf(x[c] - mx);
    se = warp_sum(se);
    const int lab = labels[row];
    for (int c = lane; c < cols; c += 32) {
        const float pr = expf(x[c] - mx) / se;
        dlogits[row * cols + c] = wr * (pr - (c == lab ? 1.0f - smoothing : 0.f) - smoothing / (float)cols);
    }
}

// d/draw of sum_rows w[row] * (pos_loss + ori_loss) (pose_loss_kernel in vf_misc.cu): pos = mean_3 (y m - r)^2, ori = mean_4 (y - r)^2
__global__ void pose_loss_grad_kernel(const float* __restrict__ raw, const float* __restrict__ poses, const float* __restrict__ w, long long rows,
                                      int tokens_per_view, float mult, float pos_scale, float ori_scale, float* __restrict__ draw) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows) return;
    const float* r = raw + i * 7;
    const float* y = poses + (i / tokens_per_view) * 7;
    const float wp = w[i] * pos_scale, wo = w[i] * ori_scale;
#pragma unroll
    for (int j = 0; j < 3; ++j) draw[i * 7 + j] = wp * (-2.0f / 3.0f) * (y[j] * mult - r[j]);
#pragma unroll
    for (int j = 3; j < 7; ++j) draw[i * 7 + j] = wo * (-2.0f / 4.0f) * (y[j] - r[j]);
}

// Keras Adam (TF 2.4 optimizer_v2/adam.py, non-amsgrad): lr_t = lr sqrt(1-b2^t)/(1-b1^t); m += (g-m)(1-b1); v += (g^2-v)(1-b2);
// p -= lr_t m / (sqrt(v) + eps);  preceded by the decoupled decay p -= lr wd p of AdamWeightDecay (models/utils.py:507-515) when wd != 0
__global__ void adamw_keras_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n,
                                   float lr, float lr_t, float b1, float b2, float eps, float wd, float grad_scale, float clip_scale) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float gi = g[i] * grad_scale * clip_scale;
        float pi = p[i];
        pi -= lr * wd * pi;
        const float mi = m[i] + (gi - m[i]) * (1.0f - b1);
        const float vi = v[i] + (gi * gi - v[i]) * (1.0f - b2);
        m[i] = mi;
        v[i] = vi;
        p[i] = pi - lr_t * mi / (sqrtf(vi) + eps);
    }
}

__global__ void sumsq_kernel(const float* __restrict__ x, long long n, double* __restrict__ out) {
    __shared__ double sh[8];
    double s = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) s += (double)x[i] * (double)x[i];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sh[w];
        atomicAdd(out, t);
    }
}

// inverted dropout with a counter-based hash (no state): keep = hash(seed, i) >= rate * 2^32; y = keep ? x / (1 - rate) : 0.
// The backward pass calls it again on the gradient with the same (seed, offset).
__device__ __forceinline__ uint32_t mix32(uint64_t k) {
    k ^= k >> 33; k *= 0xff51afd7ed558ccdULL; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ULL; k ^= k >> 33;
    return (uint32_t)k;
}
__global__ void dropout_kernel(const float* __restrict__ x, long long n, float rate, unsigned long long seed, float* __restrict__ y) {
    const uint32_t thr = (uint32_t)fminf(rate * 4294967296.0f, 4294967295.0f);
    const float sc = 1.0f / (1.0f - rate);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        y[i] = mix32(seed * 0x9E3779B97F4A7C15ULL + (unsigned long long)i) >= thr ? x[i] * sc : 0.f;
}

// ---- operands of the tensor-core weight gradient (vf_tc_gemm, exact split-fp16 GEMM with K = pixels) ----
// x NHWC fp32 [N,H,W,C] -> out fp16 [copies * C][2][L]: row (k * C + c) holds hi(x) at [0, L) and lo(x) at [L, 2L) (the exact GEMM's split
// operand), indexed by the linear position q = (n (H+2) + y + 1) * pitch + x + 1 of the ZERO-PADDED image (row pitch >= W + 2).  Copy k
// (k = 0 .. copies-1) is shifted by k - copies/2 pixels: column margin + q - (k - copies/2) <- x[n,y,x,c], so that reading copy k at
// column margin + q yields xpad[q + (k - copies/2)].  TMA wants 16-byte aligned box starts, hence the horizontal tap shifts are baked into
// three copies and only the vertical ones (multiples of the pitch, a multiple of 8) are left to the GEMM's K offsets.
// Everything that is not written here (borders, pitch padding, margins, tail) must be zero — callers clear the buffer first.
// Tile: 32 channels x 64 pixels through shared memory (coalesced 128-byte reads along C, contiguous writes along q).
__global__ void __launch_bounds__(256) pad_transpose_split_kernel(const float* __restrict__ x, int N, int H, int W, int C, int pitch, int copies,
                                                                  long long margin, long long L, __half* __restrict__ out) {
    __shared__ float tile[64][33];
    const long long p0 = (long long)blockIdx.x * 64;             // first unpadded pixel (n, y, x flattened) of the tile
    const int c0 = blockIdx.y * 32;
    const long long P = (long long)N * H * W;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = warp; i < 64; i += 8) {
        const long long pix = p0 + i;
        tile[i][lane] = (pix < P && c0 + lane < C) ? x[pix * C + c0 + lane] : 0.f;
    }
    __syncthreads();
    for (int cc = warp; cc < 32; cc += 8) {
        if (c0 + cc >= C) continue;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int i = lane + 32 * h;
            const long long pix = p0 + i;
            if (pix >= P) continue;
            const int xx = (int)(pix % W);
            const long long t = pix / W;
            const int yy = (int)(t % H);
            const long long n = t / H;
            const long long q = pitch ? (n * (H + 2) + yy + 1) * (long long)pitch + xx + 1 : pix;      // pitch 0: plain transpose
            const float v = tile[i][cc];
            const __half hi = __float2half_rn(v);
            const __half lo = __float2half_rn((v - __half2float(hi)) * 2048.0f);
            for (int k = 0; k < copies; ++k) {
                __half* row = out + ((long long)k * C + c0 + cc) * 2 * L;
                const long long col = margin + q - (k - copies / 2);
                row[col] = hi;
                row[L + col] = lo;
            }
        }
    }
}

// out[g * n + i] (+)= sum_s partial[(g * splits + s) * n + i]   — folds the split-K partial products of the weight-gradient GEMM
__global__ void sum_splits_kernel(const float* __restrict__ partial, int groups, int splits, long long n, int accumulate, float* __restrict__ out) {
    const long long total = (long long)groups * n;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long g = i / n, r = i - g * n;
        const float* src = partial + (g * splits) * n + r;
        float acc = 0.f;
        for (int s = 0; s < splits; ++s) acc += src[(long long)s * n];
        out[i] = accumulate ? out[i] + acc : acc;
    }
}

}  // namespace

extern "C" int vf_pad_transpose_split(const float* x, int N, int H, int W, int C, int pitch, int copies, int64_t margin, int64_t L,
                                      void* out_f16, vf_stream_t s) {
    VF_CHECK_ARG(x && out_f16 && N > 0 && H > 0 && W > 0 && C > 0, "vf_pad_transpose_split: bad args");
    VF_CHECK_ARG((pitch >= W + 2 || (pitch == 0 && copies == 1)) && (copies == 1 || copies == 3) && margin >= copies / 2,
                 "vf_pad_transpose_split: pitch / copies / margin");
    VF_CHECK_ARG(L >= margin + (pitch ? (int64_t)N * (H + 2) * pitch : (int64_t)N * H * W) + copies / 2, "vf_pad_transpose_split: row length L too small");
    const long long P = (long long)N * H * W;
    dim3 grid((unsigned)((P + 63) / 64), (unsigned)((C + 31) / 32));
    pad_transpose_split_kernel<<<grid, 256, 0, vf_s(s)>>>(x, N, H, W, C, pitch, copies, margin, L, reinterpret_cast<__half*>(out_f16));
    VF_CHECK_LAUNCH("vf_pad_transpose_split");
    return VF_OK;
}
extern "C" int vf_sum_splits(const float* partial, int groups, int splits, int64_t n, int accumulate, float* out, vf_stream_t s) {
    VF_CHECK_ARG(partial && out && groups > 0 && splits > 0 && n > 0, "vf_sum_splits: bad args");
    { long long tot_ = (long long)groups * n; unsigned g_ = (unsigned)((tot_ + 255) / 256 < 148 * 16 ? (tot_ + 255) / 256 : 148 * 16);
    sum_splits_kernel<<<g_, 256, 0, vf_s(s)>>>(partial, groups, splits, n, accumulate, out); }
    VF_CHECK_LAUNCH("vf_sum_splits");
    return VF_OK;
}

extern "C" int vf_conv_wgrad(const float* x, const float* dy, int N, int H, int W, int Cin, int OH, int OW, int Cout, int KH, int KW,
                             int stride, int pad_t, int pad_l, int upsample2x, int64_t so_k, int64_t so_n, float* dw, vf_stream_t s) {
    VF_CHECK_ARG(x && dy && dw && N > 0 && Cin > 0 && Cout > 0 && KH > 0 && KW > 0 && KH * KW <= 65535, "vf_conv_wgrad: bad args");
    const long long total = (long long)N * OH * OW;
    if (total == 0) return VF_OK;
    const int tiles = ((Cin + WT - 1) / WT) * ((Cout + WT - 1) / WT);
    // enough blocks to fill the machine a few times over, at least 256 pixels per block
    long long chunks = (148LL * 16 + (long long)KH * KW * tiles - 1) / ((long long)KH * KW * tiles);
    long long ppb = (total + chunks - 1) / chunks;
    if (ppb < 256) ppb = 256;
    ppb = (ppb + WP - 1) / WP * WP;
    chunks = (total + ppb - 1) / ppb;
    VF_CHECK_ARG(tiles <= 65535, "vf_conv_wgrad: too many channel tiles");
    dim3 grid((unsigned)chunks, KH * KW, tiles);
    conv_wgrad_kernel<<<grid, 256, 0, vf_s(s)>>>(x, dy, N, H, W, Cin, OH, OW, Cout, KH, KW, stride, pad_t, pad_l, upsample2x, ppb, so_k, so_n, dw);
    VF_CHECK_LAUNCH("vf_conv_wgrad");
    return VF_OK;
}

extern "C" int vf_col_sums(const float* x, int64_t rows, int C, float* out, vf_stream_t s) {
    VF_CHECK_ARG(x && out && C > 0, "vf_col_sums: bad args");
    if (rows == 0) return VF_OK;
    long long chunks = (rows + 1023) / 1024;
    if (chunks > 1024) chunks = 1024;
    const long long rpb = (rows + chunks - 1) / chunks;
    chunks = (rows + rpb - 1) / rpb;
    col_sums_kernel<<<dim3((C + 31) / 32, (unsigned)chunks), 256, 0, vf_s(s)>>>(x, rows, C, rpb, out);
    VF_CHECK_LAUNCH("vf_col_sums");
    return VF_OK;
}

extern "C" int vf_groupnorm_bwd(const float* x, const float* dout, const float* mean_rstd, const float* gamma, const float* beta, int N,
                                int HW, int C, int groups, int swish, const float* add, double* gsums, float* dgamma, float* dbeta,
                                float* dx, vf_stream_t s) {
    VF_CHECK_ARG(x && dout && mean_rstd && gamma && beta && gsums && dgamma && dbeta && dx, "vf_groupnorm_bwd: null pointer");
    VF_CHECK_ARG(C % groups == 0 && C % 4 == 0 && C / 4 <= 256 && 256 % (C / 4) == 0 && N <= 65535, "vf_groupnorm_bwd: unsupported C=%d groups=%d", C, groups);
    if (N == 0 || HW == 0) return VF_OK;
    cudaError_t e = cudaMemsetAsync(gsums, 0, sizeof(double) * 2 * groups * N, vf_s(s));
    if (e != cudaSuccess) { vf_set_error("vf_groupnorm_bwd: memset: %s", cudaGetErrorString(e)); return VF_ERR_CUDA; }
    const int lanes = 256 / (C / 4);
    int ppb = lanes * 128;          // few, long blocks: the per-channel sums end in global atomics
    while (ppb > lanes * 4 && (long long)((HW + ppb - 1) / ppb) * N < 148 * 4) ppb >>= 1;
    dim3 grid((HW + ppb - 1) / ppb, N);
    gn_bwd_stats_kernel<<<grid, 256, sizeof(double) * 2 * groups + sizeof(float) * 2 * C, vf_s(s)>>>(x, dout, mean_rstd, gamma, beta, HW, C, groups, swish, ppb, gsums, dgamma, dbeta);
    VF_CHECK_LAUNCH("vf_groupnorm_bwd(stats)");
    int ppb2 = lanes * 16;          // the streaming pass keeps many short blocks in flight
    while (ppb2 > lanes * 4 && (long long)((HW + ppb2 - 1) / ppb2) * N < 148 * 8) ppb2 >>= 1;
    dim3 grid2((HW + ppb2 - 1) / ppb2, N);
    gn_bwd_apply_kernel<<<grid2, 256, 0, vf_s(s)>>>(x, dout, mean_rstd, gamma, beta, gsums, add, HW, C, groups, swish, ppb2, dx);
    VF_CHECK_LAUNCH("vf_groupnorm_bwd(apply)");
    return VF_OK;
}

extern "C" int vf_softmax_bwd_rows(const float* P, const float* dP, int64_t rows, int cols, float* dS, vf_stream_t s) {
    VF_CHECK_ARG(P && dP && dS && cols > 0, "vf_softmax_bwd_rows: bad args");
    if (rows == 0) return VF_OK;
    softmax_bwd_rows_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, vf_s(s)>>>(P, dP, rows, cols, dS);
    VF_CHECK_LAUNCH("vf_softmax_bwd_rows");
    return VF_OK;
}

extern "C" int vf_l1_grad(const float* x, const float* y, int64_t n, float scale, float* dy, double* loss_sum, vf_stream_t s) {
    VF_CHECK_ARG(x && y && dy && loss_sum, "vf_l1_grad: null pointer");
    if (n == 0) return VF_OK;
    long long blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    l1_grad_kernel<<<(unsigned)blocks, 256, 0, vf_s(s)>>>(x, y, n, scale, dy, loss_sum);
    VF_CHECK_LAUNCH("vf_l1_grad");
    return VF_OK;
}

extern "C" int vf_lincomb3(float a, const float* x, float b, const float* y, float c, const float* z, int64_t n, float* out, vf_stream_t s) {
    VF_CHECK_ARG(x && out, "vf_lincomb3: null pointer");
    if (n == 0) return VF_OK;
    long long blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    lincomb3_kernel<<<(unsigned)blocks, 256, 0, vf_s(s)>>>(a, x, b, y, c, z, n, out);
    VF_CHECK_LAUNCH("vf_lincomb3");
    return VF_OK;
}

extern "C" int vf_sumpool2x2(const float* x, int N, int H, int W, int C, float* y, vf_stream_t s) {
    VF_CHECK_ARG(x && y, "vf_sumpool2x2: null pointer");
    const long long total = (long long)N * H * W * C;
    if (total == 0) return VF_OK;
    long long blocks = (total + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    sumpool2x2_kernel<<<(unsigned)blocks, 256, 0, vf_s(s)>>>(x, N, H, W, C, y);
    VF_CHECK_LAUNCH("vf_sumpool2x2");
    return VF_OK;
}

extern "C" int vf_adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps, int step,
                       float grad_scale, vf_stream_t s) {
    VF_CHECK_ARG(p && g && m && v && step >= 1, "vf_adam: bad args");
    if (n == 0) return VF_OK;
    const float bc1 = 1.0f - powf(beta1, (float)step), bc2 = 1.0f - powf(beta2, (float)step);
    long long blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    adam_kernel<<<(unsigned)blocks, 256, 0, vf_s(s)>>>(p, g, m, v, n, lr, beta1, beta2, eps, bc1, sqrtf(bc2), grad_scale);
    VF_CHECK_LAUNCH("vf_adam");
    return VF_OK;
}

static unsigned grid_for(long long n) {
    long long b = (n + 255) / 256;
    return (unsigned)(b > 148 * 16 ? 148 * 16 : b);
}

extern "C" int vf_layernorm_bwd(const float* x, const float* dy, const float* gamma, const float* add, int64_t rows, int D, float eps,
                                float* dgamma, float* dbeta, float* dx, vf_stream_t s) {
    VF_CHECK_ARG(x && dy && gamma && dgamma && dbeta && dx && D > 0 && D <= 4096, "vf_layernorm_bwd: bad args");
    if (rows == 0) return VF_OK;
    layernorm_bwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 2 * D * sizeof(float), vf_s(s)>>>(x, dy, gamma, add, rows, D, eps, dgamma, dbeta, dx);
    VF_CHECK_LAUNCH("vf_layernorm_bwd");
    return VF_OK;
}
extern "C" int vf_gelu_fwd(const float* x, int64_t n, float* y, vf_stream_t s) {
    VF_CHECK_ARG(x && y, "vf_gelu_fwd: null pointer");
    if (n == 0) return VF_OK;
    gelu_fwd_kernel<<<grid_for(n), 256, 0, vf_s(s)>>>(x, n, y);
    VF_CHECK_LAUNCH("vf_gelu_fwd");
    return VF_OK;
}
extern "C" int vf_gelu_bwd(const float* pre, const float* dy, int64_t n, float* out, vf_stream_t s) {
    VF_CHECK_ARG(pre && dy && out, "vf_gelu_bwd: null pointer");
    if (n == 0) return VF_OK;
    gelu_bwd_kernel<<<grid_for(n), 256, 0, vf_s(s)>>>(pre, dy, n, out);
    VF_CHECK_LAUNCH("vf_gelu_bwd");
    return VF_OK;
}
extern "C" int vf_migt_embed_bwd(const float* dh, const int32_t* ids, int fixed_token, int64_t BT, int L, int d, float* dwte, float* dwpe,
                                 float* dpose, vf_stream_t s) {
    VF_CHECK_ARG(dh && dwte && dwpe, "vf_migt_embed_bwd: null pointer");
    const long long total = BT * L * d;
    if (total == 0) return VF_OK;
    embed_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, vf_s(s)>>>(dh, ids, fixed_token, BT, L, d, dwte, dwpe, dpose);
    VF_CHECK_LAUNCH("vf_migt_embed_bwd");
    return VF_OK;
}
extern "C" int vf_cross_entropy_grad(const float* logits, const int32_t* labels, const float* row_weight, int64_t rows, int cols,
                                     float smoothing, float* dlogits, vf_stream_t s) {
    VF_CHECK_ARG(logits && labels && row_weight && dlogits && cols > 0, "vf_cross_entropy_grad: bad args");
    if (rows == 0) return VF_OK;
    ce_grad_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, vf_s(s)>>>(logits, labels, row_weight, rows, cols, smoothing, dlogits);
    VF_CHECK_LAUNCH("vf_cross_entropy_grad");
    return VF_OK;
}
extern "C" int vf_pose_loss_grad(const float* raw, const float* poses, const float* row_weight, int64_t rows, int tokens_per_view,
                                 float pose_multiplier, float pos_scale, float ori_scale, float* draw, vf_stream_t s) {
    VF_CHECK_ARG(raw && poses && row_weight && draw && tokens_per_view > 0, "vf_pose_loss_grad: bad args");
    if (rows == 0) return VF_OK;
    pose_loss_grad_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, vf_s(s)>>>(raw, poses, row_weight, rows, tokens_per_view, pose_multiplier, pos_scale, ori_scale, draw);
    VF_CHECK_LAUNCH("vf_pose_loss_grad");
    return VF_OK;
}
extern "C" int vf_adamw_keras(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                              float weight_decay, int step, float grad_scale, float clip_scale, vf_stream_t s) {
    VF_CHECK_ARG(p && g && m && v && step >= 1, "vf_adamw_keras: bad args");
    if (n == 0) return VF_OK;
    const float lr_t = lr * sqrtf(1.0f - powf(beta2, (float)step)) / (1.0f - powf(beta1, (float)step));
    adamw_keras_kernel<<<grid_for(n), 256, 0, vf_s(s)>>>(p, g, m, v, n, lr, lr_t, beta1, beta2, eps, weight_decay, grad_scale, clip_scale);
    VF_CHECK_LAUNCH("vf_adamw_keras");
    return VF_OK;
}
extern "C" int vf_sumsq(const float* x, int64_t n, double* out, vf_stream_t s) {
    VF_CHECK_ARG(x && out, "vf_sumsq: null pointer");
    if (n == 0) return VF_OK;
    sumsq_kernel<<<grid_for(n), 256, 0, vf_s(s)>>>(x, n, out);
    VF_CHECK_LAUNCH("vf_sumsq");
    return VF_OK;
}
extern "C" int vf_dropout(const float* x, int64_t n, float rate, uint64_t seed, float* y, vf_stream_t s) {
    VF_CHECK_ARG(x && y && rate >= 0.f && rate < 1.f, "vf_dropout: bad args");
    if (n == 0) return VF_OK;
    dropout_kernel<<<grid_for(n), 256, 0, vf_s(s)>>>(x, n, rate, seed, y);
    VF_CHECK_LAUNCH("vf_dropout");
    return VF_OK;
}
