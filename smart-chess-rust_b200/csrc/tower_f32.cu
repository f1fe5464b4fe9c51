// FP32 parity mode of the policy/value network (py/module.py:135-154): plain FP32 FFMA
// implicit-GEMM convolutions, LayerNorm over channels, squeeze-excitation, heads.
// This is the mode held to the 1e-4 gate against the reference's fp32 semantics (the ONNX
// backend, src/backends/onnx.rs:66-73); tensor cores are deliberately not used here
// because TF32/bf16 operand rounding fails that gate (SURVEY section 7, "fp32 mode").
//
// Activations are NHWC fp32: [board][square = rank*8+file][channel].
#include "common.cuh"

namespace scb {

// ---------------------------------------------------------------------------------------
// Implicit GEMM:  out[M][N] = sum_tap sum_k A[src(m,tap)][k] * W[tap*K + k][n] + bias[n]
//   TAPS = 9: rows are (board, square); src shifts the square by (tap/3-1, tap%3-1) inside
//   the board, zero outside (3x3 conv, padding 1, cross-correlation like torch.conv2d).
//   TAPS = 1: plain row-major GEMM.
// 128x128 block tile, 16-deep K slices, 256 threads, 8x8 register tile per thread.
// ---------------------------------------------------------------------------------------
constexpr int GBM = 128, GBN = 128, GBK = 16;

// x = hi + mid + lo with three bf16 (8 significant bits each, successive round-to-nearest residuals): the operand
// planes of the tensor-core FP32 parity mode (tower_bf16.cu, EPI_F32)
__device__ __forceinline__ void split3_store(float x, __nv_bfloat16 *row, int c, int C)
{
    const __nv_bfloat16 h = __float2bfloat16_rn(x);
    float r = x - __bfloat162float(h);
    const __nv_bfloat16 m = __float2bfloat16_rn(r);
    r -= __bfloat162float(m);
    row[c] = h;
    row[C + c] = m;
    row[2 * C + c] = __float2bfloat16_rn(r);
}

template <int TAPS>
__global__ void __launch_bounds__(256) gemm_f32_kernel(const float *__restrict__ A, int lda,
                                                       const float *__restrict__ W, int ldw,
                                                       const float *__restrict__ bias, float *__restrict__ out,
                                                       int ldo, int M, int N, int K)
{
    __shared__ __align__(16) float As[GBK][GBM + 4];
    __shared__ __align__(16) float Bs[GBK][GBN];
    const int tid = threadIdx.x;
    const int m0 = blockIdx.x * GBM, n0 = blockIdx.y * GBN;
    // split-K (TAPS == 1 only): slice blockIdx.z of the K range, partial sums to out[z][M][ldo]
    A += (size_t)blockIdx.z * K;
    W += (size_t)blockIdx.z * K * ldw;
    out += (size_t)blockIdx.z * M * ldo;
    const int ty = tid >> 4, tx = tid & 15;

    // A loader: thread -> (row, 8 consecutive k)
    const int a_row = tid >> 1, a_k = (tid & 1) * 8;
    const int gm = m0 + a_row;
    const int board_row0 = (gm >> 6) << 6;
    const int sq = gm & 63, h = sq >> 3, w = sq & 7;
    // B loader: thread -> (k, 8 consecutive n)
    const int b_k = tid >> 4, b_n = (tid & 15) * 8;

    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
        for (int j = 0; j < 8; j++) acc[i][j] = 0.f;

    for (int tap = 0; tap < TAPS; tap++) {
        bool valid = gm < M;
        const float *arow;
        if (TAPS == 9) {
            int hh = h + tap / 3 - 1, ww = w + tap % 3 - 1;
            valid = valid && hh >= 0 && hh < 8 && ww >= 0 && ww < 8;
            arow = A + (size_t)(board_row0 + hh * 8 + ww) * lda;
        } else {
            arow = A + (size_t)gm * lda;
        }
        const float *wtap = W + (size_t)tap * K * ldw;
        for (int k0 = 0; k0 < K; k0 += GBK) {
            float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0;
            if (valid) {
                a0 = *reinterpret_cast<const float4 *>(arow + k0 + a_k);
                a1 = *reinterpret_cast<const float4 *>(arow + k0 + a_k + 4);
            }
            const float *wp = wtap + (size_t)(k0 + b_k) * ldw + n0 + b_n;
            float4 b0 = *reinterpret_cast<const float4 *>(wp);
            float4 b1 = *reinterpret_cast<const float4 *>(wp + 4);
            __syncthreads();
            As[a_k + 0][a_row] = a0.x; As[a_k + 1][a_row] = a0.y; As[a_k + 2][a_row] = a0.z; As[a_k + 3][a_row] = a0.w;
            As[a_k + 4][a_row] = a1.x; As[a_k + 5][a_row] = a1.y; As[a_k + 6][a_row] = a1.z; As[a_k + 7][a_row] = a1.w;
            *reinterpret_cast<float4 *>(&Bs[b_k][b_n]) = b0;
            *reinterpret_cast<float4 *>(&Bs[b_k][b_n + 4]) = b1;
            __syncthreads();
#pragma unroll
            for (int kk = 0; kk < GBK; kk++) {
                float4 x0 = *reinterpret_cast<const float4 *>(&As[kk][ty * 8]);
                float4 x1 = *reinterpret_cast<const float4 *>(&As[kk][ty * 8 + 4]);
                float4 y0 = *reinterpret_cast<const float4 *>(&Bs[kk][tx * 8]);
                float4 y1 = *reinterpret_cast<const float4 *>(&Bs[kk][tx * 8 + 4]);
                float a[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
                float b[8] = {y0.x, y0.y, y0.z, y0.w, y1.x, y1.y, y1.z, y1.w};
#pragma unroll
                for (int i = 0; i < 8; i++)
#pragma unroll
                    for (int j = 0; j < 8; j++) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 8; i++) {
        int m = m0 + ty * 8 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            int nn = n0 + tx * 8 + j;
            if (nn < N) out[(size_t)m * ldo + nn] = acc[i][j] + (bias ? bias[nn] : 0.f);
        }
    }
}

int launch_gemm_f32(int taps, const float *A, int lda, const float *W, int ldw, const float *bias, float *out,
                    int ldo, int M, int N, int K, cudaStream_t st, int n_splits)
{
    if (M <= 0) return SC_OK;
    if (n_splits > 1) {
        if (taps != 1 || bias || K % n_splits) {
            set_error("gemm_f32: split-K needs taps == 1, no bias and K divisible by the split count");
            return SC_E_INVAL;
        }
        K /= n_splits;
    } else
        n_splits = 1;
    if (K % GBK != 0 || ldw % GBN != 0 || (lda & 3)) {
        set_error("gemm_f32: K must be a multiple of 16, ldw of 128, lda of 4");
        return SC_E_INVAL;
    }
    dim3 grid((M + GBM - 1) / GBM, (N + GBN - 1) / GBN, n_splits);
    if (taps == 9)
        gemm_f32_kernel<9><<<grid, 256, 0, st>>>(A, lda, W, ldw, bias, out, ldo, M, N, K);
    else
        gemm_f32_kernel<1><<<grid, 256, 0, st>>>(A, lda, W, ldw, bias, out, ldo, M, N, K);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

// ---------------------------------------------------------------------------------------
// LayerNorm over channels of each (board, square) row, in place (timm LayerNorm2d,
// eps 1e-6), optional ReLU.  One warp per row; two-pass mean / variance in registers.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ln_f32_kernel(float *__restrict__ x, int rows, int C, int ld,
                                                     const float *__restrict__ gamma,
                                                     const float *__restrict__ beta, int relu,
                                                     __nv_bfloat16 *__restrict__ planes)
{
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= rows) return;
    float *p = x + (size_t)row * ld;
    float v[8];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        int c = lane + 32 * i;
        v[i] = c < C ? p[c] : 0.f;
        s += v[i];
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    float mean = s / (float)C;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        int c = lane + 32 * i;
        float d = c < C ? v[i] - mean : 0.f;
        q += d * d;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    float rstd = rsqrtf(q / (float)C + LN_EPS);
    if (!gamma) {  // layer without normalisation (BatchNorm folded into the convolution at export)
        mean = 0.f;
        rstd = 1.f;
    }
#pragma unroll
    for (int i = 0; i < 8; i++) {
        int c = lane + 32 * i;
        if (c < C) {
            float y = gamma ? (v[i] - mean) * rstd * gamma[c] + beta[c] : v[i];
            y = relu ? fmaxf(y, 0.f) : y;
            p[c] = y;
            if (planes) split3_store(y, planes + (size_t)row * 3 * C, c, C);
        }
    }
}

int launch_ln_f32(float *x, int rows, int C, int ld, const float *gamma, const float *beta, int relu,
                  cudaStream_t st, __nv_bfloat16 *planes)
{
    if (rows <= 0) return SC_OK;
    if (C > 256) {
        set_error("ln_f32: C > 256");
        return SC_E_INVAL;
    }
    ln_f32_kernel<<<(rows + 7) / 8, 256, 0, st>>>(x, rows, C, ld, gamma, beta, relu, planes);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

// ---------------------------------------------------------------------------------------
// Squeeze-excitation + residual + ReLU (py/module.py:43-45, torchvision SqueezeExcitation):
//   s = mean over the 64 squares of y[:, c];  h = relu(W1 s + b1);  g = sigmoid(W2 h + b2)
//   out = relu(g[c] * y + x)
// One block per board, thread c owns channel c.  w1t is [256][128] (input-major),
// w2t is [128][256].
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) se_res_f32_kernel(const float *__restrict__ y, const float *__restrict__ x,
                                                         float *__restrict__ out, const float *__restrict__ w1t,
                                                         const float *__restrict__ b1,
                                                         const float *__restrict__ w2t,
                                                         const float *__restrict__ b2,
                                                         __nv_bfloat16 *__restrict__ planes)
{
    __shared__ float s_mean[C_TOWER];
    __shared__ float s_hid[C_SE];
    const int b = blockIdx.x, c = threadIdx.x;
    const float *yb = y + (size_t)b * 64 * C_TOWER;
    float g = 1.f;  // w1t == nullptr: `use_se=False`, the block is relu(y + x)
    if (w1t) {
        float sum = 0.f;
        for (int s = 0; s < 64; s++) sum += yb[s * C_TOWER + c];
        s_mean[c] = sum * (1.f / 64.f);
        __syncthreads();
        if (c < C_SE) {
            float a = b1[c];
            for (int k = 0; k < C_TOWER; k++) a = fmaf(w1t[k * C_SE + c], s_mean[k], a);
            s_hid[c] = fmaxf(a, 0.f);
        }
        __syncthreads();
        g = b2[c];
        for (int k = 0; k < C_SE; k++) g = fmaf(w2t[k * C_TOWER + c], s_hid[k], g);
        g = 1.f / (1.f + expf(-g));
    }
    const float *xb = x + (size_t)b * 64 * C_TOWER;
    float *ob = out + (size_t)b * 64 * C_TOWER;
    for (int s = 0; s < 64; s++) {
        const float o = fmaxf(fmaf(g, yb[s * C_TOWER + c], xb[s * C_TOWER + c]), 0.f);
        ob[s * C_TOWER + c] = o;
        if (planes) split3_store(o, planes + ((size_t)b * 64 + s) * 3 * C_TOWER, c, C_TOWER);
    }
}

int launch_se_res_f32(const float *y, const float *x, float *out, int n, const float *w1t, const float *b1,
                      const float *w2t, const float *b2, cudaStream_t st, __nv_bfloat16 *planes)
{
    if (n <= 0) return SC_OK;
    se_res_f32_kernel<<<n, 256, 0, st>>>(y, x, out, w1t, b1, w2t, b2, planes);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

// ---------------------------------------------------------------------------------------
// Value head tail (py/module.py:95-106, :147-149): hidden = relu(sum_splits pre + W_meta
// meta + b1); v = tanh(w2 . hidden + b2) * (2*turn - 1).  One warp per leaf.
// ---------------------------------------------------------------------------------------
// SCALED (fp8 mode): the split sum is multiplied by the hidden unit's weight scale first, as in the fused tail
template <bool SCALED>
__global__ void __launch_bounds__(128) value_finish_kernel(const float *__restrict__ pre, int n_split, int n,
                                                           const float *__restrict__ meta,
                                                           const float *__restrict__ w_meta /*[7][128]*/,
                                                           const float *__restrict__ b1,
                                                           const float *__restrict__ w2,
                                                           const float *__restrict__ b2,
                                                           float *__restrict__ value_out,
                                                           const float *__restrict__ scale)
{
    // lane = hidden units 4 lane .. 4 lane + 3: one coalesced 512-byte row per split.  The arithmetic (split-order sum,
    // meta fma chain, + b1, ReLU, fma with w2 over the lane's four units, xor-shuffle sum) is, operation for operation,
    // the fused tail of the bf16 value-FC GEMM (tower_bf16.cu, EPI_RAW): small batches use that one, large batches
    // this kernel, and a leaf's value must not depend on which.
    const int b = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= n) return;
    const float *mt = meta + b * 8;
    float4 h = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int sp = 0; sp < n_split; sp++) {
        const float4 p = __ldcg(reinterpret_cast<const float4 *>(pre + ((size_t)sp * n + b) * N_VALUE_HIDDEN) + lane);
        h.x += p.x;
        h.y += p.y;
        h.z += p.z;
        h.w += p.w;
    }
    float hv[4] = {h.x, h.y, h.z, h.w};
    if constexpr (SCALED)
#pragma unroll
        for (int i = 0; i < 4; i++) hv[i] = __fmul_rn(hv[i], scale[4 * lane + i]);
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int j = 4 * lane + i;
#pragma unroll
        for (int k = 0; k < SC_N_META; k++) hv[i] = fmaf(w_meta[k * N_VALUE_HIDDEN + j], mt[k], hv[i]);
        acc = fmaf(w2[j], fmaxf(hv[i] + b1[j], 0.f), acc);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) value_out[b] = tanhf(acc + b2[0]) * (mt[0] * 2.f - 1.f);
}

int launch_value_finish(const float *hidden_pre, int n_split, int n, const float *meta, const float *w_meta,
                        const float *b1, const float *w2, const float *b2, float *value_out, cudaStream_t st,
                        const float *scale)
{
    if (n <= 0) return SC_OK;
    if (scale)
        value_finish_kernel<true><<<(n + 3) / 4, 128, 0, st>>>(hidden_pre, n_split, n, meta, w_meta, b1, w2, b2, value_out, scale);
    else
        value_finish_kernel<false><<<(n + 3) / 4, 128, 0, st>>>(hidden_pre, n_split, n, meta, w_meta, b1, w2, b2, value_out, nullptr);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

}  // namespace scb
