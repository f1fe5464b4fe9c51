// Plane encoder: packed positions -> the 112x8x8 network input.
//
// Replaces `_encode` / `BoardHistory::view` / `Board::rotate` / `encode_pieces`
// (reference src/chess.rs:845-877, 828-842, 594-621, 623-650) and the host-side cast +
// HWC->CHW permute of the backends (src/backends/torch.rs:115-123, onnx.rs:66-72).
//
// One warp per position.  The warp turns the 8 x 8 bitboard words of a position into 112
// per-channel 64-bit square masks (rank flip for Black = one byte swap per mask), keeps
// them in shared memory, then streams the [64 squares][C] row-major tile out with 16-byte
// stores so that every store instruction of the warp covers 512 contiguous bytes.
// Channel c of square s is bit s of mask c:  c = 14*t + k,
//   k 0..5  side-to-move's P,N,B,R,Q,K   k 6..11 opponent's   k 12 rep>=2   k 13 rep>=3
// "side to move" is that of the CURRENT position for every history slot (src/chess.rs:871).
#include "common.cuh"

#include <cuda_fp8.h>

namespace scb {

constexpr int ENC_WARPS = 4;

__device__ __forceinline__ uint64_t bswap64(uint64_t x)
{
    uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
    return ((uint64_t)__byte_perm(lo, 0, 0x0123) << 32) | (uint64_t)__byte_perm(hi, 0, 0x0123);
}

// builds masks[128] for one position (lanes cooperate); masks 112..127 are zero
__device__ __forceinline__ void build_masks(const sc_position *p, uint64_t *slots /*smem[64]*/,
                                            uint64_t *masks /*smem[128]*/, int lane)
{
    const uint64_t *src = reinterpret_cast<const uint64_t *>(p->slot);
    slots[lane] = src[lane];
    slots[lane + 32] = src[lane + 32];
    const int turn = p->meta[0];
    const int n_hist = p->n_hist;
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 4; i++) {
        int c = lane + 32 * i;
        uint64_t m = 0;
        int t = c / 14, k = c - 14 * t;
        if (c < SC_N_PLANES && t < n_hist) {
            const uint64_t *s = slots + 8 * t;
            if (k < 12) {
                uint64_t all = s[0] | s[1] | s[2] | s[3] | s[4] | s[5];
                uint64_t white = s[6];
                uint64_t own = turn ? white : (all & ~white);
                uint64_t opp = all & ~own;
                m = (k < 6) ? (s[k] & own) : (s[k - 6] & opp);
                if (!turn) m = bswap64(m);  // Square::rotate: rank -> 7 - rank (chess.rs:504-509)
            } else {
                m = ((s[7] >> (k - 12)) & 1ULL) ? ~0ULL : 0ULL;
            }
        }
        masks[c] = m;
    }
    __syncwarp();
}

__global__ void __launch_bounds__(ENC_WARPS * 32) encode_i8_kernel(const sc_position *__restrict__ pos, int n,
                                                                   int8_t *__restrict__ out,
                                                                   int32_t *__restrict__ meta_out)
{
    __shared__ uint64_t s_slots[ENC_WARPS][64];
    __shared__ uint64_t s_masks[ENC_WARPS][128];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * ENC_WARPS + warp;
    if (b >= n) return;
    build_masks(pos + b, s_slots[warp], s_masks[warp], lane);
    const uint64_t *masks = s_masks[warp];
    uint4 *dst = reinterpret_cast<uint4 *>(out + (size_t)b * 64 * SC_N_PLANES);
    // 64 rows x 7 chunks of 16 channels
    for (int idx = lane; idx < 64 * 7; idx += 32) {
        int s = idx / 7, c0 = (idx - s * 7) * 16;
        uint32_t w[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            uint32_t v = 0;
#pragma unroll
            for (int q = 0; q < 4; q++) v |= (uint32_t)((masks[c0 + 4 * j + q] >> s) & 1ULL) << (8 * q);
            w[j] = v;
        }
        dst[idx] = make_uint4(w[0], w[1], w[2], w[3]);
    }
    if (lane < SC_N_META) meta_out[b * SC_N_META + lane] = pos[b].meta[lane];
}

__global__ void __launch_bounds__(ENC_WARPS * 32) encode_f32_kernel(const sc_position *__restrict__ pos, int n,
                                                                    float *__restrict__ out,
                                                                    float *__restrict__ meta_out)
{
    __shared__ uint64_t s_slots[ENC_WARPS][64];
    __shared__ uint64_t s_masks[ENC_WARPS][128];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * ENC_WARPS + warp;
    if (b >= n) return;
    build_masks(pos + b, s_slots[warp], s_masks[warp], lane);
    const uint64_t *masks = s_masks[warp];
    float4 *dst = reinterpret_cast<float4 *>(out + (size_t)b * 64 * C_IN);
    for (int idx = lane; idx < 64 * 28; idx += 32) {
        int s = idx / 28, c0 = (idx - s * 28) * 4;
        float4 v;
        v.x = (float)((masks[c0 + 0] >> s) & 1ULL);
        v.y = (float)((masks[c0 + 1] >> s) & 1ULL);
        v.z = (float)((masks[c0 + 2] >> s) & 1ULL);
        v.w = (float)((masks[c0 + 3] >> s) & 1ULL);
        dst[idx] = v;
    }
    if (lane < 8) meta_out[b * 8 + lane] = lane < SC_N_META ? (float)pos[b].meta[lane] : 0.f;
}

// 16-bit form (the network's own input, ONE = the bit pattern of 1.0: 0x3F80 bf16, 0x3C00 fp16): FOUR warps per
// position, 16 squares each.  The kernel is short (34 MB at 2048 leaves) and ends in a store stream, so it is bound by
// how many bytes are in flight when it starts: with one warp per position the 32 store instructions of a position were
// issued one after another by a single warp.
template <uint32_t ONE>
__global__ void __launch_bounds__(ENC_WARPS * 32) encode_16bit_kernel(const sc_position *__restrict__ pos, int n,
                                                                      uint16_t *__restrict__ out,
                                                                      float *__restrict__ meta_out)
{
    __shared__ uint64_t s_slots[64];
    __shared__ uint64_t s_masks[128];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x;
    if (b >= n) return;
    if (warp == 0) build_masks(pos + b, s_slots, s_masks, lane);
    __syncthreads();
    uint4 *dst = reinterpret_cast<uint4 *>(out + (size_t)b * 64 * C_IN_PAD);
    const int c0 = (lane & 15) * 8;
    uint64_t m[8];
#pragma unroll
    for (int j = 0; j < 8; j++) m[j] = s_masks[c0 + j];
    // two rows (2 x 256 B) per warp store instruction; this warp: squares [16 warp, 16 warp + 16)
#pragma unroll
    for (int it8 = 0; it8 < 8; it8++) {
        const int it = warp * 8 + it8;
        const int s = it * 2 + (lane >> 4);
        uint32_t w[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            uint32_t lo = (uint32_t)((m[2 * j] >> s) & 1ULL) * ONE;
            uint32_t hi = (uint32_t)((m[2 * j + 1] >> s) & 1ULL) * ONE;
            w[j] = lo | (hi << 16);
        }
        dst[it * 32 + lane] = make_uint4(w[0], w[1], w[2], w[3]);
    }
    if (warp == 0 && lane < 8) meta_out[b * 8 + lane] = lane < SC_N_META ? (float)pos[b].meta[lane] : 0.f;
}

// e4m3 form (fp8 mode; 1.0 = 0x38): the 16-bit kernel's work split, 8 bytes per lane and row
__global__ void __launch_bounds__(ENC_WARPS * 32) encode_e4m3_kernel(const sc_position *__restrict__ pos, int n,
                                                                     uint8_t *__restrict__ out,
                                                                     float *__restrict__ meta_out)
{
    __shared__ uint64_t s_slots[64];
    __shared__ uint64_t s_masks[128];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x;
    if (b >= n) return;
    if (warp == 0) build_masks(pos + b, s_slots, s_masks, lane);
    __syncthreads();
    uint2 *dst = reinterpret_cast<uint2 *>(out + (size_t)b * 64 * C_IN_PAD);
    const int c0 = (lane & 15) * 8;
    uint64_t m[8];
#pragma unroll
    for (int j = 0; j < 8; j++) m[j] = s_masks[c0 + j];
#pragma unroll
    for (int it8 = 0; it8 < 8; it8++) {
        const int it = warp * 8 + it8;
        const int s = it * 2 + (lane >> 4);
        uint32_t w[2] = {0u, 0u};
#pragma unroll
        for (int j = 0; j < 8; j++) w[j >> 2] |= (uint32_t)((m[j] >> s) & 1ULL) * 0x38u << (8 * (j & 3));
        dst[it * 32 + lane] = make_uint2(w[0], w[1]);
    }
    if (warp == 0 && lane < 8) meta_out[b * 8 + lane] = lane < SC_N_META ? (float)pos[b].meta[lane] : 0.f;
}

int launch_encode_i8(const sc_position *d_pos, int n, int8_t *out, int32_t *meta_out, cudaStream_t st)
{
    if (n <= 0) return SC_OK;
    encode_i8_kernel<<<(n + ENC_WARPS - 1) / ENC_WARPS, ENC_WARPS * 32, 0, st>>>(d_pos, n, out, meta_out);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

int launch_encode_f32(const sc_position *d_pos, int n, float *out, float *meta_out, cudaStream_t st)
{
    if (n <= 0) return SC_OK;
    encode_f32_kernel<<<(n + ENC_WARPS - 1) / ENC_WARPS, ENC_WARPS * 32, 0, st>>>(d_pos, n, out, meta_out);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

int launch_encode_bf16(const sc_position *d_pos, int n, __nv_bfloat16 *out, float *meta_out, cudaStream_t st)
{
    if (n <= 0) return SC_OK;
    encode_16bit_kernel<0x3F80u><<<n, ENC_WARPS * 32, 0, st>>>(d_pos, n, reinterpret_cast<uint16_t *>(out), meta_out);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

int launch_encode_fp16(const sc_position *d_pos, int n, __half *out, float *meta_out, cudaStream_t st)
{
    if (n <= 0) return SC_OK;
    encode_16bit_kernel<0x3C00u><<<n, ENC_WARPS * 32, 0, st>>>(d_pos, n, reinterpret_cast<uint16_t *>(out), meta_out);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

int launch_encode_e4m3(const sc_position *d_pos, int n, uint8_t *out, float *meta_out, cudaStream_t st)
{
    if (n <= 0) return SC_OK;
    encode_e4m3_kernel<<<n, ENC_WARPS * 32, 0, st>>>(d_pos, n, out, meta_out);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

// ---- NCHW float (what the reference backends feed the net) -> NHWC ------------------------
template <typename T> __device__ __forceinline__ T cvt(float v);
template <> __device__ __forceinline__ float cvt<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 cvt<__nv_bfloat16>(float v) { return __float2bfloat16(v); }
template <> __device__ __forceinline__ __half cvt<__half>(float v) { return __float2half_rn(v); }
// e4m3, round to nearest even, satfinite (+-448)
template <> __device__ __forceinline__ __nv_fp8_e4m3 cvt<__nv_fp8_e4m3>(float v) { return __nv_fp8_e4m3(v); }

template <typename T, int LD>
__global__ void __launch_bounds__(256) nchw_to_nhwc_kernel(const float *__restrict__ in, int n, T *__restrict__ out)
{
    __shared__ float tile[64][SC_N_PLANES + 1];
    const int b = blockIdx.x;
    const float *src = in + (size_t)b * SC_N_PLANES * 64;
    for (int i = threadIdx.x; i < SC_N_PLANES * 64; i += 256) {
        int c = i >> 6, s = i & 63;
        tile[s][c] = src[i];
    }
    __syncthreads();
    T *dst = out + (size_t)b * 64 * LD;
    for (int i = threadIdx.x; i < 64 * LD; i += 256) {
        int s = i / LD, c = i - s * LD;
        dst[i] = cvt<T>(c < SC_N_PLANES ? tile[s][c] : 0.f);
    }
}

int launch_nchw_to_nhwc_f32(const float *in, int n, float *out, cudaStream_t st)
{
    if (n <= 0) return SC_OK;
    nchw_to_nhwc_kernel<float, C_IN><<<n, 256, 0, st>>>(in, n, out);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

int launch_nchw_to_nhwc_bf16(const float *in, int n, __nv_bfloat16 *out, cudaStream_t st)
{
    if (n <= 0) return SC_OK;
    nchw_to_nhwc_kernel<__nv_bfloat16, C_IN_PAD><<<n, 256, 0, st>>>(in, n, out);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

int launch_nchw_to_nhwc_fp16(const float *in, int n, __half *out, cudaStream_t st)
{
    if (n <= 0) return SC_OK;
    nchw_to_nhwc_kernel<__half, C_IN_PAD><<<n, 256, 0, st>>>(in, n, out);
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

int launch_nchw_to_nhwc_e4m3(const float *in, int n, uint8_t *out, cudaStream_t st)
{
    if (n <= 0) return SC_OK;
    nchw_to_nhwc_kernel<__nv_fp8_e4m3, C_IN_PAD><<<n, 256, 0, st>>>(in, n, reinterpret_cast<__nv_fp8_e4m3 *>(out));
    SCB_CUDA(cudaGetLastError());
    return SC_OK;
}

}  // namespace scb
