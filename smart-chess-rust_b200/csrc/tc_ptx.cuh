// PTX wrappers (mbarrier, TMA, tcgen05 / TMEM, cluster) and small warp-level helpers shared by the tcgen05 kernels
// of tower_bf16.cu (throughput: CTA pairs, whole tower per launch) and tower_lat.cu (latency: one 2-board tile split
// over a cluster of 4 / 8 CTAs).  sm_100a only.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

namespace scb {

constexpr int TC_BM = 128;
constexpr int TC_BK = 64;

// ---- PTX wrappers ------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    while (!mbar_try_wait(bar, parity)) {
    }
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1,
                                            int c2, int c3)
{
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::
            "r"(dst),
        "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            dst),
        "l"(map), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
// ---- cta_group::2 (CTA pair) variants -------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster addresses carry the CTA rank in bit 24; clearing it addresses the even (leader) CTA
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;
__device__ __forceinline__ void tma2_load_4d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1,
                                             int c2, int c3)
{
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::
            "r"(dst),
        "l"(map), "r"(bar & PEER_BIT_MASK), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma2_load_2d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            dst),
        "l"(map), "r"(bar & PEER_BIT_MASK), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tc2_mma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// the same with 8-bit operands (kind::f8f6f4): K = 32 elements = 32 bytes per instruction, as kind::f16's K = 16
__device__ __forceinline__ void tc2_mma_f8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                           uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives on the barrier at the same shared-memory offset in BOTH CTAs of the pair
__device__ __forceinline__ void tc2_commit_mc(uint32_t bar)
{
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
        "h"((uint16_t)3)
        : "memory");
}
// arrive on a barrier of the leader CTA (rank 0) of the pair
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar)
{
    asm volatile(
        "{\n\t"
        ".reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, 0;\n\t"
        "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t"
        "}" ::"r"(bar)
        : "memory");
}

// true in exactly one lane of a converged warp
__device__ __forceinline__ bool elect_one()
{
    uint32_t p;
    asm volatile(
        "{\n\t"
        ".reg .pred q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, q;\n\t"
        "}"
        : "=r"(p));
    return p != 0;
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_mma_f8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major, 128-byte-swizzled shared-memory operand descriptor (sm_100 UMMA):
//   bits 0-13 start address >> 4, 16-29 leading byte offset >> 4 (unused for swizzled
//   K-major, 1), 32-45 stride byte offset >> 4 (8 rows x 128 B = 1024 B between 8-row core
//   groups), 46-47 descriptor version 1, 61-63 layout type 2 = SWIZZLE_128B.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr)
{
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// instruction descriptor: fp32 accumulate (bit 4), A/B bf16 (bits 7, 10), both K-major,
// N >> 3 at bits 17-22, M >> 4 at bits 24-28.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N)
{
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// Tensor-core operand types (fp32 accumulate): the kernels are templates on one of these, so each type is its own
// instantiation and the bf16 code is unchanged by the others.  A K chunk is one 128-byte swizzle row whatever the type
// (BK * BYTES == 128), so TMA boxes, swizzle, descriptors and shared-memory layouts are the same in bytes.
//   IDESC_AB  a_format / b_format bits of the instruction descriptor (bits 7-9 / 10-12; kind::f16: 0 = F16, 1 = BF16;
//             kind::f8f6f4: 0 = E4M3)
//   F8        the instruction kind: kind::f8f6f4 instead of kind::f16 (the format bits alone do not tell them apart)
//   TMAP      tensor-map element type
//   BYTES     bytes per element; BK = elements per K chunk
//   SCALED    the weights carry a per-output-channel power-of-two scale that the epilogue applies (acc * s + bias)
//   Park      the type the kernels keep internal values in (the SE layers' LayerNorm output, parked in shared memory)
//   pack2     two floats -> two operands, round to nearest even, first argument in the low half
//   lo, hi    the inverse: the low / high operand of a packed pair as float (exact)
//   round     a float rounded to the operand type and back: a value the kernels park in that type
//   unpack8   eight packed SE weights -> floats
__device__ __forceinline__ void bf16x8_to_float(const uint4 &u, float (&f)[8]);
struct OpBf16 {
    static constexpr uint32_t IDESC_AB = (1u << 7) | (1u << 10);
    static constexpr bool F8 = false, SCALED = false;
    static constexpr int BYTES = 2, BK = 64;
    using Park = OpBf16;
    static constexpr CUtensorMapDataType TMAP = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    __device__ __forceinline__ static uint32_t pack2(float lo, float hi)
    {
        __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
        return *reinterpret_cast<uint32_t *>(&h);
    }
    __device__ __forceinline__ static float lo(uint32_t w) { return __uint_as_float(w << 16); }
    __device__ __forceinline__ static float hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }
    __device__ __forceinline__ static float round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
    __device__ __forceinline__ static void unpack8(const uint4 &u, float (&f)[8]) { bf16x8_to_float(u, f); }
};
// fp16: 11 significant bits against bf16's 8; a value beyond +-65504 becomes +-inf, as in fp16 autocast
struct OpFp16 {
    static constexpr uint32_t IDESC_AB = 0u;
    static constexpr bool F8 = false, SCALED = false;
    static constexpr int BYTES = 2, BK = 64;
    using Park = OpFp16;
    static constexpr CUtensorMapDataType TMAP = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    __device__ __forceinline__ static uint32_t pack2(float lo, float hi)
    {
        __half2 h = __floats2half2_rn(lo, hi);
        return *reinterpret_cast<uint32_t *>(&h);
    }
    __device__ __forceinline__ static float lo(uint32_t w) { return __half2float(__ushort_as_half((unsigned short)(w & 0xffffu))); }
    __device__ __forceinline__ static float hi(uint32_t w) { return __half2float(__ushort_as_half((unsigned short)(w >> 16))); }
    __device__ __forceinline__ static float round(float x) { return __half2float(__float2half_rn(x)); }
    __device__ __forceinline__ static void unpack8(const uint4 &u, float (&f)[8])
    {
        const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const float2 p = __half22float2(*reinterpret_cast<const __half2 *>(&w[i]));
            f[2 * i] = p.x;
            f[2 * i + 1] = p.y;
        }
    }
};
// fp8 e4m3 (SC_MODE_FP8): 4 significant bits, largest finite value 448.  A K chunk is 128 channels.  The weights are
// e4m3 with a power-of-two scale per output channel (SCALED); a stored activation is e4m3 without a scale, saturated to
// +-448 (satfinite).  The SE layers' parked LayerNorm output and the SE weights stay bf16.
struct OpE4m3 {
    static constexpr uint32_t IDESC_AB = 0u;
    static constexpr bool F8 = true, SCALED = true;
    static constexpr int BYTES = 1, BK = 128;
    using Park = OpBf16;
    static constexpr CUtensorMapDataType TMAP = CU_TENSOR_MAP_DATA_TYPE_UINT8;
    // four floats -> four e4m3 (round to nearest even, satfinite), first argument in the lowest byte
    __device__ __forceinline__ static uint32_t pack4(float a, float b, float c, float d)
    {
        uint16_t lo, hi;
        asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(lo) : "f"(b), "f"(a));
        asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(hi) : "f"(d), "f"(c));
        return (uint32_t)lo | ((uint32_t)hi << 16);
    }
    // the inverse (exact: every e4m3 value is an fp16 value)
    __device__ __forceinline__ static void unpack4(uint32_t w, float (&f)[4])
    {
        uint32_t h0, h1;
        asm("cvt.rn.f16x2.e4m3x2 %0, %1;" : "=r"(h0) : "h"((uint16_t)(w & 0xffffu)));
        asm("cvt.rn.f16x2.e4m3x2 %0, %1;" : "=r"(h1) : "h"((uint16_t)(w >> 16)));
        const float2 p = __half22float2(*reinterpret_cast<const __half2 *>(&h0));
        const float2 q = __half22float2(*reinterpret_cast<const __half2 *>(&h1));
        f[0] = p.x;
        f[1] = p.y;
        f[2] = q.x;
        f[3] = q.y;
    }
    __device__ __forceinline__ static void unpack8(const uint4 &u, float (&f)[8]) { bf16x8_to_float(u, f); }
};
static_assert(OpBf16::BK * OpBf16::BYTES == 128 && OpFp16::BK * OpFp16::BYTES == 128 && OpE4m3::BK * OpE4m3::BYTES == 128,
              "a K chunk is one 128-byte swizzle row");
// one MMA of operand type OT: 4 instructions cover a 128-byte row of K for every type (K = 16 x 2 B or 32 x 1 B)
template <class OT>
__device__ __forceinline__ void tc2_mma(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate)
{
    if constexpr (OT::F8) tc2_mma_f8(tmem_d, desc_a, desc_b, idesc, accumulate);
    else tc2_mma_bf16(tmem_d, desc_a, desc_b, idesc, accumulate);
}
template <class OT>
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate)
{
    if constexpr (OT::F8) tc_mma_f8(tmem_d, desc_a, desc_b, idesc, accumulate);
    else tc_mma_bf16(tmem_d, desc_a, desc_b, idesc, accumulate);
}
// instruction descriptor of operand type OT (umma_idesc_bf16 for OpBf16)
template <class OT> __host__ __device__ constexpr uint32_t umma_idesc(int M, int N)
{
    return (1u << 4) | OT::IDESC_AB | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
static_assert(umma_idesc<OpBf16>(256, 256) == umma_idesc_bf16(256, 256), "bf16 instruction descriptor");

__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void bf16x8_to_float(const uint4 &u, float (&f)[8])
{
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; i++) {
        f[2 * i] = __uint_as_float(w[i] << 16);
        f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
}

// Column sums over the 16 lanes of each board for rows ordered (rank, board, file): lane bit 3 is the board, so
// the recursive halving skips that bit.  Lane l ends with the sums of its board for indices i0, i0 + 1,
// i0 = 16 b16 + 8 b4 + 4 b2 + 2 b1 (30 shuffles).
__device__ __forceinline__ float2 warp_transpose_reduce_2boards(float (&v)[32], int lane, int &i0)
{
    const bool b16 = lane & 16, b4 = lane & 4, b2 = lane & 2, b1 = lane & 1;
    float w16[16], w8[8], w4[4], w2[2];
#pragma unroll
    for (int i = 0; i < 16; i++) {
        float send = b16 ? v[i] : v[i + 16];
        float keep = b16 ? v[i + 16] : v[i];
        w16[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
#pragma unroll
    for (int i = 0; i < 8; i++) {
        float send = b4 ? w16[i] : w16[i + 8];
        float keep = b4 ? w16[i + 8] : w16[i];
        w8[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        float send = b2 ? w8[i] : w8[i + 4];
        float keep = b2 ? w8[i + 4] : w8[i];
        w4[i] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
#pragma unroll
    for (int i = 0; i < 2; i++) {
        float send = b1 ? w4[i] : w4[i + 2];
        float keep = b1 ? w4[i + 2] : w4[i];
        w2[i] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
    }
    i0 = (b16 ? 16 : 0) + (b4 ? 8 : 0) + (b2 ? 4 : 0) + (b1 ? 2 : 0);
    return make_float2(w2[0], w2[1]);
}


// ---- LayerNorm arithmetic shared by both kernels -------------------------------------------------------------
// Written with explicit round-to-nearest intrinsics so that the compiler cannot contract / reassociate it
// differently in different kernels: the latency kernel must produce the bits of the throughput kernel.
// Statistics: per group of channels the pair (s, M2) = (sum of a = acc + bias, sum of squares of a about the group's own
// mean).  A 32-channel chunk computes both from its registers (ln_chunk_stats); chunks are merged with the pairwise
// formula of ln_combine, in a fixed tree:
//   half0 = (p0 + p1) + (p2 + p3), half1 = (p4 + p5) + (p6 + p7), total = half0 + half1
// so the chunks may be computed by different threads / CTAs.  The variance is M2 / 256: unlike the one-pass
// E[a^2] - mean^2 it does not cancel when the channel mean of a square is large next to its spread (a checkpoint whose
// conv biases share a common offset), because no sum of squares is taken about a point far from the values.
// A chunk: the deviations d = a - a[0] from its first channel as eight interleaved sequential chains (j mod 8) of sums
// and of squares and a fixed tree, then s = sum d + 32 a[0] and M2 = sum d^2 - (sum d)^2 / 32.  a[0] lies within
// sqrt(31) standard deviations of the chunk's mean, so that subtraction loses at most five bits; shifting by a[0]
// rather than by the chunk's mean keeps the two chains independent (one pass, as short as unshifted sums).
__device__ __forceinline__ void ln_chunk_stats(const float (&a)[32], float &s, float &m2)
{
    float s8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, q8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const float k = a[0];
#pragma unroll
    for (int j = 1; j < 32; j++) {
        const float d = __fsub_rn(a[j], k);
        s8[j & 7] = __fadd_rn(s8[j & 7], d);
        q8[j & 7] = __fmaf_rn(d, d, q8[j & 7]);
    }
    const float sd = __fadd_rn(__fadd_rn(__fadd_rn(s8[0], s8[1]), __fadd_rn(s8[2], s8[3])),
                               __fadd_rn(__fadd_rn(s8[4], s8[5]), __fadd_rn(s8[6], s8[7])));
    const float qd = __fadd_rn(__fadd_rn(__fadd_rn(q8[0], q8[1]), __fadd_rn(q8[2], q8[3])),
                               __fadd_rn(__fadd_rn(q8[4], q8[5]), __fadd_rn(q8[6], q8[7])));
    s = __fmaf_rn(32.f, k, sd);
    m2 = fmaxf(__fmaf_rn(__fmul_rn(sd, -1.f / 32.f), sd, qd), 0.f);
}
// (s, M2) of two groups of n channels each -> the union: M2 = M2a + M2b + (sa - sb)^2 / (2n), inv_2n = 1 / (2n)
__device__ __forceinline__ float2 ln_combine(const float2 p, const float2 q, float inv_2n)
{
    const float d = __fsub_rn(p.x, q.x);
    return make_float2(__fadd_rn(p.x, q.x), __fmaf_rn(__fmul_rn(d, d), inv_2n, __fadd_rn(p.y, q.y)));
}
// four 32-channel chunks -> 128 channels
__device__ __forceinline__ float2 ln_half(const float2 p0, const float2 p1, const float2 p2, const float2 p3)
{
    return ln_combine(ln_combine(p0, p1, 1.f / 64.f), ln_combine(p2, p3, 1.f / 64.f), 1.f / 128.f);
}
// two 128-channel halves -> mean and 1 / sqrt(var + eps) of all 256
__device__ __forceinline__ void ln_finish(const float2 h0, const float2 h1, float eps, float &mean, float &rstd)
{
    const float2 t = ln_combine(h0, h1, 1.f / 256.f);
    mean = __fmul_rn(t.x, 1.f / 256.f);
    rstd = rsqrtf(__fadd_rn(__fmul_rn(t.y, 1.f / 256.f), eps));
}
// (a - mean) * rstd * gamma + beta with a = acc + bias already formed
__device__ __forceinline__ float ln_apply(float a, float mean, float rstd, float gamma, float beta)
{
    return __fmaf_rn(__fmul_rn(__fsub_rn(a, mean), rstd), gamma, beta);
}

// squeeze-excitation scalar pieces, shared for the same reason
__device__ __forceinline__ float se_hidden(float b1, float half0, float half1)
{
    return fmaxf(__fadd_rn(__fadd_rn(b1, half0), half1), 0.f);
}
// Both SE matrix-vector products are defined chunk-wise so that the chunks can be computed by different threads / CTAs:
// per 32-input chunk one sequential fma chain from 0 (se_chain8 = 8 inputs of it), the chunk sums combined in fixed trees.
__device__ __forceinline__ float se_chain8(const float (&w)[8], const float4 a, const float4 b, float acc)
{
    acc = fmaf(w[0], a.x, acc); acc = fmaf(w[1], a.y, acc); acc = fmaf(w[2], a.z, acc); acc = fmaf(w[3], a.w, acc);
    acc = fmaf(w[4], b.x, acc); acc = fmaf(w[5], b.y, acc); acc = fmaf(w[6], b.z, acc); acc = fmaf(w[7], b.w, acc);
    return acc;
}
__device__ __forceinline__ float se_tree4(float p0, float p1, float p2, float p3)
{
    return __fadd_rn(__fadd_rn(p0, p1), __fadd_rn(p2, p3));
}
// FC2 pre-activation: bias + the four 32-hidden-unit chunk sums
__device__ __forceinline__ float se_fc2_sum(float b2, float c0, float c1, float c2, float c3)
{
    return __fadd_rn(b2, se_tree4(c0, c1, c2, c3));
}
__device__ __forceinline__ float se_sigmoid(float g) { return __fdiv_rn(1.f, __fadd_rn(1.f, __expf(-g))); }

}  // namespace scb
