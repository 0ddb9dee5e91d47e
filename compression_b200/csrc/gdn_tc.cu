// GDN / IGDN forward and backward on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//
//   n[pix, i] = sum_j p[pix, j] * gamma[j, i]      p = |x|, x^2 or relu(x) variants (py/layers/gdn.py:377-398)
//
// is a [n_pix x C] x [C x C] GEMM with 2*C^2 FLOP per 8*C bytes of HBM traffic: on fp32 CUDA cores it is
// compute bound at ~1/3 of the HBM roofline.  Here the contraction runs as  tcgen05.mma kind::f16  on an
// error-compensated bf16 split (3 products: hi*hi + lo*hi + hi*lo, fp32 accumulation in TMEM), which keeps the
// result within ~4e-6 of fp32 (SURVEY.md App. D; the contract is 1e-5) at bf16 tensor throughput.
// Every kernel is persistent (one CTA per SM, 128-pixel tiles) and specialised at compile time for FAST, the default
// GDN / IGDN (alpha = 1, epsilon = 1, no rectification); the other instantiation honours TcFlags at run time.  IO is
// the element type of the activations x, dy, y, dx in memory (0 float32, 1 float16, 2 bfloat16; see IoBytes): 16-bit
// elements are widened exactly on load and rounded once at the store, everything else is the same for every IO.
//
//   gdn_tc_fwd2_kernel<FAST, IO>         forward, C = 128: the x tile resident in shared memory (bulk async
//                                        copies), y written over it in place
//   gdn_tc_fwd4_kernel<C, FAST, IO>      forward, C = 192: x in 2-D TMA boxes, gamma's lo plane streamed
//   gdn_tc_bwd3_kernel<FAST, IO>         backward, C = 128: dx and the per-CTA dgamma / dbeta partials in one kernel
//   gdn_tc_bwd_dx2_kernel<FAST, IO>      backward, C = 192: dx and q = dL/dn (handed over as bf16 operand planes)
//   gdn_tc_bwd_dgamma2_kernel<FAST, IO>  backward, C = 192: dgamma / dbeta partials from x and q
//   gdn_tc_prep_kernel, gdn_tc_prep2_kernel   gamma -> bf16 hi / lo operand planes
//
// tc_rule (at the end of the file) decides which calls these kernels take, for both directions and every IO;
// gdn_tc_forward / gdn_tc_backward apply it for gdn.cu, and tfcb_gdn_native_16bit answers it for the caller of the
// 16-bit entries.  gdn.cu runs the fp32 kernels for a float32 call the rule refuses.
#include <cuda.h>  // CUtensorMap (types only; cuTensorMapEncodeTiled is fetched through the runtime)
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <type_traits>

#include "common.cuh"

namespace tfcb {
namespace {

constexpr int kTileM = 128;    // pixels per tile (UMMA M)

struct TcFlags {
  int inverse, rectify, alpha_mode, eps_mode;  // alpha_mode: 1 |u|, 2 u^2; eps_mode: 1 identity, 2 sqrt
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// UMMA shared-memory descriptor, K-major, SWIZZLE_NONE (cute/arch/mma_sm100_desc.hpp SmemDescriptor):
// bits [0,14) start >> 4, [16,30) leading byte offset >> 4 (between the two 8-element K chunks of one MMA),
// [32,46) stride byte offset >> 4 (between 8-row groups), [46,48) version = 1, [61,64) layout = 0.
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) | (1ull << 46);
}

// Instruction descriptor for kind::f16: D = f32 (bits [4,6) = 1), A = B = bf16 ([7,10) = [10,13) = 1), both
// K-major ([15], [16] = 0), N >> 3 at [17,23), M >> 4 at [24,29).
__host__ __device__ constexpr uint32_t umma_idesc(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

__device__ __forceinline__ void umma_commit(uint32_t mbar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mbar) : "memory");
}

__device__ __forceinline__ bool mbar_wait(uint32_t mbar, uint32_t parity) {
  for (int spin = 0; spin < (1 << 24); ++spin) {
    uint32_t done;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(done)
        : "r"(mbar), "r"(parity)
        : "memory");
    if (done) return true;
  }
  return false;  // never spin forever on a bad descriptor: the host reports an error instead of hanging
}

// FAST = the default GDN / IGDN of bls2017 / bmshj2018 (alpha = 1, epsilon = 1, no rectification): no
// per-element branches.  Otherwise the runtime flags are honoured.
template <bool FAST>
__device__ __forceinline__ float tc_pool(float x, const TcFlags& f) {
  if (FAST) return fabsf(x);
  const float u = f.rectify ? fmaxf(x, 0.f) : x;
  if (f.alpha_mode == 2) return u * u;
  return f.rectify ? u : fabsf(u);
}

// y = u / m (GDN) or u * m (IGDN).  The quotient uses the hardware reciprocal (MUFU.RCP, <= 2 ulp): an IEEE
// divide costs ~20 instructions per element, which made the whole kernel ALU bound (ncu, profiles/), and
// 2.4e-7 is far inside the 1e-5 contract.
__device__ __forceinline__ float rcp_approx(float v) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));  // MUFU.RCP, <= 1 ulp; n = beta + pool is a normal, moderate number
  return r;
}

template <bool FAST>
__device__ __forceinline__ float tc_out(float x, float n, const TcFlags& f) {
  if (FAST) return f.inverse ? x * n : x * rcp_approx(n);
  const float u = f.rectify ? fmaxf(x, 0.f) : x;
  const float m = (f.eps_mode == 2) ? sqrtf(n) : n;
  return f.inverse ? u * m : u * rcp_approx(m);
}

// bf16 split of 8 consecutive values -> two 16-byte rows of the hi / lo operand planes.
// Packed conversions (cvt.rn.bf16x2.f32) and integer re-expansion of the hi part keep this at ~3
// instructions per element.
__device__ __forceinline__ uint32_t pack_bf16x2(float lo_elem, float hi_elem) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi_elem), "f"(lo_elem));
  return r;
}

__device__ __forceinline__ void split8(const float (&v)[8], uint4* hi, uint4* lo) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    h[i] = pack_bf16x2(v[2 * i], v[2 * i + 1]);
    const float h0 = __uint_as_float(h[i] << 16), h1 = __uint_as_float(h[i] & 0xFFFF0000u);
    l[i] = pack_bf16x2(v[2 * i] - h0, v[2 * i + 1] - h1);
  }
  *hi = make_uint4(h[0], h[1], h[2], h[3]);
  *lo = make_uint4(l[0], l[1], l[2], l[3]);
}

// gamma [C, C] fp32 (gamma[j, i]) -> hi / lo bf16 planes in the B-operand layout [j / 8][i][j % 8].
__global__ void gdn_tc_prep_kernel(const float* __restrict__ gamma, int C, __nv_bfloat16* __restrict__ planes) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;  // over (j / 8, i)
  if (idx >= (C / 8) * C) return;
  const int jc = idx / C, i = idx % C;
  float v[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) v[e] = gamma[(jc * 8 + e) * C + i];
  uint4 hi, lo;
  split8(v, &hi, &lo);
  reinterpret_cast<uint4*>(planes)[idx] = hi;
  reinterpret_cast<uint4*>(planes + (size_t)C * C)[idx] = lo;
}

template <int N>
__device__ __forceinline__ void tmem_load(uint32_t taddr, uint32_t (&r)[N]);

template <>
__device__ __forceinline__ void tmem_load<32>(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}

template <>
__device__ __forceinline__ void tmem_load<8>(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}

template <>
__device__ __forceinline__ void tmem_load<16>(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}

// =============================================================================================
// Forward, second generation (C = 128): the whole x tile lives in shared memory.
//
//   bulk async copies (cp.async.bulk, one 512-byte pixel row each, completion on an mbarrier) bring tile t+1
//   into a padded [128][132] fp32 buffer while tile t is processed; the same buffer is the epilogue's x source
//   and, rewritten in place with y, the source of the bulk stores.  Nothing is re-read from L2, no thread ever
//   waits on a global load, and the 528-byte row stride makes the thread-per-pixel-row accesses (the mapping
//   tcgen05.ld imposes) bank-conflict free, so no staging transposes and no barriers inside the epilogue.
//   K is consumed in chunks of 16 channels through two small operand-plane buffers.
// =============================================================================================
constexpr int kF2Threads = 320;   // 8 compute warps + 1 copy warp + 1 MMA-issue warp
constexpr int kF2Compute = 256;
constexpr int kF2XBuf = kTileM * 128 * 4;          // one x / y tile, dense [128][128] fp32 (one bulk copy)
constexpr int kF2Kg = kTileM * 16 + 160;           // plane group stride: padding = 2 (mod 8) 16-byte units -> conflict-free
                                                   // stores; sized so that the epilogue's [128][68] staging fits in the planes
constexpr int kF2StLd = 68;                        // floats per staging row (64 + 4)
constexpr int kF2Plane = 4 * kF2Kg;                // one hi or lo plane of a 32-channel chunk

struct Fwd2Smem {
  static constexpr int C = 128;
  static constexpr int kOffBh = 0;
  static constexpr int kOffBl = kOffBh + C * C * 2;
  static constexpr int kOffX = kOffBl + C * C * 2;            // [2] x / y tiles
  static constexpr int kOffP = kOffX + 2 * kF2XBuf;           // [2 buffers][hi, lo]; the epilogue's staging aliases it
  static constexpr int kOffBar = kOffP + 4 * kF2Plane;        // full[2], plane[2], y ready[2], TMEM slot
  static constexpr int kBytes = kOffBar + 64;
  static_assert(4 * kF2Plane >= kTileM * kF2StLd * 4, "staging must fit in the operand-plane area");
  static_assert(kBytes <= 232448, "shared memory budget");
};

// Element type of x / y in memory: 0 float32, 1 float16, 2 bfloat16 (the reference's mixed-precision policy keeps the
// variables in float32 and the activations in 16 bits, gdn_test.py:200-210; arithmetic is float32 here either way).
template <int IO>
struct IoBytes { static constexpr int value = IO == 0 ? 4 : 2; };

template <int IO>
__device__ __forceinline__ void io_widen8(const uint4 raw, float (&v)[8]) {  // 8 consecutive 16-bit elements, exactly
  const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (IO == 2) {
      v[2 * i] = __uint_as_float(w[i] << 16);
      v[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
    } else {
      const __half2 hh = *reinterpret_cast<const __half2*>(&w[i]);
      const float2 ff = __half22float2(hh);
      v[2 * i] = ff.x;
      v[2 * i + 1] = ff.y;
    }
  }
}

template <int IO>
__device__ __forceinline__ void io_load8(const uint8_t* src, float (&v)[8]) {
  io_widen8<IO>(*reinterpret_cast<const uint4*>(src), v);
}

template <int IO>
__device__ __forceinline__ void io_store8(uint8_t* dst, const float (&v)[8]) {
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (IO == 2) {
      w[i] = pack_bf16x2(v[2 * i], v[2 * i + 1]);
    } else {
      const __half2 hh = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<const uint32_t*>(&hh);
    }
  }
  *reinterpret_cast<uint4*>(dst) = make_uint4(w[0], w[1], w[2], w[3]);
}

// One [128 rows x 32 channels] TMA box of x / dy / dx in shared memory (the C = 192 forward and every backward kernel):
//   float32: 128-byte rows, 128-byte swizzle: 16-byte chunk j (4 channels) of row r sits at chunk j ^ (r & 7);
//   16-bit:   64-byte rows,  64-byte swizzle: 16-byte chunk j (8 channels) of row r sits at chunk j ^ ((r >> 1) & 3).
// The thread that owns row r and channel octet `oct` of a box moves its 8 values with two 16-byte accesses (float32)
// or one (16-bit).  Both are conflict free: the 8 lanes of each 16-byte access phase are 8 consecutive rows, which
// land on 8 different 16-byte bank groups.  A ring slot keeps the float32 size (kF4Box below); a 16-bit box fills half.
template <int IO>
struct Box {
  static constexpr int kRowB = 32 * IoBytes<IO>::value;  // bytes per box row
  static constexpr int kBytes = kTileM * kRowB;          // bytes per box: the expect_tx count of one copy
};

template <int IO>
__device__ __forceinline__ uint8_t* box_chunk(uint8_t* box, int row, int j) {  // 16-byte chunk j of box row `row`
  if constexpr (IO == 0) return box + row * 128 + ((j ^ (row & 7)) << 4);
  else return box + row * 64 + ((j ^ ((row >> 1) & 3)) << 4);
}

template <int IO>
__device__ __forceinline__ void box_load8(uint8_t* box, int row, int oct, float (&v)[8]) {
  if constexpr (IO == 0) {
    const float4 a = *reinterpret_cast<const float4*>(box_chunk<0>(box, row, 2 * oct));
    const float4 b = *reinterpret_cast<const float4*>(box_chunk<0>(box, row, 2 * oct + 1));
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
    v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  } else {
    io_load8<IO>(box_chunk<IO>(box, row, oct), v);  // widened exactly
  }
}

template <int IO>
__device__ __forceinline__ void box_store8(uint8_t* box, int row, int oct, const float (&v)[8]) {
  if constexpr (IO == 0) {
    *reinterpret_cast<float4*>(box_chunk<0>(box, row, 2 * oct)) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(box_chunk<0>(box, row, 2 * oct + 1)) = make_float4(v[4], v[5], v[6], v[7]);
  } else {
    io_store8<IO>(box_chunk<IO>(box, row, oct), v);  // rounded once, to nearest even
  }
}

template <bool FAST, int IO>
__global__ void __launch_bounds__(kF2Threads, 1)
gdn_tc_fwd2_kernel(const void* __restrict__ x_, const float* __restrict__ gamma,
                   const float* __restrict__ beta, void* __restrict__ y_, long long n_pix, TcFlags f) {
  using L = Fwd2Smem;
  constexpr int C = 128;
  constexpr int EB = IoBytes<IO>::value, kRowB = C * EB;  // bytes per element / per pixel row
  const uint8_t* x = static_cast<const uint8_t*>(x_);
  uint8_t* y = static_cast<uint8_t*>(y_);
  extern __shared__ __align__(1024) uint8_t smem[];
  float* stage = reinterpret_cast<float*>(smem + L::kOffP);          // [128][68] fp32, only during the epilogue
  uint64_t* mbars = reinterpret_cast<uint64_t*>(smem + L::kOffBar);  // [0,1] full, [2,3] plane, [4,5] y tile ready
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + L::kOffBar + 56);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int r = tid & 127, h = tid >> 7, gwarp = warp & 3;
  constexpr uint32_t kIdesc = umma_idesc(kTileM, C);

  // gamma [C, C] fp32 (64 KB, L2 resident) -> hi / lo bf16 planes [j / 8][i][j % 8], converted by every CTA in its
  // prologue: no per-call allocation and no separate preparation launch (they cost the small shapes 10 %)
  for (int idx = tid; idx < (C / 8) * C; idx += kF2Threads) {
    const int jc = idx / C, i = idx % C;
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = __ldg(gamma + (jc * 8 + e) * C + i);
    uint4 hi, lo;
    split8(v, &hi, &lo);
    reinterpret_cast<uint4*>(smem + L::kOffBh)[idx] = hi;
    reinterpret_cast<uint4*>(smem + L::kOffBl)[idx] = lo;
  }
  if (tid == 0) {
    for (int i = 0; i < 6; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(mbars + i)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(128));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_n = *tmem_slot;
  const uint32_t lane_sel = (uint32_t)(gwarp * 32) << 16;
  const uint32_t b_hi = smem_u32(smem + L::kOffBh), b_lo = smem_u32(smem + L::kOffBl);
  const uint32_t xs = smem_u32(smem + L::kOffX);
  uint32_t par_full[2] = {0u, 0u}, par_plane[2] = {0u, 0u};

  const long long n_tiles = (n_pix + kTileM - 1) / kTileM;
  // thread 0 moves the tiles: a tile is one contiguous block of rows * 512 bytes
  auto issue_load = [&](long long tile, int b) {
    const long long p0 = tile * kTileM;
    const uint32_t bytes = (uint32_t)min((long long)kTileM, n_pix - p0) * (uint32_t)kRowB;
    const uint32_t mbar = smem_u32(mbars + b);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     xs + b * kF2XBuf),
                 "l"(x + p0 * kRowB), "r"(bytes), "r"(mbar)
                 : "memory");
  };
  if (warp == kF2Compute / 32) {
    // ------------------------------ copy warp ------------------------------
    // Both buffers are filled up front; afterwards, per tile: wait until the compute warps have rewritten the
    // buffer with y, store it, and as soon as the store has read the buffer refill it with the tile after next.
    if (lane == 0) {
      uint32_t par_y[2] = {0u, 0u};
      if (blockIdx.x < n_tiles) issue_load(blockIdx.x, 0);
      if (blockIdx.x + (long long)gridDim.x < n_tiles) issue_load(blockIdx.x + gridDim.x, 1);
      int it = 0;
      for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const int b = it & 1;
        const long long p0 = tile * kTileM;
        const uint32_t bytes = (uint32_t)min((long long)kTileM, n_pix - p0) * (uint32_t)kRowB;
        if (!mbar_wait(smem_u32(mbars + 4 + b), par_y[b])) __trap();
        par_y[b] ^= 1u;
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(y + p0 * kRowB),
                     "r"(xs + b * kF2XBuf), "r"(bytes)
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        const long long nxt = tile + 2ll * gridDim.x;
        if (nxt < n_tiles) {
          asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          issue_load(nxt, b);
        }
      }
      asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
    __syncwarp();
  } else if (warp == kF2Compute / 32 + 1) {
    // ---------------------------- MMA-issue warp ----------------------------
    // The compute warps only ARRIVE on the chunk's named barrier once their operand planes are written and
    // fenced; this warp waits on it, issues the chunk's MMAs and commits to the plane mbarrier.  (Barrier ids
    // alternate with the plane buffer: a buffer is rewritten only after its commit has been waited for.)
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
#pragma unroll
      for (int c = 0; c < C / 32; ++c) {
        const int pb = c & 1;
        asm volatile("bar.sync %0, %1;" ::"r"(2 + pb), "n"(kF2Compute + 32) : "memory");
        if (lane == 0) {
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t ph = smem_u32(smem + L::kOffP + pb * 2 * kF2Plane), pl = ph + kF2Plane;
#pragma unroll
          for (int s2 = 0; s2 < 2; ++s2) {
            const uint64_t dah = umma_desc(ph + (uint32_t)(2 * s2) * kF2Kg, kF2Kg, 128);
            const uint64_t dal = umma_desc(pl + (uint32_t)(2 * s2) * kF2Kg, kF2Kg, 128);
            const uint32_t b_off = (uint32_t)(c * 4 + 2 * s2) * (C * 16);
            const uint64_t dbh = umma_desc(b_hi + b_off, C * 16, 128);
            const uint64_t dbl = umma_desc(b_lo + b_off, C * 16, 128);
            umma_bf16(tmem_n, dah, dbh, kIdesc, (c | s2) ? 1u : 0u);
            umma_bf16(tmem_n, dal, dbh, kIdesc, 1u);
            umma_bf16(tmem_n, dah, dbl, kIdesc, 1u);
          }
          umma_commit(smem_u32(mbars + 2 + pb));
        }
        __syncwarp();
      }
    }
  } else {
  // ----------------------------- compute warps -----------------------------

  // memory-side items of a 32-channel chunk: (row, kg) = 8 channels of one pixel, two per thread.  Odd rows touch
  // the two 16-byte halves of their 32 bytes in the opposite order: with the dense 512-byte row stride two
  // neighbouring rows would otherwise hit the same banks.
  const int ckg = tid & 3, crow = tid >> 2;
  const int swap = crow & 1;

  auto compute_sync = [] { asm volatile("bar.sync 1, %0;" ::"n"(kF2Compute) : "memory"); };
  int it = 0;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
    const int b = it & 1;
    // (b) this tile has landed
    if (!mbar_wait(smem_u32(mbars + b), par_full[b])) __trap();
    par_full[b] ^= 1u;
    uint8_t* xt = smem + L::kOffX + b * kF2XBuf;
    // (c) pool + bf16 split, 32 channels at a time
#pragma unroll
    for (int c = 0; c < C / 32; ++c) {
      const int pb = c & 1;
      if (c >= 2) {
        if (!mbar_wait(smem_u32(mbars + 2 + pb), par_plane[pb])) __trap();
        par_plane[pb] ^= 1u;
      }
      uint8_t* ph = smem + L::kOffP + pb * 2 * kF2Plane;
      uint8_t* pl = ph + kF2Plane;
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int row = crow + 64 * i;
        const uint8_t* src = xt + row * kRowB + (c * 32 + ckg * 8) * EB;
        float v[8];
        if (IO == 0) {
          const float4 va = *reinterpret_cast<const float4*>(src + (swap ? 16 : 0));
          const float4 vb = *reinterpret_cast<const float4*>(src + (swap ? 0 : 16));
          const float4 v0 = swap ? vb : va, v1 = swap ? va : vb;
          v[0] = v0.x; v[1] = v0.y; v[2] = v0.z; v[3] = v0.w;
          v[4] = v1.x; v[5] = v1.y; v[6] = v1.z; v[7] = v1.w;
        } else {
          io_load8<IO>(src, v);
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = tc_pool<FAST>(v[e], f);
        uint4 hi, lo;
        split8(v, &hi, &lo);
        *reinterpret_cast<uint4*>(ph + ckg * kF2Kg + row * 16) = hi;
        *reinterpret_cast<uint4*>(pl + ckg * kF2Kg + row * 16) = lo;
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      asm volatile("bar.arrive %0, %1;" ::"r"(2 + pb), "n"(kF2Compute + 32) : "memory");
    }
    // (d) epilogue in place: y = x / (beta + n).  The last two commits cover every MMA of the tile, after which
    // the operand planes are dead and their memory is the staging buffer for the TMEM -> row-major transpose.
#pragma unroll
    for (int pb = 0; pb < 2; ++pb) {
      if (!mbar_wait(smem_u32(mbars + 2 + pb), par_plane[pb])) __trap();
      par_plane[pb] ^= 1u;
    }
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    // 64 output channels at a time: thread (r, h) moves 32 accumulator columns of its row to the staging buffer,
    // then every thread finishes four (row, 8-channel) items; lanes 4..7 of each 8-lane group touch the two
    // 16-byte halves in the opposite order (a row's eight items span 256 B = two passes over the banks).
    const int ekg = tid & 7, erow = tid >> 3, eswap = (ekg >> 2) & 1;
#pragma unroll
    for (int cc = 0; cc < C / 64; ++cc) {
      {
        uint32_t acc[32];
        tmem_load<32>(tmem_n + lane_sel + (uint32_t)(cc * 64 + h * 32), acc);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        float* dst = stage + r * kF2StLd + h * 32;
#pragma unroll
        for (int i = 0; i < 8; ++i)
          *reinterpret_cast<float4*>(dst + 4 * i) = make_float4(__uint_as_float(acc[4 * i]), __uint_as_float(acc[4 * i + 1]),
                                                                 __uint_as_float(acc[4 * i + 2]), __uint_as_float(acc[4 * i + 3]));
      }
      compute_sync();
      const float4 bv0 = __ldg(reinterpret_cast<const float4*>(beta + cc * 64 + ekg * 8));
      const float4 bv1 = __ldg(reinterpret_cast<const float4*>(beta + cc * 64 + ekg * 8) + 1);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int row = erow + 32 * i;
        uint8_t* src = xt + row * kRowB + (cc * 64 + ekg * 8) * EB;
        const uint8_t* nsrc = reinterpret_cast<const uint8_t*>(stage + row * kF2StLd + ekg * 8);
        if (IO != 0) {  // 16-bit elements: one 16-byte load and store per item
          float xv[8], o[8];
          io_load8<IO>(src, xv);
          const float4 na = *reinterpret_cast<const float4*>(nsrc), nb = *reinterpret_cast<const float4*>(nsrc + 16);
          const float nn[8] = {bv0.x + na.x, bv0.y + na.y, bv0.z + na.z, bv0.w + na.w,
                               bv1.x + nb.x, bv1.y + nb.y, bv1.z + nb.z, bv1.w + nb.w};
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] = tc_out<FAST>(xv[e], nn[e], f);
          io_store8<IO>(src, o);
          continue;
        }
        float4* pa = reinterpret_cast<float4*>(src + (eswap ? 16 : 0));
        float4* pb2 = reinterpret_cast<float4*>(src + (eswap ? 0 : 16));
        const float4 va = *pa, vb = *pb2;
        const float4 na = *reinterpret_cast<const float4*>(nsrc + (eswap ? 16 : 0));
        const float4 nb = *reinterpret_cast<const float4*>(nsrc + (eswap ? 0 : 16));
        const float4 ba = eswap ? bv1 : bv0, bb = eswap ? bv0 : bv1;
        float4 oa, ob;
        oa.x = tc_out<FAST>(va.x, ba.x + na.x, f);
        oa.y = tc_out<FAST>(va.y, ba.y + na.y, f);
        oa.z = tc_out<FAST>(va.z, ba.z + na.z, f);
        oa.w = tc_out<FAST>(va.w, ba.w + na.w, f);
        ob.x = tc_out<FAST>(vb.x, bb.x + nb.x, f);
        ob.y = tc_out<FAST>(vb.y, bb.y + nb.y, f);
        ob.z = tc_out<FAST>(vb.z, bb.z + nb.z, f);
        ob.w = tc_out<FAST>(vb.w, bb.w + nb.w, f);
        *pa = oa;
        *pb2 = ob;
      }
      if (cc == C / 64 - 1) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // y tile -> bulk store
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      compute_sync();  // staging free again (and, after the last chunk, for the next tile's operand planes)
    }
    // (e) hand the y tile to the copy warp
    if (tid == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(mbars + 4 + b)) : "memory");
  }
  }  // compute warps
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (tid < 32) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(*tmem_slot), "n"(128));
  }
}

template <bool FAST, int IO>
int launch_tc_fwd2(const void* x, const float* gamma, const float* beta, void* y, long long n_pix, TcFlags f,
                   cudaStream_t s) {
  constexpr int C = 128;
  using L = Fwd2Smem;
  {  // the attribute is per device: set it on every launch (microseconds)
    cudaError_t e = cudaFuncSetAttribute(gdn_tc_fwd2_kernel<FAST, IO>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kBytes);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      return fail(TFCB_CUDA_ERROR, "cannot reserve %d bytes of shared memory: %s", L::kBytes, cudaGetErrorString(e));
    }
  }
  const long long n_tiles = (n_pix + kTileM - 1) / kTileM;
  const int grid = (int)std::min<long long>(n_tiles, device_sm_count());
  gdn_tc_fwd2_kernel<FAST, IO><<<grid, kF2Threads, L::kBytes, s>>>(x, gamma, beta, y, n_pix, f);
  TFCB_LAUNCHED();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(TFCB_CUDA_ERROR, "GDN tensor-core kernel launch failed: %s", cudaGetErrorString(e));
  return TFCB_OK;
}


// =============================================================================================
// Forward, C = 192, fourth kernel shape: everything that touches HBM is asynchronous, and the epilogue of one
// tile runs between the conversion chunks of the next.
//
// gamma's hi + lo planes (144 KB) leave no room for x, and feeding the conversion and the epilogue from registers
// (the round-1 kernel, 52 % of the HBM roofline) leaves every compute thread waiting on its own loads and stores
// (clock64 trace of a ring-fed variant with register stores: 5.2 k of 15.9 k cycles per tile in the epilogue's store
// back-pressure, 3 k waiting for boxes of a three-slot ring, 1.7 k waiting for the tensor pipe).  So:
//   * only gamma's HI plane is resident (72 KB); the LO plane is needed by one of the three products only and is
//     streamed from L2 per 32-channel K chunk (12 KB bulk copies, double buffered) by a "gamma" warp;
//   * x arrives as [128 rows x 32 channels] 2-D TMA boxes (Box<IO>) in two three-slot rings, twice per
//     tile: boxes C0..C5 feed the pool + bf16 split, boxes E0..E5 (L2 hits) feed the epilogue; the whole next tile is
//     prefetched into L2 with one bulk prefetch;
//   * the epilogue needs no transpose: thread (r, h) takes 16 accumulator columns of ITS pixel row from TMEM,
//     reads the same 64 bytes of x from its row of the E box (the swizzle makes the row-per-lane access conflict
//     free), overwrites them with y = x / (beta + n), and a "store" warp sends the box out with a 2-D TMA store;
//   * two accumulators in TMEM: while the tensor pipe works on tile t + 1 (it is the slower side of the conversion
//     phase), the compute warps finish box c - 1 of tile t after converting chunk c of tile t + 1.
// No compute thread ever waits on a global load or store, and there is no CTA-wide barrier in the steady state.
// Rows past n_pix: zero-filled on load, clipped on store.
// =============================================================================================
// L2 eviction-priority descriptors for bulk / tensor copies (the values createpolicy.fractional.L2::evict_* produces
// for fraction 1.0; same constants as CUTLASS's TMA::CacheHintSm90)
constexpr unsigned long long kEvictFirst = 0x12F0000000000000ull, kEvictLast = 0x14F0000000000000ull;

constexpr int kF4Compute = 512;                  // 16 compute warps: four per scheduler, the work is latency bound
constexpr int kF4Threads = kF4Compute + 160;     // + MMA-issue, C-copy, E-copy, gamma and store warps
constexpr int kF4Sync = kF4Compute + 32;         // compute + issue warps (the named barriers of the plane hand-off)
constexpr int kF4Box = kTileM * 32 * 4;          // one ring slot: a [128][32] fp32 box (a 16-bit box fills half, Box<IO>)
constexpr int kF4Kg = kTileM * 16 + 32;          // plane group stride: padding = 2 (mod 8) 16-byte units (see kF2Kg)
constexpr int kF4Plane = 4 * kF4Kg;              // hi or lo plane of a 32-channel chunk

template <int C>
struct Fwd4Smem {
  static constexpr int kPlaneB = C * C * 2;                 // gamma hi (resident)
  static constexpr int kGlo = 4 * C * 16;                   // one 32-channel K chunk of gamma lo
  static constexpr int kOffBh = 0;
  static constexpr int kOffRing = kOffBh + kPlaneB;         // [3] C boxes, [3] E boxes (1024-byte aligned: swizzle atom)
  static constexpr int kOffGlo = kOffRing + 6 * kF4Box;     // [2] gamma lo chunks
  static constexpr int kOffP = kOffGlo + 2 * kGlo;          // [2 buffers][hi, lo] operand planes
  static constexpr int kOffBeta = kOffP + 4 * kF4Plane;
  static constexpr int kOffBar = kOffBeta + C * 4;
  // mbarriers: plane[2], gfull[2], cfull[3], cempty[3], efull[3], eempty[3], yready[3]; then the TMEM slot
  static constexpr int kBarPlane = 0, kBarGfull = 2, kBarCfull = 4, kBarCempty = 7, kBarEfull = 10, kBarEempty = 13,
                       kBarY = 16, kNumBars = 19;
  static constexpr int kBytes = kOffBar + kNumBars * 8 + 16;
  static_assert(kOffRing % 1024 == 0 && kOffGlo % 128 == 0 && kOffP % 128 == 0, "alignment");
  static_assert(kBytes <= 232448, "shared memory budget");
};

template <int C, bool FAST, int IO>
__global__ void __launch_bounds__(kF4Threads, 1)
gdn_tc_fwd4_kernel(const __grid_constant__ CUtensorMap x_map, const __grid_constant__ CUtensorMap y_map,
                   const void* __restrict__ x_, const __nv_bfloat16* __restrict__ planes,
                   const float* __restrict__ beta, long long n_pix, TcFlags f) {
  using L = Fwd4Smem<C>;
  constexpr int NCH = C / 32;  // 6 boxes per pass over a tile
  constexpr int kRowB = C * IoBytes<IO>::value;  // bytes per pixel row of x / y
  const uint8_t* x = static_cast<const uint8_t*>(x_);
  extern __shared__ __align__(1024) uint8_t smem[];
  float* beta_s = reinterpret_cast<float*>(smem + L::kOffBeta);
  uint64_t* mbars = reinterpret_cast<uint64_t*>(smem + L::kOffBar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + L::kOffBar + L::kNumBars * 8);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int r = tid & 127, h = (tid >> 7) & 3, gwarp = warp & 3;  // compute thread (r, h): pixel row r, column quarter h
  constexpr uint32_t kIdesc = umma_idesc(kTileM, C);
  auto bar = [&](int i) { return smem_u32(mbars + i); };
  {
    const uint4* src = reinterpret_cast<const uint4*>(planes);  // hi plane first
    uint4* dst = reinterpret_cast<uint4*>(smem + L::kOffBh);
    for (int i = tid; i < L::kPlaneB / 16; i += kF4Threads) dst[i] = src[i];
    for (int i = tid; i < C; i += kF4Threads) beta_s[i] = beta[i];
  }
  if (tid == 0) {
    for (int i = 0; i < L::kNumBars; ++i) {
      const int count = (i >= L::kBarY) ? kF4Compute / 32 : 1;  // y ready: one arrival per compute warp
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar(i)), "r"(count));
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;            // accumulator of tile t: columns (t & 1) * 256 ..
  const uint32_t lane_sel = (uint32_t)(gwarp * 32) << 16;
  const uint32_t b_hi = smem_u32(smem + L::kOffBh);
  const long long n_tiles = (n_pix + kTileM - 1) / kTileM;

  // A box ring of three slots: request n uses slot n % 3 in its (n / 3)-th round.
  auto load_boxes = [&](int ring, bool prefetch_l2) {  // ring 0: C boxes, 1: E boxes
    const int full0 = ring ? L::kBarEfull : L::kBarCfull, empty0 = ring ? L::kBarEempty : L::kBarCempty;
    uint32_t n = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      const int row0 = (int)(tile * kTileM);
      if (prefetch_l2) {  // the next tile of this CTA -> L2 (one contiguous block): its boxes become L2 hits
        const long long pn = (tile + gridDim.x) * kTileM;
        const long long rows = min((long long)kTileM, n_pix - pn);
        if (rows > 0)
          asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;" ::"l"(x + pn * kRowB),
                       "r"((uint32_t)(rows * kRowB)), "l"(kEvictLast)
                       : "memory");
      }
#pragma unroll 1
      for (int k = 0; k < NCH; ++k, ++n) {
        const uint32_t slot = n % 3u, round = n / 3u;
        if (round > 0) {
          if (!mbar_wait(bar(empty0 + slot), (round - 1u) & 1u)) __trap();
        }
        const uint32_t full = bar(full0 + slot);
        const uint32_t dst = smem_u32(smem + L::kOffRing + (ring * 3 + slot) * kF4Box);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full), "n"(Box<IO>::kBytes) : "memory");
        // x is read twice (C box, then E box about a tile later): the first read asks L2 to keep the lines, the
        // second releases them (ncu before the hints: 1.54x the algorithmic DRAM reads at 16.7 M pixels)
        asm volatile(
            "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;" ::"r"(dst),
            "l"(&x_map), "r"(k * 32), "r"(row0), "r"(full), "l"(ring ? kEvictFirst : kEvictLast)
            : "memory");
      }
    }
  };

  constexpr int W0 = kF4Compute / 32;  // first auxiliary warp
  if (warp == W0 + 1 || warp == W0 + 2) {
    // ---------------------------------- copy warps: C boxes / E boxes ----------------------------------
    if (lane == 0) load_boxes(warp - (W0 + 1), warp == W0 + 1);
    __syncwarp();
  } else if (warp == W0 + 3) {
    // ---------------------------------- gamma warp: lo-plane chunks ----------------------------------
    if (lane == 0) {
      const uint8_t* lo_plane = reinterpret_cast<const uint8_t*>(planes) + L::kPlaneB;
      uint32_t n = 0;  // chunks requested so far; chunk n uses buffer n & 1
      for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
#pragma unroll 1
        for (int c = 0; c < NCH; ++c, ++n) {
          const uint32_t buf = n & 1u;
          if (n >= 2) {  // the MMAs of chunk n - 2 (same buffer, same plane mbarrier) have completed
            if (!mbar_wait(bar(L::kBarPlane + buf), ((n >> 1) - 1u) & 1u)) __trap();
          }
          const uint32_t gfull = bar(L::kBarGfull + buf);
          asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(gfull), "n"(L::kGlo) : "memory");
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                           smem_u32(smem + L::kOffGlo + buf * L::kGlo)),
                       "l"(lo_plane + (size_t)c * L::kGlo), "n"(L::kGlo), "r"(gfull)
                       : "memory");
        }
      }
    }
    __syncwarp();
  } else if (warp == W0 + 4) {
    // ---------------------------------- store warp: y boxes ----------------------------------
    if (lane == 0) {
      uint32_t n = 0;
      for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int row0 = (int)(tile * kTileM);
#pragma unroll 1
        for (int k = 0; k < NCH; ++k, ++n) {
          const uint32_t slot = n % 3u, round = n / 3u;
          if (!mbar_wait(bar(L::kBarY + slot), round & 1u)) __trap();
          asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%1, %2}], [%3], %4;" ::"l"(&y_map),
                       "r"(k * 32), "r"(row0), "r"(smem_u32(smem + L::kOffRing + (3 + slot) * kF4Box)), "l"(kEvictFirst)
                       : "memory");
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // the box has been read: the slot is free
          asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar(L::kBarEempty + slot)) : "memory");
        }
      }
      asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
    __syncwarp();
  } else if (warp == W0) {
    // ------------------------------- MMA-issue warp -------------------------------
    uint32_t parg[2] = {0u, 0u};
    uint32_t n = 0;  // chunk counter = C box counter
    int t = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++t) {
      const uint32_t tmem_n = tmem_base + (uint32_t)(t & 1) * 256u;
#pragma unroll 1
      for (int c = 0; c < NCH; ++c, ++n) {
        const int pb = c & 1;
        asm volatile("bar.sync %0, %1;" ::"r"(2 + pb), "n"(kF4Sync) : "memory");  // planes of chunk c are written
        if (lane == 0) {
          // every compute thread is done with this C box: hand its slot back to the copy warp
          asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar(L::kBarCempty + n % 3u)) : "memory");
          if (!mbar_wait(bar(L::kBarGfull + pb), parg[pb])) __trap();
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t ph = smem_u32(smem + L::kOffP + pb * 2 * kF4Plane), pl = ph + kF4Plane;
          const uint32_t g_lo = smem_u32(smem + L::kOffGlo + pb * L::kGlo);
#pragma unroll
          for (int s2 = 0; s2 < 2; ++s2) {
            const uint64_t dah = umma_desc(ph + (uint32_t)(2 * s2) * kF4Kg, kF4Kg, 128);
            const uint64_t dal = umma_desc(pl + (uint32_t)(2 * s2) * kF4Kg, kF4Kg, 128);
            const uint64_t dbh = umma_desc(b_hi + (uint32_t)(c * 4 + 2 * s2) * (C * 16), C * 16, 128);
            const uint64_t dbl = umma_desc(g_lo + (uint32_t)(2 * s2) * (C * 16), C * 16, 128);
            umma_bf16(tmem_n, dah, dbh, kIdesc, (c | s2) ? 1u : 0u);
            umma_bf16(tmem_n, dal, dbh, kIdesc, 1u);
            umma_bf16(tmem_n, dah, dbl, kIdesc, 1u);
          }
          umma_commit(bar(L::kBarPlane + pb));
        }
        parg[pb] ^= 1u;
        __syncwarp();
      }
    }
  } else {
  // --------------------------------- compute warps ---------------------------------
  uint32_t parp[2] = {0u, 0u};
  uint32_t nc = 0, ne = 0;                     // C boxes converted / E boxes finished so far
  const int ckg = tid & 3, crow = tid >> 2;    // conversion item of a box: row crow, 8 channels

  auto convert = [&](int c, bool wait_planes) {
    const int pb = c & 1;
    const uint32_t slot = nc % 3u, round = nc / 3u;
    uint8_t* box = smem + L::kOffRing + slot * kF4Box;
    if (!mbar_wait(bar(L::kBarCfull + slot), round & 1u)) __trap();
    float v[8];
    box_load8<IO>(box, crow, ckg, v);
    if (wait_planes) {  // the plane buffer is still being read by the MMAs of the chunk two before this one
      if (!mbar_wait(bar(L::kBarPlane + pb), parp[pb])) __trap();
      parp[pb] ^= 1u;
    }
    uint8_t* ph = smem + L::kOffP + pb * 2 * kF4Plane;
    {
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = tc_pool<FAST>(v[e], f);
      uint4 hi, lo;
      split8(v, &hi, &lo);
      *reinterpret_cast<uint4*>(ph + ckg * kF4Kg + crow * 16) = hi;
      *reinterpret_cast<uint4*>(ph + kF4Plane + ckg * kF4Kg + crow * 16) = lo;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    asm volatile("bar.arrive %0, %1;" ::"r"(2 + pb), "n"(kF4Sync) : "memory");  // (also releases the box, see issue warp)
    ++nc;
  };

  // y = x / (beta + n) for box k (channels 32 k ..) of the tile whose accumulator starts at column `acc`:
  // thread (r, h) owns pixel row r and the 8 channels 32 k + 8 h ..
  auto finish_box = [&](int k, uint32_t acc) {
    const uint32_t slot = ne % 3u, round = ne / 3u;
    uint8_t* box = smem + L::kOffRing + (3 + slot) * kF4Box;
    uint32_t nacc[8];
    tmem_load<8>(tmem_base + acc + lane_sel + (uint32_t)(k * 32 + h * 8), nacc);
    if (!mbar_wait(bar(L::kBarEfull + slot), round & 1u)) __trap();
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    const float* bs = beta_s + k * 32 + h * 8;
    if constexpr (IO == 0) {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        float4* px = reinterpret_cast<float4*>(box_chunk<0>(box, r, 2 * h + j));
        const float4 xv = *px;
        const float4 bv = *reinterpret_cast<const float4*>(bs + 4 * j);  // same address in every lane: broadcast
        float4 o;
        o.x = tc_out<FAST>(xv.x, bv.x + __uint_as_float(nacc[4 * j]), f);
        o.y = tc_out<FAST>(xv.y, bv.y + __uint_as_float(nacc[4 * j + 1]), f);
        o.z = tc_out<FAST>(xv.z, bv.z + __uint_as_float(nacc[4 * j + 2]), f);
        o.w = tc_out<FAST>(xv.w, bv.w + __uint_as_float(nacc[4 * j + 3]), f);
        *px = o;
      }
    } else {  // 16-bit: the row's 8 channels are one 16-byte chunk, y written over x in place
      float xv[8], o[8];
      box_load8<IO>(box, r, h, xv);
#pragma unroll
      for (int e = 0; e < 8; ++e) o[e] = tc_out<FAST>(xv[e], bs[e] + __uint_as_float(nacc[e]), f);
      box_store8<IO>(box, r, h, o);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // y box -> TMA store
    __syncwarp();
    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar(L::kBarY + slot)) : "memory");
    ++ne;
  };

  int t = 0;
  for (long long tile = blockIdx.x;; tile += gridDim.x, ++t) {
    const bool has_cur = tile < n_tiles;   // tile t: converted now, accumulator (t & 1)
    const bool has_prev = t > 0;           // tile t - 1: finished now, accumulator ((t - 1) & 1)
    if (!has_cur && !has_prev) break;
    const uint32_t acc_prev = (uint32_t)((t - 1) & 1) * 256u;
    if (!has_cur) {  // drain: the last two commits cover every MMA of the last tile
#pragma unroll
      for (int pb = 0; pb < 2; ++pb) {
        if (!mbar_wait(bar(L::kBarPlane + pb), parp[pb])) __trap();
        parp[pb] ^= 1u;
      }
    }
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    // Chunks 0 and 1 of this tile first: their plane-buffer waits are the commits of the previous tile's last two
    // chunks, i.e. after them every MMA of the previous tile has completed.  Then box c - 2 of the previous tile is
    // finished BEFORE chunk c is converted, which gives the tensor pipe (the slower side) a box worth of slack.
    if (has_cur) {
      convert(0, t > 0);
      convert(1, t > 0);
    }
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
    for (int c = 2; c < NCH; ++c) {
      if (has_prev) finish_box(c - 2, acc_prev);
      if (has_cur) convert(c, true);
    }
    if (has_prev) {
      finish_box(NCH - 2, acc_prev);
      finish_box(NCH - 1, acc_prev);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");  // accumulator reads precede its next MMAs
    if (!has_cur) break;
  }
  }  // compute warps
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (tid < 32) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(*tmem_slot), "n"(512));
  }
}

// cuTensorMapEncodeTiled is a driver entry point; it is looked up through the runtime so that the library keeps
// linking against libcudart only.
typedef CUresult (*TensorMapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                      const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                      CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
TensorMapEncodeFn tensor_map_encoder() {
  static TensorMapEncodeFn encode = [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult st;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &st) != cudaSuccess ||
        st != cudaDriverEntryPointSuccess)
      fn = nullptr;
    (void)cudaGetLastError();
    return reinterpret_cast<TensorMapEncodeFn>(fn);
  }();
  return encode;
}

// Element type and swizzle of the [128 rows x 32 channels] activation boxes (see Box<IO>): 128-byte rows of float32
// with the 128-byte swizzle, or 64-byte rows of float16 / bfloat16 with the 64-byte swizzle.
template <int IO>
struct IoMap {
  static constexpr CUtensorMapDataType kType =
      IO == 0 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : (IO == 1 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
  static constexpr CUtensorMapSwizzle kSwizzle = IO == 0 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
};

inline int tensor_map_elem_bytes(CUtensorMapDataType t) { return t == CU_TENSOR_MAP_DATA_TYPE_FLOAT32 ? 4 : 2; }

// 2-D tensor map of a row-major [rows, cols] array of `type` elements with [box_rows x box_cols] boxes (zero fill).
int make_tensor_map_2d(CUtensorMap* map, const void* base, long long rows, int cols, int box_rows, int box_cols,
                       CUtensorMapDataType type, CUtensorMapSwizzle swizzle) {
  const TensorMapEncodeFn encode = tensor_map_encoder();
  if (!encode) return fail(TFCB_CUDA_ERROR, "cuTensorMapEncodeTiled is not available from this driver");
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)cols * tensor_map_elem_bytes(type)};
  const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1u, 1u};
  const CUresult rc = encode(map, type, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) return fail(TFCB_CUDA_ERROR, "cuTensorMapEncodeTiled failed (%d)", (int)rc);
  return TFCB_OK;
}

// 3-D view of a row-major [rows, cols] array as (32 channels, rows, cols / 32 chunks) with boxes of
// [chunks_per_box][box_rows][32 channels]: ONE copy instruction moves several of the kernels' [128 rows x 32 channels]
// boxes, which land back to back in shared memory exactly as separate 2-D boxes would.
// (The SM's async-copy engine retires ~2.5 copy instructions per microsecond whatever their size -- 0.39 us per 16 KB
// box, tools/tma_probe.py -- so the number of instructions per tile, not the bytes, bounded the box-fed kernels.)
int make_tensor_map_3d(CUtensorMap* map, const void* base, long long rows, int cols, int box_rows, int chunks_per_box,
                       CUtensorMapDataType type, CUtensorMapSwizzle swizzle) {
  const TensorMapEncodeFn encode = tensor_map_encoder();
  if (!encode) return fail(TFCB_CUDA_ERROR, "cuTensorMapEncodeTiled is not available from this driver");
  const int eb = tensor_map_elem_bytes(type);
  const cuuint64_t dims[3] = {32u, (cuuint64_t)rows, (cuuint64_t)(cols / 32)};
  const cuuint64_t strides[2] = {(cuuint64_t)cols * eb, 32u * (cuuint64_t)eb};  // row stride, chunk stride
  const cuuint32_t box[3] = {32u, (cuuint32_t)box_rows, (cuuint32_t)chunks_per_box};
  const cuuint32_t estr[3] = {1u, 1u, 1u};
  const CUresult rc = encode(map, type, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) return fail(TFCB_CUDA_ERROR, "cuTensorMapEncodeTiled (3-D) failed (%d)", (int)rc);
  return TFCB_OK;
}

// [128 x 32] activation boxes of a row-major [n_pix, C] array of IO elements
template <int IO>
int make_box_map(CUtensorMap* map, const void* base, long long n_pix, int C) {
  return make_tensor_map_2d(map, base, n_pix, C, kTileM, 32, IoMap<IO>::kType, IoMap<IO>::kSwizzle);
}

template <bool FAST, int IO>
int launch_tc_fwd4(const void* x, const float* gamma, const float* beta, void* y, long long n_pix, TcFlags f,
                   cudaStream_t s) {
  constexpr int C = 192;
  using L = Fwd4Smem<C>;
  CUtensorMap x_map, y_map;
  TFCB_TRY(make_box_map<IO>(&x_map, x, n_pix, C));
  TFCB_TRY(make_box_map<IO>(&y_map, y, n_pix, C));
  __nv_bfloat16* planes = nullptr;
  TFCB_TRY(dev_alloc((void**)&planes, (size_t)2 * C * C * sizeof(__nv_bfloat16), s));
  gdn_tc_prep_kernel<<<((C / 8) * C + 255) / 256, 256, 0, s>>>(gamma, C, planes);
  TFCB_LAUNCHED();
  cudaError_t e = cudaFuncSetAttribute(gdn_tc_fwd4_kernel<C, FAST, IO>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kBytes);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    dev_free(planes, s);
    return fail(TFCB_CUDA_ERROR, "cannot reserve %d bytes of shared memory: %s", L::kBytes, cudaGetErrorString(e));
  }
  const long long n_tiles = (n_pix + kTileM - 1) / kTileM;
  const int grid = (int)std::min<long long>(n_tiles, device_sm_count());
  gdn_tc_fwd4_kernel<C, FAST, IO><<<grid, kF4Threads, L::kBytes, s>>>(x_map, y_map, x, planes, beta, n_pix, f);
  TFCB_LAUNCHED();
  e = cudaGetLastError();
  dev_free(planes, s);
  if (e != cudaSuccess) return fail(TFCB_CUDA_ERROR, "GDN tensor-core kernel launch failed: %s", cudaGetErrorString(e));
  return TFCB_OK;
}

// =============================================================================================
// Backward.  Per 128-pixel tile:
//
//   n  = beta + p . gamma                 MMA1   A = p planes (K-major),        B = gamma (K-major)
//   q  = dL/dn (elementwise, from g, x, n)
//   dp = q . gamma^T                      MMA2   A = q planes (K-major),        B = gamma^T
//   dx = g / m + dpool/du * dp            (IGDN: g * m + ...; 0 where the rectifier cuts x off)
//   dgamma[j, i] += sum_pix p[pix, j] q[pix, i]
//                                         MMA3   A = p planes (MN-major view),  B = q planes (MN-major view)
//   dbeta[i] += sum_pix q[pix, i]
//
// The MN-major views reuse the very same shared-memory planes: a K-major plane [k / 8][row][8] read with the
// "transposed" descriptor (instruction-descriptor bits 15 / 16) is the operand with the roles of row and k
// swapped (core matrix = 8 k-rows of 16 bytes, LBO = 128 B between k groups, SBO = plane row-group stride).
// =============================================================================================
constexpr int kKg = kTileM * 16 + 16;  // byte stride between 8-channel groups of an operand plane: one 16-byte row
                                       // of padding makes the row-per-lane stores bank-conflict free;
                                       // the descriptors take it as LBO (K-major view) or SBO (MN-major view)

// dgamma accumulates in TMEM across a CTA's tiles.  The tensor core adds every MMA into the fp32 accumulator with
// TRUNCATION, so a long-running accumulator shrinks by ~2^-25 per accumulation step: measured 6e-6 of max |dgamma|
// after one tile per CTA, 6.4e-5 after 110 (2 M pixels), linear in the tile count.  The accumulator is therefore
// flushed into the CTA's fp32 partial in global memory (round-to-nearest adds, L2 resident) every kDgFlush tiles
// and restarted; the drift stays below 3e-6 at any pixel count.
constexpr int kDgFlush = 4;

// q = dL/dn = -g u / n^2 (IGDN: g u; epsilon = 1/2: -g u / (2 n^1.5), IGDN g u / (2 sqrt(n))), u = x or relu(x)
template <bool FAST>
__device__ __forceinline__ float tc_dl_dn(float g, float x, float n, const TcFlags& f) {
  const float u = (!FAST && f.rectify) ? fmaxf(x, 0.f) : x;
  const float r = rcp_approx(n);
  if (FAST || f.eps_mode == 1) return f.inverse ? g * u : -g * u * r * r;
  const float rs = rsqrtf(n);
  return f.inverse ? 0.5f * g * u * rs : -0.5f * g * u * r * rs;
}

// The direct term of dx: g / m (IGDN: g * m), m = n or sqrt(n)
template <bool FAST>
__device__ __forceinline__ float tc_direct(float g, float n, const TcFlags& f) {
  if (FAST || f.eps_mode == 1) return f.inverse ? g * n : g * rcp_approx(n);
  return f.inverse ? g * sqrtf(n) : g * rsqrtf(n);
}

// dx = direct + dpool/du * dp, 0 where the rectifier cuts x off.  The default GDN (FAST) does not call this: its
// dpool/du is sign(x), which the kernels carry in the low mantissa bits of the direct term instead of x.
__device__ __forceinline__ float tc_dx(float direct, float x, float dp, const TcFlags& f) {
  const float u = f.rectify ? fmaxf(x, 0.f) : x;
  float dpool;
  if (f.alpha_mode == 1) dpool = f.rectify ? 1.f : ((u > 0.f) ? 1.f : ((u < 0.f) ? -1.f : 0.f));
  else dpool = 2.f * u;
  return (f.rectify && !(x > 0.f)) ? 0.f : direct + dpool * dp;
}

__device__ __forceinline__ void tmem_store8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}

// gamma [C, C] -> bf16 K chunks for the streamed kernels: for t in {gamma (MMA1: K = j), gamma^T (MMA2: K = i)} and each
// 32-channel K chunk c one block [hi: 4 groups x C x 8][lo: the same], i.e. chunk (t, c) is ONE contiguous copy of
// C * 128 bytes (a copy instruction costs the SM's copy engine ~0.35 us whatever its size).  INTERLEAVED = false keeps
// four whole planes [gamma hi, gamma lo, gamma^T hi, gamma^T lo] (the C = 192 dx kernel keeps a whole hi plane resident).
template <bool INTERLEAVED>
__global__ void gdn_tc_prep2_kernel(const float* __restrict__ gamma, int C, __nv_bfloat16* __restrict__ planes) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;  // over (k / 8, n)
  if (idx >= (C / 8) * C) return;
  const int kc = idx / C, n = idx % C;
  float v[8], w[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    v[e] = gamma[(kc * 8 + e) * C + n];  // k = j (input channel), n = i
    w[e] = gamma[n * C + kc * 8 + e];    // k = i, n = j
  }
  uint4* out = reinterpret_cast<uint4*>(planes);
  const size_t plane16 = (size_t)C * C / 8;  // 16-byte units per plane
  uint4 hi, lo;
  split8(v, &hi, &lo);
  if (INTERLEAVED) {
    const size_t chunk16 = (size_t)4 * C;  // units of one chunk of one plane
    const size_t at = ((size_t)(kc / 4) * 2) * chunk16 + (size_t)(kc % 4) * C + n;
    out[at] = hi;
    out[at + chunk16] = lo;
    split8(w, &hi, &lo);
    out[2 * plane16 + at] = hi;
    out[2 * plane16 + at + chunk16] = lo;
  } else {
    out[idx] = hi;
    out[plane16 + idx] = lo;
    split8(w, &hi, &lo);
    out[2 * plane16 + idx] = hi;
    out[3 * plane16 + idx] = lo;
  }
}

// =============================================================================================
// Backward, C = 128: one fused kernel.
//
// Everything that touches HBM is an asynchronous 2-D TMA box, every compute thread (r, h) owns pixel row r (= its
// TMEM lane) and 8 of the 32 channels of a box, so there are no staging transposes and no CTA-wide barriers, and x
// and dy are read exactly once:
//
//   conv(t)   x boxes -> p = pool(x) hi / lo planes (whole K)            -> MMA1  n = p . gamma
//             the raw x values are parked in 128 spare TMEM columns (tcgen05.st) for pass 2
//   pass2(t)  g boxes + n, x from TMEM -> q hi / lo planes (whole tile, written 32 channels at a time)
//                                                                         -> MMA2  dp += q_chunk . gamma^T  per chunk
//             the direct term g / m (IGDN: g * m) goes back into n's TMEM columns; for the default GDN (FAST) with
//             sign(x) in the two low mantissa bits (2 ulp, the contract is 1e-5), so that its dx pass needs neither
//             x nor g again
//   pass3(t)  dx = direct + dpool/du * dp  from TMEM -> box -> TMA store;  meanwhile
//                                                                         -> MMA3  dgamma += p^T q, 24 full-width MMAs
//             (the variants read dpool/du off the parked x: the next tile's conversion overwrites it only after
//             this pass)
//
// (With 32-channel q buffers MMA3 was 96 MMAs of N = 32 per tile, each re-reading its 4 KB A operand from shared
// memory for 16 cycles of math: switching them off saved 20 % of the kernel.)  The whole-tile q planes take the
// place of resident gamma planes: gamma (and gamma^T for MMA2) is streamed from L2 in 32-channel K chunks
// (16 KB hi + lo, double buffered) by a "gamma" warp, 128 KB per tile.
// One ring of four 16 KB boxes serves every box request in program order: g x 4 (pass 2), output x 4 (pass 3),
// x x 4 (conversion of the CTA's next tile).  TMEM: n | dp | dgamma partial | parked x (4 x 128 columns).
// HBM traffic: x, dy in, dx out, nothing else.
// =============================================================================================
constexpr int kB3Compute = 512;                // 16 compute warps
constexpr int kB3Threads = kB3Compute + 160;   // + two MMA-issue warps, box-copy, gamma and store warps
constexpr int kB3SyncA = kB3Compute + 32;      // compute + first issue warp
constexpr int kB3SyncB = kB3Compute + 64;      // compute + both issue warps (last q chunk of a tile)
constexpr int kB3Slots = 4;

struct BwdFusedSmem {
  static constexpr int C = 128;
  static constexpr int kGChunk = 4 * C * 16;                      // one 32-channel K chunk of one gamma plane (8 KB)
  static constexpr int kOffRing = 0;                              // [4] boxes (1024-byte aligned: swizzle atom)
  static constexpr int kOffG = kOffRing + kB3Slots * kF4Box;      // [2 buffers][hi, lo] gamma K chunks
  static constexpr int kPlane = (C / 8) * kKg;                    // one whole-K operand plane (p or q, hi or lo)
  static constexpr int kOffPh = kOffG + 4 * kGChunk;
  static constexpr int kOffPl = kOffPh + kPlane;
  static constexpr int kOffQh = kOffPl + kPlane;
  static constexpr int kOffQl = kOffQh + kPlane;
  static constexpr int kOffBeta = kOffQl + kPlane;
  static constexpr int kOffDbeta = kOffBeta + C * 4;
  static constexpr int kOffBar = kOffDbeta + C * 4;
  // mbarriers: full[4], empty[4], yready[4], gfull[2], gfree[2], nfull, dpfull, m3done; then the TMEM slot
  static constexpr int kBarFull = 0, kBarEmpty = 4, kBarY = 8, kBarGfull = 12, kBarGfree = 14, kBarN = 16, kBarDp = 17,
                       kBarM3 = 18, kNumBars = 19;
  static constexpr int kBytes = kOffBar + kNumBars * 8 + 16;
  static_assert(kOffG % 128 == 0 && kOffPh % 16 == 0 && kOffQh % 16 == 0 && kOffBar % 8 == 0, "alignment");
  static_assert(kBytes <= 232448, "shared memory budget");
};

template <bool FAST, int IO>
__global__ void __launch_bounds__(kB3Threads, 1)
gdn_tc_bwd3_kernel(const __grid_constant__ CUtensorMap x_map, const __grid_constant__ CUtensorMap g_map,
                   const __grid_constant__ CUtensorMap dx_map, const void* __restrict__ x_, const void* __restrict__ dy_,
                   const __nv_bfloat16* __restrict__ planes, const float* __restrict__ beta, float* __restrict__ part_g,
                   float* __restrict__ part_b, long long n_pix, TcFlags f) {
  using L = BwdFusedSmem;
  constexpr int C = L::C, NCH = C / 32;
  constexpr int kRowB = C * IoBytes<IO>::value;  // bytes per pixel row of x / dy / dx
  const uint8_t* x = static_cast<const uint8_t*>(x_);
  const uint8_t* dy = static_cast<const uint8_t*>(dy_);
  extern __shared__ __align__(1024) uint8_t smem[];
  float* beta_s = reinterpret_cast<float*>(smem + L::kOffBeta);
  float* dbeta_s = reinterpret_cast<float*>(smem + L::kOffDbeta);
  uint64_t* mbars = reinterpret_cast<uint64_t*>(smem + L::kOffBar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + L::kOffBar + L::kNumBars * 8);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int r = tid & 127, h = (tid >> 7) & 3, gwarp = warp & 3;  // compute thread (r, h): pixel row r, channel octet h of a box
  auto bar = [&](int i) { return smem_u32(mbars + i); };
  for (int i = tid; i < C; i += kB3Threads) {
    beta_s[i] = beta[i];
    dbeta_s[i] = 0.f;
  }
  if (tid == 0) {
    for (int i = 0; i < L::kNumBars; ++i) {
      const int count = (i >= L::kBarY && i < L::kBarGfull) ? kB3Compute / 32 : 1;  // y ready: one arrival per compute warp
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar(i)), "r"(count));
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_n = *tmem_slot, tmem_dp = tmem_n + C, tmem_dg = tmem_n + 2 * C, tmem_x = tmem_n + 3 * C;
  const uint32_t lane_sel = (uint32_t)(gwarp * 32) << 16;
  const uint32_t p_hi = smem_u32(smem + L::kOffPh), p_lo = smem_u32(smem + L::kOffPl);
  const uint32_t q_hi = smem_u32(smem + L::kOffQh), q_lo = smem_u32(smem + L::kOffQl);
  const long long n_tiles = (n_pix + kTileM - 1) / kTileM;
  const long long first = blockIdx.x;
  // The dgamma accumulator is flushed every kDgFlush tiles; CTAs take turns (all 148 flushing in the same
  // microsecond made the L2 the bottleneck of the flush)
  const int fphase = (int)(blockIdx.x % kDgFlush);
  // Box requests are numbered in program order; request n uses ring slot n % 4 in its (n / 4)-th round:
  //   4 x boxes (conversion of the CTA's first tile), then per tile  g x 4, out x 4, (x of the next tile) x 4.
  // Gamma K chunks likewise, buffer m % 2:  4 chunks of gamma (MMA1 of the first tile), then per tile 4 chunks of
  // gamma^T (MMA2), 4 chunks of gamma (MMA1 of the next tile).
  constexpr int W0 = kB3Compute / 32;  // first auxiliary warp

  if (warp == W0 + 2) {
    // ---------------------------------- box-copy warp ----------------------------------
    if (lane == 0) {
      uint32_t n = 0;
      auto acquire = [&]() {
        const uint32_t slot = n & 3u, round = n >> 2;
        if (round > 0) {
          if (!mbar_wait(bar(L::kBarEmpty + slot), (round - 1u) & 1u)) __trap();
        }
        return slot;
      };
      auto load = [&](const CUtensorMap* map, int c, int row0) {
        const uint32_t slot = acquire();
        const uint32_t full = bar(L::kBarFull + slot);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full), "n"(Box<IO>::kBytes) : "memory");
        asm volatile(
            "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;" ::"r"(
                smem_u32(smem + L::kOffRing + slot * kF4Box)),
            "l"(map), "r"(c * 32), "r"(row0), "r"(full), "l"(kEvictFirst)
            : "memory");
        ++n;
      };
      auto prefetch_tile = [&](const uint8_t* base, long long tile) {  // one contiguous block -> L2
        const long long p0 = tile * kTileM;
        const long long rows = min((long long)kTileM, n_pix - p0);
        if (rows > 0)
          asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;" ::"l"(base + p0 * kRowB),
                       "r"((uint32_t)(rows * kRowB)), "l"(kEvictLast)
                       : "memory");
      };
      if (first < n_tiles) {
        prefetch_tile(dy, first);
#pragma unroll 1
        for (int c = 0; c < NCH; ++c) load(&x_map, c, (int)(first * kTileM));
      }
      for (long long tile = first; tile < n_tiles; tile += gridDim.x) {
        const long long next = tile + gridDim.x;
        const bool has_next = next < n_tiles;
        const int row0 = (int)(tile * kTileM);
        if (has_next) {  // the next tile of this CTA -> L2: its boxes become L2 hits
          prefetch_tile(x, next);
          prefetch_tile(dy, next);
        }
#pragma unroll 1
        for (int c = 0; c < NCH; ++c) load(&g_map, c, row0);
#pragma unroll 1
        for (int c = 0; c < NCH; ++c) {
          const uint32_t slot = acquire();      // output box: nothing to load, the slot only has to be free
          asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar(L::kBarFull + slot)) : "memory");
          ++n;
        }
        if (has_next) {
#pragma unroll 1
          for (int c = 0; c < NCH; ++c) load(&x_map, c, (int)(next * kTileM));
        }
      }
    }
    __syncwarp();
  } else if (warp == W0 + 3) {
    // ---------------------------------- gamma warp: K chunks of gamma / gamma^T ----------------------------------
    if (lane == 0) {
      const uint8_t* gp = reinterpret_cast<const uint8_t*>(planes);
      constexpr size_t kPlaneBytes = (size_t)C * C * 2;
      uint32_t m = 0;
      auto chunk = [&](int transposed, int c) {
        const uint32_t buf = m & 1u;
        if (m >= 2) {  // the MMAs of chunk m - 2 (same buffer) have completed
          if (!mbar_wait(bar(L::kBarGfree + buf), ((m >> 1) - 1u) & 1u)) __trap();
        }
        const uint32_t gfull = bar(L::kBarGfull + buf);
        const uint32_t dst = smem_u32(smem + L::kOffG + buf * 2 * L::kGChunk);
        // chunk (t, c) = [hi 8 KB][lo 8 KB], contiguous in the prepared buffer: one copy
        const uint8_t* src = gp + (size_t)(2 * transposed) * kPlaneBytes + (size_t)c * (2 * L::kGChunk);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(gfull), "n"(2 * L::kGChunk) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst),
                     "l"(src), "n"(2 * L::kGChunk), "r"(gfull), "l"(kEvictLast)
                     : "memory");
        ++m;
      };
      if (first < n_tiles) {
#pragma unroll 1
        for (int c = 0; c < NCH; ++c) chunk(0, c);
      }
      for (long long tile = first; tile < n_tiles; tile += gridDim.x) {
#pragma unroll 1
        for (int c = 0; c < NCH; ++c) chunk(1, c);
        if (tile + gridDim.x < n_tiles) {
#pragma unroll 1
          for (int c = 0; c < NCH; ++c) chunk(0, c);
        }
      }
    }
    __syncwarp();
  } else if (warp == W0 + 4) {
    // ---------------------------------- store warp: dx boxes ----------------------------------
    if (lane == 0) {
      uint32_t n = (first < n_tiles) ? (uint32_t)NCH : 0u;
      uint32_t ypar = 0u;  // per-slot phase of the y-ready barrier (a slot is an output box only now and then)
      for (long long tile = first; tile < n_tiles; tile += gridDim.x) {
        const bool has_next = tile + gridDim.x < n_tiles;
        const int row0 = (int)(tile * kTileM);
        n += NCH;
#pragma unroll 1
        for (int c = 0; c < NCH; ++c, ++n) {
          const uint32_t slot = n & 3u;
          if (!mbar_wait(bar(L::kBarY + slot), (ypar >> slot) & 1u)) __trap();
          ypar ^= 1u << slot;
          asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%1, %2}], [%3], %4;" ::"l"(&dx_map),
                       "r"(c * 32), "r"(row0), "r"(smem_u32(smem + L::kOffRing + slot * kF4Box)), "l"(kEvictFirst)
                       : "memory");
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // the box has been read: the slot is free
          asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar(L::kBarEmpty + slot)) : "memory");
        }
        if (has_next) n += NCH;
      }
      asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
    __syncwarp();
  } else if (warp == W0) {
    // ------------------------------- first MMA-issue warp: MMA1, MMA2 (K-chunked, gamma streamed) ------------------
    constexpr uint32_t kIdesc = umma_idesc(kTileM, C);  // A, B both K-major
    uint32_t n = 0, m = 0;
    // six MMAs of one 32-channel K chunk: A planes (hi, lo) x gamma chunk (hi, lo), three products
    auto chunk_mmas = [&](uint32_t a_hi, uint32_t a_lo, uint32_t acc, bool first_chunk) {
      const uint32_t buf = m & 1u;
      if (!mbar_wait(bar(L::kBarGfull + buf), (m >> 1) & 1u)) __trap();
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t g_hi = smem_u32(smem + L::kOffG + buf * 2 * L::kGChunk), g_lo = g_hi + L::kGChunk;
#pragma unroll
      for (int s2 = 0; s2 < 2; ++s2) {
        const uint64_t dah = umma_desc(a_hi + (uint32_t)(2 * s2) * kKg, kKg, 128);
        const uint64_t dal = umma_desc(a_lo + (uint32_t)(2 * s2) * kKg, kKg, 128);
        const uint64_t dbh = umma_desc(g_hi + (uint32_t)(2 * s2) * (C * 16), C * 16, 128);
        const uint64_t dbl = umma_desc(g_lo + (uint32_t)(2 * s2) * (C * 16), C * 16, 128);
        umma_bf16(acc, dah, dbh, kIdesc, (first_chunk && s2 == 0) ? 0u : 1u);
        umma_bf16(acc, dal, dbh, kIdesc, 1u);
        umma_bf16(acc, dah, dbl, kIdesc, 1u);
      }
      umma_commit(bar(L::kBarGfree + buf));
      ++m;
    };
    auto release = [&](uint32_t req) {
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar(L::kBarEmpty + (req & 3u))) : "memory");
    };
    auto mma1_tile = [&]() {  // n = p . gamma of the tile being converted, K chunk by K chunk
#pragma unroll 1
      for (int c = 0; c < NCH; ++c, ++n) {
        asm volatile("bar.sync %0, %1;" ::"r"(2 + c), "n"(kB3SyncA) : "memory");  // p planes of chunk c are written
        if (lane == 0) {
          release(n);
          chunk_mmas(p_hi + (uint32_t)(4 * c) * kKg, p_lo + (uint32_t)(4 * c) * kKg, tmem_n, c == 0);
          if (c == NCH - 1) umma_commit(bar(L::kBarN));
        }
        __syncwarp();
      }
    };
    if (first < n_tiles) mma1_tile();
    for (long long tile = first; tile < n_tiles; tile += gridDim.x) {
      const bool has_next = tile + gridDim.x < n_tiles;
#pragma unroll 1
      for (int c = 0; c < NCH; ++c, ++n) {
        if (c == NCH - 1) asm volatile("bar.sync %0, %1;" ::"r"(6 + c), "n"(kB3SyncB) : "memory");
        else asm volatile("bar.sync %0, %1;" ::"r"(6 + c), "n"(kB3SyncA) : "memory");  // q planes of chunk c are written
        if (lane == 0) {
          release(n);  // the g box of this chunk
          // MMA2: dp[pix, j] += sum_{i in chunk} q[pix, i] gamma[j, i]
          chunk_mmas(q_hi + (uint32_t)(4 * c) * kKg, q_lo + (uint32_t)(4 * c) * kKg, tmem_dp, c == 0);
          if (c == NCH - 1) umma_commit(bar(L::kBarDp));  // dp is complete: the dx pass may start
        }
        __syncwarp();
      }
      n += NCH;  // the output boxes: handed back by the store warp
      if (has_next) mma1_tile();
    }
  } else if (warp == W0 + 1) {
    // ------------------------------- second MMA-issue warp: MMA3, once per tile -------------------------------
    constexpr uint32_t kIdesc3 = umma_idesc(C, C) | (1u << 15) | (1u << 16);    // A = p^T, B = q (both MN-major views)
    int t = 0;
    for (long long tile = first; tile < n_tiles; tile += gridDim.x, ++t) {
      asm volatile("bar.sync %0, %1;" ::"r"(6 + NCH - 1), "n"(kB3SyncB) : "memory");  // the whole tile of q is written
      if (lane == 0) {
        // let the tile's last MMA2s through first: the dx pass waits for them, nothing waits for MMA3 until the next
        // conversion (both issue warps leave the same barrier; 24 MMAs ahead of 6 cost the dx pass ~0.8 us per tile)
        if (!mbar_wait(bar(L::kBarDp), (uint32_t)t & 1u)) __trap();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // dgamma[j, i] += sum_pix p[pix, j] q[pix, i]   (K = pix: 8 steps of 16)
        const bool restart = (t == 0) || (((t + fphase) % kDgFlush) == 0);  // first MMA after a flush
#pragma unroll
        for (int s = 0; s < kTileM / 16; ++s) {
          const uint32_t koff = (uint32_t)(s * 16) * 16u;
          const uint64_t dah = umma_desc(p_hi + koff, 128, kKg);
          const uint64_t dal = umma_desc(p_lo + koff, 128, kKg);
          const uint64_t dbh = umma_desc(q_hi + koff, 128, kKg);
          const uint64_t dbl = umma_desc(q_lo + koff, 128, kKg);
          umma_bf16(tmem_dg, dah, dbh, kIdesc3, (restart && s == 0) ? 0u : 1u);
          umma_bf16(tmem_dg, dal, dbh, kIdesc3, 1u);
          umma_bf16(tmem_dg, dah, dbl, kIdesc3, 1u);
        }
        umma_commit(bar(L::kBarM3));
      }
      __syncwarp();
    }
  } else if (warp < W0) {
  // --------------------------------- compute warps ---------------------------------
  uint32_t n = 0;
  float dbeta_acc[NCH][8];  // channels 32 c + 8 h + e, summed over this thread's rows
#pragma unroll
  for (int c = 0; c < NCH; ++c)
#pragma unroll
    for (int e = 0; e < 8; ++e) dbeta_acc[c][e] = 0.f;
  bool flushed = false;  // the global partial holds earlier flushes
  // The accumulator (TMEM lane = input channel j, 32 columns per thread) is transposed through the dead q planes
  // ([128][128] fp32, 16-byte units XOR-swizzled by the row) so that every warp adds 512 contiguous bytes to the CTA's
  // partial: with one row per lane each vector add touched 32 different L2 lines (8 % of the kernel).
  auto flush_dgamma = [&]() {
    uint8_t* stage = smem + L::kOffQh;
#pragma unroll
    for (int cb = 0; cb < 2; ++cb) {
      uint32_t a[16];
      tmem_load<16>(tmem_dg + lane_sel + (uint32_t)(h * 32 + cb * 16), a);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
      for (int i = 0; i < 4; ++i)
        *reinterpret_cast<uint4*>(stage + r * 512 + (((h * 8 + cb * 4 + i) ^ (r & 7)) << 4)) =
            make_uint4(a[4 * i], a[4 * i + 1], a[4 * i + 2], a[4 * i + 3]);
    }
    asm volatile("bar.sync 1, %0;" ::"n"(kB3Compute) : "memory");
    float* pg = part_g + (long long)blockIdx.x * C * C;
#pragma unroll
    for (int it = 0; it < (C * C / 4) / kB3Compute; ++it) {
      const int item = it * kB3Compute + tid, row = item >> 5, c4 = item & 31;
      const uint4 v = *reinterpret_cast<const uint4*>(stage + row * 512 + ((c4 ^ (row & 7)) << 4));
      float* dst = pg + row * C + c4 * 4;
      // first flush: plain stores; later ones: fire-and-forget vector adds in L2
      if (!flushed)
        asm volatile("st.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
      else
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
    }
    flushed = true;
  };

  // One tile: p = pool(x) -> hi / lo planes chunk by chunk (each chunk arrives on its own named barrier), raw x -> TMEM
  auto conv_tile = [&]() {
#pragma unroll 1
    for (int c = 0; c < NCH; ++c, ++n) {
      const uint32_t slot = n & 3u, round = n >> 2;
      uint8_t* box = smem + L::kOffRing + slot * kF4Box;
      if (!mbar_wait(bar(L::kBarFull + slot), round & 1u)) __trap();
      float v[8];
      box_load8<IO>(box, r, h, v);
      uint32_t raw[8];  // x widened to float32 is what pass 2 and the variants' pass 3 read back
#pragma unroll
      for (int e = 0; e < 8; ++e) raw[e] = __float_as_uint(v[e]);
      tmem_store8(tmem_x + lane_sel + (uint32_t)(c * 32 + h * 8), raw);
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = tc_pool<FAST>(v[e], f);
      uint4 hi, lo;
      split8(v, &hi, &lo);
      *reinterpret_cast<uint4*>(smem + L::kOffPh + (4 * c + h) * kKg + r * 16) = hi;
      *reinterpret_cast<uint4*>(smem + L::kOffPl + (4 * c + h) * kKg + r * 16) = lo;
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      asm volatile("bar.arrive %0, %1;" ::"r"(2 + c), "n"(kB3SyncA) : "memory");  // (also releases the box, see issue warp)
    }
  };

  if (first < n_tiles) conv_tile();
  int t = 0;
  for (long long tile = first; tile < n_tiles; tile += gridDim.x, ++t) {
    const bool has_next = tile + gridDim.x < n_tiles;
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");  // this thread's parked x values are in TMEM
    if (!mbar_wait(bar(L::kBarN), (uint32_t)t & 1u)) __trap();  // MMA1 of this tile has completed
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    // ---- pass 2: q = dL/dn -> q planes; the direct term (FAST: and sign(x)) goes back into n's columns ----
#pragma unroll
    for (int c = 0; c < NCH; ++c, ++n) {
      const uint32_t slot = n & 3u;
      const uint32_t col = lane_sel + (uint32_t)(c * 32 + h * 8);
      uint32_t nacc[8], xraw[8];
      tmem_load<8>(tmem_n + col, nacc);
      tmem_load<8>(tmem_x + col, xraw);
      if (!mbar_wait(bar(L::kBarFull + slot), (n >> 2) & 1u)) __trap();
      uint8_t* bg = smem + L::kOffRing + slot * kF4Box;
      float gs[8];
      box_load8<IO>(bg, r, h, gs);
      const float4 bv0 = *reinterpret_cast<const float4*>(beta_s + c * 32 + h * 8);      // same address in every lane
      const float4 bv1 = *reinterpret_cast<const float4*>(beta_s + c * 32 + h * 8 + 4);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      const float bs[8] = {bv0.x, bv0.y, bv0.z, bv0.w, bv1.x, bv1.y, bv1.z, bv1.w};
      float q[8];
      uint32_t dbits[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float xe = __uint_as_float(xraw[e]);
        const float nn = bs[e] + __uint_as_float(nacc[e]);
        q[e] = tc_dl_dn<FAST>(gs[e], xe, nn, f);
        dbits[e] = __float_as_uint(tc_direct<FAST>(gs[e], nn, f));
        if (FAST) dbits[e] = (dbits[e] & ~3u) | ((xe > 0.f) ? 1u : ((xe < 0.f) ? 2u : 0u));
        dbeta_acc[c][e] += q[e];
      }
      uint4 hi, lo;
      split8(q, &hi, &lo);
      *reinterpret_cast<uint4*>(smem + L::kOffQh + (4 * c + h) * kKg + r * 16) = hi;
      *reinterpret_cast<uint4*>(smem + L::kOffQl + (4 * c + h) * kKg + r * 16) = lo;
      tmem_store8(tmem_n + col, dbits);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      if (c == NCH - 1) asm volatile("bar.arrive %0, %1;" ::"r"(6 + c), "n"(kB3SyncB) : "memory");
      else asm volatile("bar.arrive %0, %1;" ::"r"(6 + c), "n"(kB3SyncA) : "memory");  // (also releases the g box)
    }
    // ---- pass 3: dx = direct + dpool/du * dp, from TMEM only ----
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");  // this thread's direct terms are in TMEM
    if (!mbar_wait(bar(L::kBarDp), (uint32_t)t & 1u)) __trap();  // every MMA2 of this tile has completed
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
    for (int c = 0; c < NCH; ++c, ++n) {
      const uint32_t slot = n & 3u, round = n >> 2;
      uint32_t d[8], p[8], xraw[8];
      tmem_load<8>(tmem_n + lane_sel + (uint32_t)(c * 32 + h * 8), d);
      tmem_load<8>(tmem_dp + lane_sel + (uint32_t)(c * 32 + h * 8), p);
      if (!FAST) tmem_load<8>(tmem_x + lane_sel + (uint32_t)(c * 32 + h * 8), xraw);
      uint8_t* box = smem + L::kOffRing + slot * kF4Box;
      if (!mbar_wait(bar(L::kBarFull + slot), round & 1u)) __trap();  // the slot's previous user has left
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      float o[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        if (FAST) {
          const uint32_t code = d[e] & 3u;
          const float s = (code == 1u) ? 1.f : ((code == 2u) ? -1.f : 0.f);
          o[e] = fmaf(s, __uint_as_float(p[e]), __uint_as_float(d[e]));
        } else {
          o[e] = tc_dx(__uint_as_float(d[e]), __uint_as_float(xraw[e]), __uint_as_float(p[e]), f);
        }
      }
      box_store8<IO>(box, r, h, o);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // dx box -> TMA store
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar(L::kBarY + slot)) : "memory");
    }
    // MMA3 of this tile has completed: the p and q planes are dead, the dgamma accumulator is up to date
    if (!mbar_wait(bar(L::kBarM3), (uint32_t)t & 1u)) __trap();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (((t + fphase) % kDgFlush) == kDgFlush - 1) flush_dgamma();
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");  // TMEM reads precede the next tile's MMAs
    if (has_next) conv_tile();
  }

  // ---- this CTA's partial sums ----
  if (t > 0) {
    if (((t + fphase) % kDgFlush) != 0) flush_dgamma();  // tiles since the last flush
    // dbeta: the 32 lanes of a warp hold the same channels (32 c + 8 h + e) for 32 different rows
#pragma unroll
    for (int c = 0; c < NCH; ++c)
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        float v = dbeta_acc[c][e];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
        if (lane == 0) atomicAdd(dbeta_s + c * 32 + h * 8 + e, v);
      }
  }
  }  // compute warps
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (tid < C) part_b[(long long)blockIdx.x * C + tid] = dbeta_s[tid];
  if (tid < 32) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(*tmem_slot), "n"(512));
  }
}

template <bool FAST, int IO>
int launch_tc_bwd3(const void* x, const float* gamma, const float* beta, const void* dy, void* dx, float* part_g,
                   float* part_b, int* n_parts, long long n_pix, TcFlags f, cudaStream_t s) {
  constexpr int C = 128;
  using L = BwdFusedSmem;
  CUtensorMap x_map, g_map, dx_map;
  TFCB_TRY(make_box_map<IO>(&x_map, x, n_pix, C));
  TFCB_TRY(make_box_map<IO>(&g_map, dy, n_pix, C));
  TFCB_TRY(make_box_map<IO>(&dx_map, dx, n_pix, C));
  __nv_bfloat16* planes = nullptr;
  TFCB_TRY(dev_alloc((void**)&planes, (size_t)4 * C * C * sizeof(__nv_bfloat16), s));
  gdn_tc_prep2_kernel<true><<<((C / 8) * C + 255) / 256, 256, 0, s>>>(gamma, C, planes);
  TFCB_LAUNCHED();
  cudaError_t e = cudaFuncSetAttribute(gdn_tc_bwd3_kernel<FAST, IO>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kBytes);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    dev_free(planes, s);
    return fail(TFCB_CUDA_ERROR, "cannot reserve %d bytes of shared memory: %s", L::kBytes, cudaGetErrorString(e));
  }
  const long long n_tiles = (n_pix + kTileM - 1) / kTileM;
  const int grid = (int)std::min<long long>(n_tiles, std::min(device_sm_count(), kGdnPartSlots));
  gdn_tc_bwd3_kernel<FAST, IO><<<grid, kB3Threads, L::kBytes, s>>>(x_map, g_map, dx_map, x, dy, planes, beta, part_g,
                                                                  part_b, n_pix, f);
  TFCB_LAUNCHED();
  e = cudaGetLastError();
  dev_free(planes, s);
  if (e != cudaSuccess) return fail(TFCB_CUDA_ERROR, "GDN tensor-core backward launch failed: %s", cudaGetErrorString(e));
  *n_parts = grid;
  return TFCB_OK;
}

// =============================================================================================
// Backward, C = 192, first of the two kernels (dx and q), box-fed like gdn_tc_bwd3_kernel.
//
// n, dp and a dgamma accumulator need 3 x 192 TMEM columns and whole-tile p and q planes 198 KB of shared memory, so
// C = 192 keeps the two-kernel split: this kernel produces dx and q = dL/dn, and gdn_tc_bwd_dgamma2_kernel contracts
// x and q into dgamma / dbeta.  q travels through the workspace AS THE bf16 hi / lo OPERAND PLANES the second kernel
// needs ([tile][hi, lo][24 groups][128 rows][8], 4 B/element like fp32): this kernel's q chunk buffers are bulk-stored
// as they are, the second kernel bulk-loads a tile's planes with one copy and converts nothing.  Per 128-pixel tile:
//
//   conv(t)   x boxes -> p = pool(x) hi / lo planes, one 32-channel K chunk at a time (two chunk buffers) -> MMA1  n += p_c . gamma_c
//   pass2(t)  x (L2 hit), g boxes + n from TMEM -> q hi / lo planes of the chunk (also bulk-stored to the workspace)
//                                                                                                      -> MMA2  dp += q_c . gammaT_c
//             the direct term g / m (IGDN: g * m) goes back into n's columns; FAST: with sign(x) in the two low
//             mantissa bits
//   pass3(t)  dx = direct + dpool/du * dp, from TMEM (the variants read x again, plain loads that hit L2)
//             -> output box -> TMA store
//
// gamma's hi plane is resident (72 KB; MMA2 reads it through the MN-major view); the lo planes of gamma (MMA1) and
// gamma^T (MMA2) arrive as 12 KB K chunks, double buffered, from a "gamma" warp, and each chunk's two hi products are
// issued before the one that needs the streamed chunk.  Chunk m of the stream uses operand buffer and gamma buffer
// m % 2, so ONE commit per chunk frees both (a q chunk's buffer additionally waits for its bulk store to have read
// it).  A ring of six 16 KB boxes serves every box request in program order.
// TMEM: n | dp (2 x 192 columns).
// =============================================================================================
constexpr int kD2Compute = 512;
constexpr int kD2Threads = kD2Compute + 128;   // + MMA-issue, box-copy, gamma and store warps
constexpr int kD2Sync = kD2Compute + 32;
constexpr int kD2Slots = 6;
constexpr int kDKg = kTileM * 16;  // dense group stride of the operand planes (row-per-lane stores need no padding)

struct BwdDx2Smem {
  static constexpr int C = 192;
  static constexpr int kGChunk = 4 * C * 16;                      // one 32-channel K chunk of one gamma plane (12 KB)
  static constexpr int kOpPlane = 4 * kDKg;                       // hi or lo plane of one 32-channel operand chunk (8 KB)
  static constexpr int kOffRing = 0;                              // [7] boxes (1024-byte aligned: swizzle atom)
  static constexpr int kOffGh = kOffRing + kD2Slots * kF4Box;     // gamma hi plane [j / 8][i][8], resident
  static constexpr int kOffG = kOffGh + C * C * 2;                // [2 buffers] lo K chunks of gamma / gamma^T
  static constexpr int kOffOp = kOffG + 2 * kGChunk;              // [2 buffers][hi, lo] operand (p or q) chunks
  static constexpr int kOffBeta = kOffOp + 4 * kOpPlane;
  static constexpr int kOffBar = kOffBeta + C * 4;
  // mbarriers: full[7], empty[7], yready[7], gfull[2], cfree[2], nfull, dpfull, qready[2], sfree[2]; then the TMEM slot
  static constexpr int kBarFull = 0, kBarEmpty = 7, kBarY = 14, kBarGfull = 21, kBarCfree = 23, kBarN = 25, kBarDp = 26,
                       kBarQready = 27, kBarSfree = 29, kNumBars = 31;
  static constexpr int kBytes = kOffBar + kNumBars * 8 + 16;
  static_assert(kOffGh % 128 == 0 && kOffG % 128 == 0 && kOffOp % 16 == 0 && kOffBar % 8 == 0, "alignment");
  static_assert(kBytes <= 232448, "shared memory budget");
};

template <bool FAST, int IO>
__global__ void __launch_bounds__(kD2Threads, 1)
gdn_tc_bwd_dx2_kernel(const __grid_constant__ CUtensorMap x_map, const __grid_constant__ CUtensorMap g_map,
                      const __grid_constant__ CUtensorMap dx_map, const void* __restrict__ x_,
                      const void* __restrict__ dy_, const __nv_bfloat16* __restrict__ planes,
                      const float* __restrict__ beta, uint8_t* __restrict__ q_planes, long long n_pix, TcFlags f) {
  using L = BwdDx2Smem;
  constexpr int C = L::C, NCH = C / 32;
  constexpr int EB = IoBytes<IO>::value, kRowB = C * EB;  // bytes per element / per pixel row of x / dy / dx
  const uint8_t* x = static_cast<const uint8_t*>(x_);
  const uint8_t* dy = static_cast<const uint8_t*>(dy_);
  extern __shared__ __align__(1024) uint8_t smem[];
  float* beta_s = reinterpret_cast<float*>(smem + L::kOffBeta);
  uint64_t* mbars = reinterpret_cast<uint64_t*>(smem + L::kOffBar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + L::kOffBar + L::kNumBars * 8);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int r = tid & 127, h = (tid >> 7) & 3, gwarp = warp & 3;  // compute thread (r, h): pixel row r, channel octet h of a box
  auto bar = [&](int i) { return smem_u32(mbars + i); };
  for (int i = tid; i < C; i += kD2Threads) beta_s[i] = beta[i];
  {
    const uint4* src = reinterpret_cast<const uint4*>(planes);  // first plane: gamma hi, [j / 8][i][8]
    uint4* dst = reinterpret_cast<uint4*>(smem + L::kOffGh);
    for (int i = tid; i < C * C * 2 / 16; i += kD2Threads) dst[i] = src[i];
  }
  if (tid == 0) {
    for (int i = 0; i < L::kNumBars; ++i) {
      // y ready / q ready: one arrival per compute warp
      const int count = ((i >= L::kBarY && i < L::kBarGfull) || (i >= L::kBarQready && i < L::kBarSfree)) ? kD2Compute / 32 : 1;
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar(i)), "r"(count));
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_n = *tmem_slot, tmem_dp = tmem_n + C;
  const uint32_t lane_sel = (uint32_t)(gwarp * 32) << 16;
  const long long n_tiles = (n_pix + kTileM - 1) / kTileM;
  const long long first = blockIdx.x;
  // Box request n uses ring slot n % 7 in its (n / 7)-th round:
  //   6 x boxes (conversion of the CTA's first tile), then per tile {x, g} x 6 (pass 2), dx-out x 6 (pass 3),
  //   (x of the next tile) x 6.
  // Chunk m of the operand / gamma stream uses buffers m % 2: 6 conversion chunks of the first tile, then per tile 6 q
  // chunks, 6 conversion chunks of the next tile.
  constexpr int W0 = kD2Compute / 32;  // first auxiliary warp
  auto slot_of = [](uint32_t n) { return n % (uint32_t)kD2Slots; };
  auto round_of = [](uint32_t n) { return n / (uint32_t)kD2Slots; };

  if (warp == W0 + 1) {
    // ---------------------------------- box-copy warp ----------------------------------
    if (lane == 0) {
      uint32_t n = 0;
      auto acquire = [&]() {
        const uint32_t slot = slot_of(n), round = round_of(n);
        if (round > 0) {
          if (!mbar_wait(bar(L::kBarEmpty + slot), (round - 1u) & 1u)) __trap();
        }
        return slot;
      };
      auto load = [&](const CUtensorMap* map, int c, int row0) {
        const uint32_t slot = acquire();
        const uint32_t full = bar(L::kBarFull + slot);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full), "n"(Box<IO>::kBytes) : "memory");
        asm volatile(
            "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;" ::"r"(
                smem_u32(smem + L::kOffRing + slot * kF4Box)),
            "l"(map), "r"(c * 32), "r"(row0), "r"(full), "l"(kEvictFirst)
            : "memory");
        ++n;
      };
      auto reserve = [&]() {  // output box: nothing to load, the slot only has to be free
        const uint32_t slot = acquire();
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar(L::kBarFull + slot)) : "memory");
        ++n;
      };
      auto prefetch_tile = [&](const uint8_t* base, long long tile) {  // one contiguous block -> L2
        const long long p0 = tile * kTileM;
        const long long rows = min((long long)kTileM, n_pix - p0);
        if (rows > 0)
          asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;" ::"l"(base + p0 * kRowB),
                       "r"((uint32_t)(rows * kRowB)), "l"(kEvictLast)
                       : "memory");
      };
      if (first < n_tiles) {
        prefetch_tile(x, first);
        prefetch_tile(dy, first);
#pragma unroll 1
        for (int c = 0; c < NCH; ++c) load(&x_map, c, (int)(first * kTileM));
      }
      for (long long tile = first; tile < n_tiles; tile += gridDim.x) {
        const long long next = tile + gridDim.x;
        const bool has_next = next < n_tiles;
        const int row0 = (int)(tile * kTileM);
        if (has_next) {  // the next tile of this CTA -> L2: its boxes become L2 hits
          prefetch_tile(x, next);
          prefetch_tile(dy, next);
        }
#pragma unroll 1
        for (int c = 0; c < NCH; ++c) {
          load(&x_map, c, row0);  // second read of x: an L2 hit
          load(&g_map, c, row0);
        }
#pragma unroll 1
        for (int c = 0; c < NCH; ++c) reserve();  // dx out
        if (has_next) {
#pragma unroll 1
          for (int c = 0; c < NCH; ++c) load(&x_map, c, (int)(next * kTileM));
        }
      }
    }
    __syncwarp();
  } else if (warp == W0 + 2) {
    // ---------------------------------- gamma warp: K chunks of gamma / gamma^T ----------------------------------
    if (lane == 0) {
      const uint8_t* gp = reinterpret_cast<const uint8_t*>(planes);
      constexpr size_t kPlaneBytes = (size_t)C * C * 2;
      uint32_t m = 0;
      auto chunk = [&](int transposed, int c) {
        const uint32_t buf = m & 1u;
        if (m >= 2) {  // the MMAs of chunk m - 2 (same buffers) have completed
          if (!mbar_wait(bar(L::kBarCfree + buf), ((m >> 1) - 1u) & 1u)) __trap();
        }
        const uint32_t gfull = bar(L::kBarGfull + buf);
        const uint32_t dst = smem_u32(smem + L::kOffG + buf * L::kGChunk);
        const uint8_t* src = gp + (size_t)(2 * transposed + 1) * kPlaneBytes + (size_t)c * L::kGChunk;  // the lo plane
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(gfull), "n"(L::kGChunk) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst),
                     "l"(src), "n"(L::kGChunk), "r"(gfull), "l"(kEvictLast)
                     : "memory");
        ++m;
      };
      if (first < n_tiles) {
#pragma unroll 1
        for (int c = 0; c < NCH; ++c) chunk(0, c);
      }
      for (long long tile = first; tile < n_tiles; tile += gridDim.x) {
#pragma unroll 1
        for (int c = 0; c < NCH; ++c) chunk(1, c);
        if (tile + gridDim.x < n_tiles) {
#pragma unroll 1
          for (int c = 0; c < NCH; ++c) chunk(0, c);
        }
      }
    }
    __syncwarp();
  } else if (warp == W0 + 3) {
    // ---------------------------------- store warp: q planes and dx boxes ----------------------------------
    if (lane == 0) {
      uint32_t n = (first < n_tiles) ? (uint32_t)NCH : 0u;
      uint32_t m = (first < n_tiles) ? (uint32_t)NCH : 0u;  // operand chunk counter (q chunks are stored, p chunks skipped)
      uint32_t ypar = 0u;  // per-slot phase of the y-ready barrier (a slot is an output box only now and then)
      uint32_t qcnt[2] = {0u, 0u};
      for (long long tile = first; tile < n_tiles; tile += gridDim.x) {
        const bool has_next = tile + gridDim.x < n_tiles;
        const int row0 = (int)(tile * kTileM);
        uint8_t* qt = q_planes + (size_t)tile * (2 * (C / 8) * kDKg);  // this tile's [hi, lo][24][128][8] planes
#pragma unroll 1
        for (int c = 0; c < NCH; ++c, ++m) {
          const uint32_t buf = m & 1u;
          if (!mbar_wait(bar(L::kBarQready + buf), qcnt[buf] & 1u)) __trap();
          ++qcnt[buf];
          const uint32_t src = smem_u32(smem + L::kOffOp + buf * 2 * L::kOpPlane);
#pragma unroll
          for (int pl = 0; pl < 2; ++pl)
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(
                             qt + (size_t)pl * ((C / 8) * kDKg) + (size_t)c * L::kOpPlane),
                         "r"(src + pl * L::kOpPlane), "n"(L::kOpPlane), "l"(kEvictLast)
                         : "memory");
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // the buffer has been read
          asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar(L::kBarSfree + buf)) : "memory");
        }
        n += 2 * NCH;  // x and g boxes of pass 2
#pragma unroll 1
        for (int c = 0; c < NCH; ++c, ++n) {
          const uint32_t slot = slot_of(n);
          if (!mbar_wait(bar(L::kBarY + slot), (ypar >> slot) & 1u)) __trap();
          ypar ^= 1u << slot;
          asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%1, %2}], [%3], %4;" ::"l"(&dx_map),
                       "r"(c * 32), "r"(row0), "r"(smem_u32(smem + L::kOffRing + slot * kF4Box)), "l"(kEvictFirst)
                       : "memory");
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // the box has been read: the slot is free
          asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar(L::kBarEmpty + slot)) : "memory");
        }
        if (has_next) {
          n += NCH;
          m += NCH;
        }
      }
      asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
    __syncwarp();
  } else if (warp == W0) {
    // ------------------------------- MMA-issue warp: MMA1, MMA2 (K-chunked, everything streamed) -------------------
    constexpr uint32_t kIdesc = umma_idesc(kTileM, C);  // A, B both K-major
    uint32_t n = 0, m = 0;
    constexpr uint32_t kIdescT = umma_idesc(kTileM, C) | (1u << 16);  // B = resident gamma hi read transposed (MMA2)
    const uint32_t gh = smem_u32(smem + L::kOffGh);
    // Six MMAs of chunk m (K chunk c of the tile): the four that only need the resident hi plane first, then the two
    // against the streamed lo chunk.  MMA1: B = gamma[j in chunk, :] (K-major); MMA2: B = gamma[:, i in chunk]^T, the
    // same plane through the MN-major view (hi) / the gamma^T lo chunk (K-major).
    auto chunk_mmas = [&](uint32_t acc, int c, bool transposed) {
      const uint32_t buf = m & 1u;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t a_hi = smem_u32(smem + L::kOffOp + buf * 2 * L::kOpPlane), a_lo = a_hi + L::kOpPlane;
      const uint32_t g_lo = smem_u32(smem + L::kOffG + buf * L::kGChunk);
#pragma unroll
      for (int s2 = 0; s2 < 2; ++s2) {
        const uint64_t dah = umma_desc(a_hi + (uint32_t)(2 * s2) * kDKg, kDKg, 128);
        const uint64_t dal = umma_desc(a_lo + (uint32_t)(2 * s2) * kDKg, kDKg, 128);
        const uint64_t dbh = transposed ? umma_desc(gh + (uint32_t)(c * 32 + s2 * 16) * 16u, 128, C * 16)
                                        : umma_desc(gh + (uint32_t)(c * 4 + 2 * s2) * (C * 16), C * 16, 128);
        const uint32_t idesc = transposed ? kIdescT : kIdesc;
        umma_bf16(acc, dah, dbh, idesc, (c == 0 && s2 == 0) ? 0u : 1u);
        umma_bf16(acc, dal, dbh, idesc, 1u);
      }
      if (!mbar_wait(bar(L::kBarGfull + buf), (m >> 1) & 1u)) __trap();
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
      for (int s2 = 0; s2 < 2; ++s2) {
        const uint64_t dah = umma_desc(a_hi + (uint32_t)(2 * s2) * kDKg, kDKg, 128);
        const uint64_t dbl = umma_desc(g_lo + (uint32_t)(2 * s2) * (C * 16), C * 16, 128);
        umma_bf16(acc, dah, dbl, kIdesc, 1u);
      }
      umma_commit(bar(L::kBarCfree + buf));
      ++m;
    };
    auto release = [&](uint32_t req) {
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar(L::kBarEmpty + slot_of(req))) : "memory");
    };
    auto mma1_tile = [&]() {
#pragma unroll 1
      for (int c = 0; c < NCH; ++c, ++n) {
        asm volatile("bar.sync %0, %1;" ::"r"(2 + (int)(m & 1u)), "n"(kD2Sync) : "memory");  // p planes of this chunk are written
        if (lane == 0) {
          release(n);
          chunk_mmas(tmem_n, c, false);
          if (c == NCH - 1) umma_commit(bar(L::kBarN));
        } else {
          ++m;
        }
        m = __shfl_sync(0xFFFFFFFFu, m, 0);
      }
    };
    if (first < n_tiles) mma1_tile();
    for (long long tile = first; tile < n_tiles; tile += gridDim.x) {
      const bool has_next = tile + gridDim.x < n_tiles;
#pragma unroll 1
      for (int c = 0; c < NCH; ++c, n += 2) {
        asm volatile("bar.sync %0, %1;" ::"r"(4 + (int)(m & 1u)), "n"(kD2Sync) : "memory");  // q planes of this chunk are written
        if (lane == 0) {
          release(n);      // x box
          release(n + 1);  // g box
          chunk_mmas(tmem_dp, c, true);
          if (c == NCH - 1) umma_commit(bar(L::kBarDp));  // dp is complete: the dx pass may start
        } else {
          ++m;
        }
        m = __shfl_sync(0xFFFFFFFFu, m, 0);
      }
      n += NCH;  // dx-out boxes
      if (has_next) mma1_tile();
    }
  } else if (warp < W0) {
  // --------------------------------- compute warps ---------------------------------
  uint32_t n = 0, m = 0;
  auto wait_full = [&](uint32_t req) {
    if (!mbar_wait(bar(L::kBarFull + slot_of(req)), round_of(req) & 1u)) __trap();
    return smem + L::kOffRing + slot_of(req) * kF4Box;
  };
  // this thread's 16-byte rows of the hi / lo planes of operand chunk m: waits until the MMAs of chunk m - 2 are done
  // and, if that chunk was a q chunk, until its bulk store has read the buffer
  uint32_t scnt[2] = {0u, 0u};
  auto operand_rows = [&](uint4** hi, uint4** lo, bool prev_was_q) {
    const uint32_t buf = m & 1u;
    if (m >= 2) {
      if (!mbar_wait(bar(L::kBarCfree + buf), ((m >> 1) - 1u) & 1u)) __trap();
    }
    if (prev_was_q) {
      if (!mbar_wait(bar(L::kBarSfree + buf), scnt[buf] & 1u)) __trap();
      ++scnt[buf];
    }
    uint8_t* base = smem + L::kOffOp + buf * 2 * L::kOpPlane + h * kDKg + r * 16;
    *hi = reinterpret_cast<uint4*>(base);
    *lo = reinterpret_cast<uint4*>(base + L::kOpPlane);
  };

  auto conv_tile = [&](bool after_pass2) {
#pragma unroll 1
    for (int c = 0; c < NCH; ++c, ++n) {
      uint8_t* box = wait_full(n);
      float v[8];
      box_load8<IO>(box, r, h, v);
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = tc_pool<FAST>(v[e], f);
      uint4 hi, lo, *ph, *pl;
      split8(v, &hi, &lo);
      operand_rows(&ph, &pl, after_pass2 && c < 2);  // chunks 0, 1 reuse the buffers of the tile's last two q chunks
      *ph = hi;
      *pl = lo;
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      asm volatile("bar.arrive %0, %1;" ::"r"(2 + (int)(m & 1u)), "n"(kD2Sync) : "memory");  // (also releases the box, see issue warp)
      ++m;
    }
  };

  if (first < n_tiles) conv_tile(false);
  int t = 0;
  for (long long tile = first; tile < n_tiles; tile += gridDim.x, ++t) {
    const bool has_next = tile + gridDim.x < n_tiles;
    if (!mbar_wait(bar(L::kBarN), (uint32_t)t & 1u)) __trap();  // MMA1 of this tile has completed
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    // ---- pass 2: q = dL/dn -> q planes; the direct term (FAST: and sign(x)) goes back into n's columns ----
#pragma unroll 1
    for (int c = 0; c < NCH; ++c, n += 2) {
      const uint32_t col = tmem_n + lane_sel + (uint32_t)(c * 32 + h * 8);
      uint32_t nacc[8];
      tmem_load<8>(col, nacc);
      uint8_t* bx = wait_full(n);
      uint8_t* bg = wait_full(n + 1);
      float xs[8], gs[8];
      box_load8<IO>(bx, r, h, xs);
      box_load8<IO>(bg, r, h, gs);
      const float4 bv0 = *reinterpret_cast<const float4*>(beta_s + c * 32 + h * 8);      // same address in every lane
      const float4 bv1 = *reinterpret_cast<const float4*>(beta_s + c * 32 + h * 8 + 4);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      const float bs[8] = {bv0.x, bv0.y, bv0.z, bv0.w, bv1.x, bv1.y, bv1.z, bv1.w};
      float q[8];
      uint32_t dbits[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float nn = bs[e] + __uint_as_float(nacc[e]);
        q[e] = tc_dl_dn<FAST>(gs[e], xs[e], nn, f);
        dbits[e] = __float_as_uint(tc_direct<FAST>(gs[e], nn, f));
        if (FAST) dbits[e] = (dbits[e] & ~3u) | ((xs[e] > 0.f) ? 1u : ((xs[e] < 0.f) ? 2u : 0u));
      }
      uint4 hi, lo, *qh, *ql;
      split8(q, &hi, &lo);
      operand_rows(&qh, &ql, c >= 2);
      *qh = hi;
      *ql = lo;
      tmem_store8(col, dbits);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // q planes -> MMA and -> bulk store
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      asm volatile("bar.arrive %0, %1;" ::"r"(4 + (int)(m & 1u)), "n"(kD2Sync) : "memory");  // (also releases the x and g boxes)
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar(L::kBarQready + (m & 1u))) : "memory");
      ++m;
    }
    // ---- pass 3: dx = direct + dpool/du * dp (FAST: from TMEM only) ----
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");  // this thread's direct terms are in TMEM
    if (!mbar_wait(bar(L::kBarDp), (uint32_t)t & 1u)) __trap();  // every MMA2 of this tile has completed
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
    for (int c = 0; c < NCH; ++c, ++n) {
      uint32_t d[8], p[8];
      tmem_load<8>(tmem_n + lane_sel + (uint32_t)(c * 32 + h * 8), d);
      tmem_load<8>(tmem_dp + lane_sel + (uint32_t)(c * 32 + h * 8), p);
      float xs[8];  // the variants: this thread's 8 values of x, read again (TMEM has no room to park them)
      if (!FAST) {
        const long long row = tile * kTileM + r;
        const uint8_t* src = x + row * kRowB + (c * 32 + h * 8) * EB;
        if (IO == 0) {
          const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
          const float4 x0 = row < n_pix ? __ldg(reinterpret_cast<const float4*>(src)) : z;
          const float4 x1 = row < n_pix ? __ldg(reinterpret_cast<const float4*>(src) + 1) : z;
          xs[0] = x0.x; xs[1] = x0.y; xs[2] = x0.z; xs[3] = x0.w;
          xs[4] = x1.x; xs[5] = x1.y; xs[6] = x1.z; xs[7] = x1.w;
        } else if (row < n_pix) {
          io_load8<IO>(src, xs);  // one 16-byte load, widened exactly
        } else {
#pragma unroll
          for (int e = 0; e < 8; ++e) xs[e] = 0.f;
        }
      }
      uint8_t* box = wait_full(n);  // the slot's previous user has left
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      float o[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        if (FAST) {
          const uint32_t code = d[e] & 3u;
          const float s = (code == 1u) ? 1.f : ((code == 2u) ? -1.f : 0.f);
          o[e] = fmaf(s, __uint_as_float(p[e]), __uint_as_float(d[e]));
        } else {
          o[e] = tc_dx(__uint_as_float(d[e]), xs[e], __uint_as_float(p[e]), f);
        }
      }
      box_store8<IO>(box, r, h, o);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // dx box -> TMA store
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar(L::kBarY + slot_of(n))) : "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");  // TMEM reads precede the next tile's MMAs
    if (has_next) conv_tile(true);
  }
  }  // compute warps
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (tid < 32) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(*tmem_slot), "n"(512));
  }
}

// =============================================================================================
// Backward, C = 192, second kernel: dgamma += p^T q, dbeta += column sums of q, box-fed.
//
// Per 128-pixel tile: the tile's q hi / lo planes arrive from the workspace with ONE bulk copy (96 KB, written in
// exactly this layout by gdn_tc_bwd_dx2_kernel); the x tile (six TMA boxes, 96 KB) lands IN THE MEMORY OF THE p PLANES
// (same size), every compute thread (r, h) takes its 48 values into registers, and after a barrier the p = pool(x) hi / lo
// planes are written over the boxes; 48 MMAs (two overlapping M = 128 row blocks [0,128) and [64,192) of p^T, N = 192,
// K = 128 pixels) accumulate into TMEM.  Nothing is double buffered (4 x 48 KB of planes): a tile costs one load
// latency + the conversion + the MMAs.  dbeta comes from the planes (q = hi + lo to 2^-17): warp w sums 8-channel
// groups w and w + 16, lane = pixel row mod 32.  The accumulator is flushed every kDgFlush tiles (CTAs take turns),
// transposed through the dead p planes one row block at a time into coalesced L2 adds.
// =============================================================================================
constexpr int kG2Compute = 512;
constexpr int kG2Threads = kG2Compute + 64;   // + MMA-issue and copy warps
constexpr int kG2Sync = kG2Compute + 32;

struct BwdDg2Smem {
  static constexpr int C = 192;
  static constexpr int kPlane = (C / 8) * kDKg;          // 49 152: one whole-K plane, dense groups
  static constexpr int kOffPh = 0;                       // p hi, lo: also the landing area of the six x boxes
  static constexpr int kOffPl = kOffPh + kPlane;
  static constexpr int kOffQh = kOffPl + kPlane;         // q hi, lo contiguous: one bulk copy per tile
  static constexpr int kOffQl = kOffQh + kPlane;
  static constexpr int kOffDbeta = kOffQl + kPlane;
  static constexpr int kOffBar = kOffDbeta + C * 4;
  // mbarriers: xfull, pfree, qfull, qdone, m3done; then the TMEM slot
  static constexpr int kBarXfull = 0, kBarPfree = 1, kBarQfull = 2, kBarQdone = 3, kBarM3 = 4, kNumBars = 5;
  static constexpr int kBytes = kOffBar + kNumBars * 8 + 16;
  static_assert(kBytes <= 232448, "shared memory budget");
  static_assert(2 * kPlane == 6 * kF4Box && 2 * kPlane >= kTileM * C * 4, "x tile / flush staging fit in the p planes");
};

template <bool FAST, int IO>
__global__ void __launch_bounds__(kG2Threads, 1)
gdn_tc_bwd_dgamma2_kernel(const __grid_constant__ CUtensorMap x_map, const void* __restrict__ x_,
                          const uint8_t* __restrict__ q_planes, float* __restrict__ part_g, float* __restrict__ part_b,
                          long long n_pix, TcFlags f) {
  using L = BwdDg2Smem;
  constexpr int C = L::C, NCH = C / 32;
  constexpr int kRowB = C * IoBytes<IO>::value;  // bytes per pixel row of x
  const uint8_t* x = static_cast<const uint8_t*>(x_);
  extern __shared__ __align__(1024) uint8_t smem[];
  float* dbeta_s = reinterpret_cast<float*>(smem + L::kOffDbeta);
  uint64_t* mbars = reinterpret_cast<uint64_t*>(smem + L::kOffBar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + L::kOffBar + L::kNumBars * 8);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int r = tid & 127, h = (tid >> 7) & 3, gwarp = warp & 3;
  auto bar = [&](int i) { return smem_u32(mbars + i); };
  for (int i = tid; i < C; i += kG2Threads) dbeta_s[i] = 0.f;
  if (tid == 0) {
    for (int i = 0; i < L::kNumBars; ++i) {
      const int count = (i == L::kBarQdone || i == L::kBarPfree) ? kG2Compute / 32 : 1;
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar(i)), "r"(count));
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_a = *tmem_slot, tmem_b = tmem_a + C;  // rows j in [0,128) | rows j in [64,192)
  const uint32_t lane_sel = (uint32_t)(gwarp * 32) << 16;
  const long long n_tiles = (n_pix + kTileM - 1) / kTileM;
  const long long first = blockIdx.x;
  const int fphase = (int)(blockIdx.x % kDgFlush);
  constexpr int W0 = kG2Compute / 32;

  if (warp == W0 + 1) {
    // ---------------------------------- copy warp: q planes and the x tile ----------------------------------
    if (lane == 0) {
      int t = 0;
      for (long long tile = first; tile < n_tiles; tile += gridDim.x, ++t) {
        const long long next = tile + gridDim.x;
        if (next < n_tiles) {  // the next tile of this CTA -> L2
          const long long p0 = next * kTileM;
          const long long rows = min((long long)kTileM, n_pix - p0);
          asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;" ::"l"(x + p0 * kRowB),
                       "r"((uint32_t)(rows * kRowB)), "l"(kEvictLast)
                       : "memory");
          asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;" ::"l"(q_planes + (size_t)next * (2 * L::kPlane)),
                       "n"(2 * L::kPlane), "l"(kEvictLast)
                       : "memory");
        }
        if (t > 0) {  // the q planes are free once the previous tile's MMAs and dbeta reads are done
          if (!mbar_wait(bar(L::kBarM3), (uint32_t)(t - 1) & 1u)) __trap();
          if (!mbar_wait(bar(L::kBarQdone), (uint32_t)(t - 1) & 1u)) __trap();
        }
        const uint32_t qfull = bar(L::kBarQfull);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(qfull), "n"(2 * L::kPlane) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                         smem_u32(smem + L::kOffQh)),
                     "l"(q_planes + (size_t)tile * (2 * L::kPlane)), "n"(2 * L::kPlane), "r"(qfull), "l"(kEvictFirst)
                     : "memory");
        // the p planes are free once the compute warps say so (previous MMAs done, flush staging consumed)
        if (!mbar_wait(bar(L::kBarPfree), (uint32_t)t & 1u)) __trap();
        const uint32_t xfull = bar(L::kBarXfull);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(xfull), "n"(NCH * Box<IO>::kBytes) : "memory");
        // ONE 3-D box: all six [128 x 32] boxes of the tile, back to back (a copy instruction costs the SM's copy
        // engine ~0.35 us whatever its size, tools/tma_probe.py)
        asm volatile(
            "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3, %4}], [%5], %6;" ::"r"(
                smem_u32(smem + L::kOffPh)),
            "l"(&x_map), "r"(0), "r"((int)(tile * kTileM)), "r"(0), "r"(xfull), "l"(kEvictFirst)
            : "memory");
      }
    }
    __syncwarp();
  } else if (warp == W0) {
    // ------------------------------- MMA-issue warp -------------------------------
    constexpr uint32_t kIdesc = umma_idesc(kTileM, C) | (1u << 15) | (1u << 16);  // A = p^T, B = q, both MN-major views
    const uint32_t p_hi = smem_u32(smem + L::kOffPh), p_lo = smem_u32(smem + L::kOffPl);
    const uint32_t q_hi = smem_u32(smem + L::kOffQh), q_lo = smem_u32(smem + L::kOffQl);
    int t = 0;
    for (long long tile = first; tile < n_tiles; tile += gridDim.x, ++t) {
      asm volatile("bar.sync 2, %0;" ::"n"(kG2Sync) : "memory");  // the p planes are written
      if (lane == 0) {
        if (!mbar_wait(bar(L::kBarQfull), (uint32_t)t & 1u)) __trap();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const bool restart = (t == 0) || (((t + fphase) % kDgFlush) == 0);
#pragma unroll 1
        for (int blk = 0; blk < 2; ++blk) {
          const uint32_t moff = (uint32_t)(blk * 8) * kDKg;  // second block starts at channel 64 = m group 8
          const uint32_t td = blk ? tmem_b : tmem_a;
#pragma unroll
          for (int s = 0; s < kTileM / 16; ++s) {
            const uint32_t koff = (uint32_t)(s * 16) * 16u;
            const uint64_t dah = umma_desc(p_hi + moff + koff, 128, kDKg);
            const uint64_t dal = umma_desc(p_lo + moff + koff, 128, kDKg);
            const uint64_t dbh = umma_desc(q_hi + koff, 128, kDKg);
            const uint64_t dbl = umma_desc(q_lo + koff, 128, kDKg);
            umma_bf16(td, dah, dbh, kIdesc, (restart && s == 0) ? 0u : 1u);
            umma_bf16(td, dal, dbh, kIdesc, 1u);
            umma_bf16(td, dah, dbl, kIdesc, 1u);
          }
        }
        umma_commit(bar(L::kBarM3));
      }
      __syncwarp();
    }
  } else if (warp < W0) {
  // --------------------------------- compute warps ---------------------------------
  float dbeta_acc[2][8];  // 8-channel groups warp and warp + 16, summed over rows lane, lane + 32, ...
#pragma unroll
  for (int k = 0; k < 2; ++k)
#pragma unroll
    for (int e = 0; e < 8; ++e) dbeta_acc[k][e] = 0.f;
  // float32 boxes (= box_chunk<0>; as a lambda the float32 instantiation compiles to the same code as before IO existed)
  auto chunk_at = [](uint8_t* box, int row, int j) { return reinterpret_cast<float4*>(box + row * 128 + ((j ^ (row & 7)) << 4)); };
  bool flushed = false;
  // one row block of the accumulator (lane r = row, 48 columns per thread) -> swizzled [128][192] fp32 staging in
  // the dead p planes -> 768 contiguous bytes per row added to the CTA's partial
  auto flush_dgamma = [&]() {
    uint8_t* stage = smem + L::kOffPh;
#pragma unroll 1
    for (int blk = 0; blk < 2; ++blk) {
#pragma unroll
      for (int cb = 0; cb < 3; ++cb) {
        uint32_t a[16];
        tmem_load<16>((blk ? tmem_b : tmem_a) + lane_sel + (uint32_t)(h * 48 + cb * 16), a);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int i = 0; i < 4; ++i)
          *reinterpret_cast<uint4*>(stage + r * 768 + (((h * 12 + cb * 4 + i) ^ (r & 7)) << 4)) =
              make_uint4(a[4 * i], a[4 * i + 1], a[4 * i + 2], a[4 * i + 3]);
      }
      asm volatile("bar.sync 1, %0;" ::"n"(kG2Compute) : "memory");
      float* pg = part_g + (long long)blockIdx.x * C * C + (long long)(blk * 64) * C;  // block b: lane r = channel 64 + r
#pragma unroll 1
      for (int it = 0; it < (kTileM * C / 4) / kG2Compute; ++it) {
        const int item = it * kG2Compute + tid, row = item / 48, u = item % 48;
        if (blk && row < 64) continue;  // rows [64,128) of block b repeat block a's
        const uint4 v = *reinterpret_cast<const uint4*>(stage + row * 768 + ((u ^ (row & 7)) << 4));
        float* dst = pg + row * C + u * 4;
        if (!flushed)
          asm volatile("st.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
        else
          asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
      }
      asm volatile("bar.sync 1, %0;" ::"n"(kG2Compute) : "memory");  // the staging is rewritten (next block / the x tile)
    }
    flushed = true;
  };

  int t = 0;
  for (long long tile = first; tile < n_tiles; tile += gridDim.x, ++t) {
    if (t > 0) {  // the previous tile's MMAs have completed: the p planes are dead, the accumulator is up to date
      if (!mbar_wait(bar(L::kBarM3), (uint32_t)(t - 1) & 1u)) __trap();
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (((t - 1 + fphase) % kDgFlush) == kDgFlush - 1) flush_dgamma();
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic accesses of the p planes precede the TMA writes
    __syncwarp();
    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar(L::kBarPfree)) : "memory");
    // the x tile has landed in the p planes: take this thread's 48 values, then overwrite the boxes with the planes
    if (!mbar_wait(bar(L::kBarXfull), (uint32_t)t & 1u)) __trap();
    // (the six boxes sit back to back: 96 KB of float32, or 48 KB of 16-bit elements in the hi plane's memory;
    // 16-bit values stay packed in registers until after the barrier)
    using XReg = typename std::conditional<IO == 0, float4, uint4>::type;
    XReg xa[NCH], xb[NCH];
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      uint8_t* box = smem + L::kOffPh + c * Box<IO>::kBytes;
      if constexpr (IO == 0) {
        xa[c] = *chunk_at(box, r, 2 * h);
        xb[c] = *chunk_at(box, r, 2 * h + 1);
      } else {
        xa[c] = *reinterpret_cast<const uint4*>(box_chunk<IO>(box, r, h));
      }
    }
    asm volatile("bar.sync 1, %0;" ::"n"(kG2Compute) : "memory");  // every thread holds its values
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      float v[8];
      if constexpr (IO == 0) {
        v[0] = xa[c].x; v[1] = xa[c].y; v[2] = xa[c].z; v[3] = xa[c].w;
        v[4] = xb[c].x; v[5] = xb[c].y; v[6] = xb[c].z; v[7] = xb[c].w;
      } else {
        io_widen8<IO>(xa[c], v);
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = tc_pool<FAST>(v[e], f);
      uint4 hi, lo;
      split8(v, &hi, &lo);
      *reinterpret_cast<uint4*>(smem + L::kOffPh + (4 * c + h) * kDKg + r * 16) = hi;
      *reinterpret_cast<uint4*>(smem + L::kOffPl + (4 * c + h) * kDKg + r * 16) = lo;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    asm volatile("bar.arrive 2, %0;" ::"n"(kG2Sync) : "memory");
    // dbeta from the q planes (q = hi + lo to 2^-17 relative): groups warp and warp + 16, rows lane + 32 k
    if (!mbar_wait(bar(L::kBarQfull), (uint32_t)t & 1u)) __trap();
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int grp = warp + 16 * k;
      if (grp < C / 8) {
#pragma unroll
        for (int rq = 0; rq < 4; ++rq) {
          const int row = lane + 32 * rq;
          const uint4 qh = *reinterpret_cast<const uint4*>(smem + L::kOffQh + grp * kDKg + row * 16);
          const uint4 ql = *reinterpret_cast<const uint4*>(smem + L::kOffQl + grp * kDKg + row * 16);
          const uint32_t wh[4] = {qh.x, qh.y, qh.z, qh.w}, wl[4] = {ql.x, ql.y, ql.z, ql.w};
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            dbeta_acc[k][2 * i] += __uint_as_float(wh[i] << 16) + __uint_as_float(wl[i] << 16);
            dbeta_acc[k][2 * i + 1] += __uint_as_float(wh[i] & 0xFFFF0000u) + __uint_as_float(wl[i] & 0xFFFF0000u);
          }
        }
      }
    }
    __syncwarp();
    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar(L::kBarQdone)) : "memory");
  }
  if (t > 0) {
    if (!mbar_wait(bar(L::kBarM3), (uint32_t)(t - 1) & 1u)) __trap();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    flush_dgamma();  // the tiles since the last restart (a turn that falls on the last tile is flushed here as well)
#pragma unroll
    for (int k = 0; k < 2; ++k)
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        float v = dbeta_acc[k][e];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
        const int grp = warp + 16 * k;
        if (lane == 0 && grp < C / 8) dbeta_s[grp * 8 + e] = v;  // one warp per group: no atomics
      }
  }
  }  // compute warps
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  for (int i = tid; i < C; i += kG2Threads) part_b[(long long)blockIdx.x * C + i] = dbeta_s[i];
  if (tid < 32) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(*tmem_slot), "n"(512));
  }
}

// q travels from the dx kernel to the dgamma kernel as bf16 hi / lo planes ([tile][2][24][128][8], 4 B/element; the
// workspace is sized in whole tiles, tfcb_gdn_backward_workspace_bytes)
template <bool FAST, int IO>
int launch_tc_bwd192(const void* x, const float* gamma, const float* beta, const void* dy, void* dx, float* q_ws,
                     float* part_g, float* part_b, int* n_parts, long long n_pix, TcFlags f, cudaStream_t s) {
  constexpr int C = 192;
  using L2 = BwdDx2Smem;
  using L3 = BwdDg2Smem;
  CUtensorMap x_map, g_map, dx_map, x_map3;  // x_map3: the whole [128 x 192] x tile as one 3-D box
  TFCB_TRY(make_box_map<IO>(&x_map, x, n_pix, C));
  TFCB_TRY(make_box_map<IO>(&g_map, dy, n_pix, C));
  TFCB_TRY(make_box_map<IO>(&dx_map, dx, n_pix, C));
  TFCB_TRY(make_tensor_map_3d(&x_map3, x, n_pix, C, kTileM, C / 32, IoMap<IO>::kType, IoMap<IO>::kSwizzle));
  if (cudaFuncSetAttribute(gdn_tc_bwd_dx2_kernel<FAST, IO>, cudaFuncAttributeMaxDynamicSharedMemorySize, L2::kBytes) != cudaSuccess ||
      cudaFuncSetAttribute(gdn_tc_bwd_dgamma2_kernel<FAST, IO>, cudaFuncAttributeMaxDynamicSharedMemorySize, L3::kBytes) != cudaSuccess) {
    (void)cudaGetLastError();
    return fail(TFCB_CUDA_ERROR, "cannot reserve shared memory for the C=192 backward");
  }
  __nv_bfloat16* planes = nullptr;
  TFCB_TRY(dev_alloc((void**)&planes, (size_t)4 * C * C * sizeof(__nv_bfloat16), s));
  gdn_tc_prep2_kernel<false><<<((C / 8) * C + 255) / 256, 256, 0, s>>>(gamma, C, planes);
  TFCB_LAUNCHED();
  const long long n_tiles = (n_pix + kTileM - 1) / kTileM;
  const int grid = (int)std::min<long long>(n_tiles, std::min(device_sm_count(), kGdnPartSlots));
  gdn_tc_bwd_dx2_kernel<FAST, IO><<<grid, kD2Threads, L2::kBytes, s>>>(x_map, g_map, dx_map, x, dy, planes, beta,
                                                                      reinterpret_cast<uint8_t*>(q_ws), n_pix, f);
  TFCB_LAUNCHED();
  gdn_tc_bwd_dgamma2_kernel<FAST, IO><<<grid, kG2Threads, L3::kBytes, s>>>(x_map3, x, reinterpret_cast<const uint8_t*>(q_ws),
                                                                           part_g, part_b, n_pix, f);
  TFCB_LAUNCHED();
  const cudaError_t e = cudaGetLastError();
  dev_free(planes, s);
  if (e != cudaSuccess) return fail(TFCB_CUDA_ERROR, "GDN tensor-core backward (C=192) launch failed: %s", cudaGetErrorString(e));
  *n_parts = grid;
  return TFCB_OK;
}

// Whether a tensor-core kernel takes a call, for either direction and every activation type io (0 float32, 1 float16,
// 2 bfloat16); if so, *f and *fast say which instantiation and with which flags.  The pointers are those the kernels
// move with 16-byte accesses: forward x, y (out) and beta; backward x, dy, dx (out) and, at C = 192, the q workspace.
// The forward ignores dy and ws, the backward beta (its kernels read beta element by element).
bool tc_rule(bool backward, int io, long long n_pix, int C, int flags, float alpha, float eps, const void* x,
             const void* beta, const void* dy, const void* out, const void* ws, TcFlags* f, bool* fast) {
  if ((io != 0 && io != 1 && io != 2) || (C != 128 && C != 192)) return false;
  if (!(alpha == 1.f || alpha == 2.f) || !(eps == 1.f || eps == 0.5f)) return false;  // fixed exponents only
  if (flags & (TFCB_GDN_POW_ALPHA | TFCB_GDN_POW_EPSILON)) return false;  // trainable exponents: literal pow
  const uintptr_t addr = backward ? (uintptr_t)x | (uintptr_t)dy | (uintptr_t)out | (C == 192 ? (uintptr_t)ws : 0)
                                  : (uintptr_t)x | (uintptr_t)out | (uintptr_t)beta;
  if (addr & 15) return false;
  // TMA boxes take 32-bit row coordinates; only the C = 128 forward moves x without them
  if ((backward || C == 192) && n_pix >= (1ll << 31)) return false;
  f->inverse = (flags & TFCB_GDN_INVERSE) ? 1 : 0;
  f->rectify = (flags & TFCB_GDN_RECTIFY) ? 1 : 0;
  f->alpha_mode = (alpha == 2.f) ? 2 : 1;
  f->eps_mode = (eps == 0.5f) ? 2 : 1;
  *fast = (alpha == 1.f) && (eps == 1.f) && !f->rectify;
  return true;
}

constexpr int tc_case(int C, bool fast, int io) { return (C == 192 ? 6 : 0) + (fast ? 3 : 0) + io; }

}  // namespace

// *handled = false: no tensor-core kernel takes this call (tc_rule).
int gdn_tc_forward(int io, const void* x, const float* gamma, const float* beta, void* y, long long n_pix, int C,
                   int flags, float alpha, float eps, cudaStream_t s, bool* handled) {
  TcFlags f;
  bool fast;
  *handled = tc_rule(false, io, n_pix, C, flags, alpha, eps, x, beta, nullptr, y, nullptr, &f, &fast);
  if (!*handled) return TFCB_OK;
  switch (tc_case(C, fast, io)) {
    case tc_case(128, false, 0): return launch_tc_fwd2<false, 0>(x, gamma, beta, y, n_pix, f, s);
    case tc_case(128, false, 1): return launch_tc_fwd2<false, 1>(x, gamma, beta, y, n_pix, f, s);
    case tc_case(128, false, 2): return launch_tc_fwd2<false, 2>(x, gamma, beta, y, n_pix, f, s);
    case tc_case(128, true, 0): return launch_tc_fwd2<true, 0>(x, gamma, beta, y, n_pix, f, s);
    case tc_case(128, true, 1): return launch_tc_fwd2<true, 1>(x, gamma, beta, y, n_pix, f, s);
    case tc_case(128, true, 2): return launch_tc_fwd2<true, 2>(x, gamma, beta, y, n_pix, f, s);
    case tc_case(192, false, 0): return launch_tc_fwd4<false, 0>(x, gamma, beta, y, n_pix, f, s);
    case tc_case(192, false, 1): return launch_tc_fwd4<false, 1>(x, gamma, beta, y, n_pix, f, s);
    case tc_case(192, false, 2): return launch_tc_fwd4<false, 2>(x, gamma, beta, y, n_pix, f, s);
    case tc_case(192, true, 0): return launch_tc_fwd4<true, 0>(x, gamma, beta, y, n_pix, f, s);
    case tc_case(192, true, 1): return launch_tc_fwd4<true, 1>(x, gamma, beta, y, n_pix, f, s);
    case tc_case(192, true, 2): return launch_tc_fwd4<true, 2>(x, gamma, beta, y, n_pix, f, s);
  }
  return fail(TFCB_INVALID_ARGUMENT, "GDN: no tensor-core forward for C=%d", C);  // not reached: tc_rule admits only the cases above
}

// Fills the per-CTA partial sums (part_g [n_parts][C][C], part_b [n_parts][C]) that the caller reduces.
// *handled = false: no tensor-core kernel takes this call (tc_rule).
int gdn_tc_backward(int io, const void* x, const float* gamma, const float* beta, const void* dy, void* dx, float* q_ws,
                    float* part_g, float* part_b, int* n_parts, long long n_pix, int C, int flags, float alpha, float eps,
                    cudaStream_t s, bool* handled) {
  TcFlags f;
  bool fast;
  *handled = tc_rule(true, io, n_pix, C, flags, alpha, eps, x, beta, dy, dx, q_ws, &f, &fast);
  if (!*handled) return TFCB_OK;
  switch (tc_case(C, fast, io)) {
    case tc_case(128, false, 0): return launch_tc_bwd3<false, 0>(x, gamma, beta, dy, dx, part_g, part_b, n_parts, n_pix, f, s);
    case tc_case(128, false, 1): return launch_tc_bwd3<false, 1>(x, gamma, beta, dy, dx, part_g, part_b, n_parts, n_pix, f, s);
    case tc_case(128, false, 2): return launch_tc_bwd3<false, 2>(x, gamma, beta, dy, dx, part_g, part_b, n_parts, n_pix, f, s);
    case tc_case(128, true, 0): return launch_tc_bwd3<true, 0>(x, gamma, beta, dy, dx, part_g, part_b, n_parts, n_pix, f, s);
    case tc_case(128, true, 1): return launch_tc_bwd3<true, 1>(x, gamma, beta, dy, dx, part_g, part_b, n_parts, n_pix, f, s);
    case tc_case(128, true, 2): return launch_tc_bwd3<true, 2>(x, gamma, beta, dy, dx, part_g, part_b, n_parts, n_pix, f, s);
    case tc_case(192, false, 0): return launch_tc_bwd192<false, 0>(x, gamma, beta, dy, dx, q_ws, part_g, part_b, n_parts, n_pix, f, s);
    case tc_case(192, false, 1): return launch_tc_bwd192<false, 1>(x, gamma, beta, dy, dx, q_ws, part_g, part_b, n_parts, n_pix, f, s);
    case tc_case(192, false, 2): return launch_tc_bwd192<false, 2>(x, gamma, beta, dy, dx, q_ws, part_g, part_b, n_parts, n_pix, f, s);
    case tc_case(192, true, 0): return launch_tc_bwd192<true, 0>(x, gamma, beta, dy, dx, q_ws, part_g, part_b, n_parts, n_pix, f, s);
    case tc_case(192, true, 1): return launch_tc_bwd192<true, 1>(x, gamma, beta, dy, dx, q_ws, part_g, part_b, n_parts, n_pix, f, s);
    case tc_case(192, true, 2): return launch_tc_bwd192<true, 2>(x, gamma, beta, dy, dx, q_ws, part_g, part_b, n_parts, n_pix, f, s);
  }
  return fail(TFCB_INVALID_ARGUMENT, "GDN: no tensor-core backward for C=%d", C);  // not reached: tc_rule admits only the cases above
}

}  // namespace tfcb

extern "C" int tfcb_gdn_native_16bit(int backward, const void* x_dev, const void* beta_dev, const void* dy_dev,
                                     int64_t n_pix, int C, int dtype, int flags, float alpha, float epsilon) {
  // the caller allocates y / dx and the workspace, so they are aligned
  tfcb::TcFlags f;
  bool fast;
  return n_pix > 0 && (dtype == 1 || dtype == 2) &&
         tfcb::tc_rule(backward != 0, dtype, n_pix, C, flags, alpha, epsilon, x_dev, beta_dev, dy_dev, nullptr, nullptr,
                       &f, &fast);
}
