// Fused shared-MLP chain on the 5th-generation tensor cores (tcgen05 + TMEM) for sm_100a.
//
// Replaces, for eval-mode inference, the reference's per-layer Conv{1,2}d -> BatchNorm -> ReLU kernels
// (nn_utils/conv.py:30-36,70-76; nn_utils/mlp.py:95-106) together with what surrounds them in
//   * PointNetSAModule.forward (pointnet2_utils/modules.py:208-244): group_points gather, centroid
//     subtraction, channel concat, 3 layers, max over the K neighbours;
//   * PointnetFPModule.forward (:498-507) and the four heads of PointNet2.forward
//     (models/PointNet2_tcls.py:126-148): plain chains, the last 1x1 conv with bias (+ sigmoid).
// BatchNorm (running statistics) is folded into the bf16 weights and an fp32 per-channel shift on the
// host, so a layer is  y = relu(W' x + b').
//
// One persistent CTA per SM walks 128-row tiles through the whole chain; nothing but the chain's input
// and output touches HBM.  The work is cut into 128-column blocks and pipelined at block granularity
// (csrc/chain_plan.cuh): the tensor pipe multiplies activation K-block k of layer l while the worker
// warps run the epilogue of the previous accumulator block and stage the next tile's input, so the
// MMA stream only stalls when a ring is genuinely empty.
//   act slots (smem, bf16, K-major core-matrix layout [C/8][128 rows][8])  -- A operand (B when transposed)
//   W ring    (smem, <= 16 KB chunks pre-tiled by the host in the same layout, one 1-D TMA copy each)
//   D blocks  (TMEM, fp32, 128 lanes x 128 columns, ring of 4)
// The last layer of a set-abstraction chain runs TRANSPOSED (A = weights, B = act), so TMEM lanes are
// output channels and the K neighbours of a centroid are adjacent columns: the max-pool is an
// in-register reduction inside the epilogue and only (centroid, channel) results reach HBM.
//
// Shared-memory operand layout (no swizzle, "interleaved" canonical K-major layout of UMMA):
//   element (row r, channel k) at byte  ((k/8) * ROWS + r) * 16 + (k%8)*2
//   -> core matrix = 8 rows x 16 B contiguous, SBO (8-row groups) = 128 B, LBO (K chunks) = ROWS*16 B.
#include <cuda_bf16.h>

#include <new>

#include "chain_plan.cuh"
#include "common.cuh"

namespace s4g {

// ------------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_n(uint64_t* bar, unsigned n) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(n) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, unsigned parity) {
  unsigned ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (-> cudaErrorLaunchFailure) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
  unsigned spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 22)) __trap();
  }
}
// non-blocking probe (try_wait may suspend the thread for a hardware-defined time when the phase is pending)
__device__ __forceinline__ bool mbar_test(uint64_t* bar, unsigned parity) {
  unsigned ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// one box of a 2-D tensor map (coordinates: c0 = innermost) into shared memory, completing `bar`'s transaction count
__device__ __forceinline__ void tma_load_2d(void* dst, const void* map, int c0, int c1, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
                   smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
// four rows (r0..r3, any order) of a 2-D tensor map with a {64, 1} box -> four consecutive 128-byte rows at dst
__device__ __forceinline__ void tma_gather4(void* dst, const void* map, int c0, int r0, int r1, int r2, int r3, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cta.global.tile::gather4.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::
          "r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(r0), "r"(r1), "r"(r2), "r"(r3) : "memory");
}
__device__ __forceinline__ void cp_async16(void* dst, const void* src, bool valid) {
  const unsigned n = valid ? 16u : 0u;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait(int pending) {
  switch (pending) {
    case 0: asm volatile("cp.async.wait_group 0;" ::: "memory"); break;
    case 1: asm volatile("cp.async.wait_group 1;" ::: "memory"); break;
    case 2: asm volatile("cp.async.wait_group 2;" ::: "memory"); break;
    case 3: asm volatile("cp.async.wait_group 3;" ::: "memory"); break;
    case 4: asm volatile("cp.async.wait_group 4;" ::: "memory"); break;
    case 5: asm volatile("cp.async.wait_group 5;" ::: "memory"); break;
    default: asm volatile("cp.async.wait_group 6;" ::: "memory"); break;
  }
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, unsigned cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, unsigned cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T ; both operands K-major bf16, fp32 accumulate
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc),
      "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// non-blocking TMEM loads of 32 / 16 accumulator columns (this warp's 32 lanes); pair with tmem_wait()
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
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
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// instruction descriptor: kind::f16, A = B = bf16, D = f32, both K-major, M x N
__device__ __forceinline__ uint32_t make_idesc(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// (a + bias) -> bf16x2, ReLU applied on the packed pair (max commutes with the monotonic rounding)
__device__ __forceinline__ uint32_t bias_act_pack(float a, float b, float ba, float bb, bool relu) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a + ba, b + bb);
  uint32_t r = *reinterpret_cast<uint32_t*>(&h);
  if (relu) asm("max.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(r), "r"(0u));  // packed zero is the zero register
  return r;
}

// 8 accumulator columns -> one 16-byte piece
__device__ __forceinline__ uint4 epi_piece(const float* v, const float* __restrict__ bias, bool relu) {
  const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias));
  const float4 b1 = __ldg(reinterpret_cast<const float4*>(bias) + 1);
  return make_uint4(bias_act_pack(v[0], v[1], b0.x, b0.y, relu), bias_act_pack(v[2], v[3], b0.z, b0.w, relu),
                    bias_act_pack(v[4], v[5], b1.x, b1.y, relu), bias_act_pack(v[6], v[7], b1.z, b1.w, relu));
}

// same with the shifts already in registers
__device__ __forceinline__ uint4 epi_piece_r(const float* v, const float4 b0, const float4 b1, bool relu) {
  return make_uint4(bias_act_pack(v[0], v[1], b0.x, b0.y, relu), bias_act_pack(v[2], v[3], b0.z, b0.w, relu),
                    bias_act_pack(v[4], v[5], b1.x, b1.y, relu), bias_act_pack(v[6], v[7], b1.z, b1.w, relu));
}

// shifts += a per-group term, NV / 4 16-byte pieces of bf16 (IN_GATHER_EDGE, layer 0); t == nullptr: no term
template <int NV>
__device__ __forceinline__ void add_term(float4* bv, const __nv_bfloat16* t) {
  if (t == nullptr) return;
#pragma unroll
  for (int g = 0; g < NV / 2; ++g) {
    const uint4 q = __ldg(reinterpret_cast<const uint4*>(t) + g);
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int h = 0; h < 2; ++h) {  // bf16 -> fp32 is a 16-bit shift
      float4& b = bv[2 * g + h];
      b.x += __uint_as_float(w[2 * h] << 16);
      b.y += __uint_as_float(w[2 * h] & 0xffff0000u);
      b.z += __uint_as_float(w[2 * h + 1] << 16);
      b.w += __uint_as_float(w[2 * h + 1] & 0xffff0000u);
    }
  }
}

template <bool PROF>
__device__ __forceinline__ long long tick() {
  if constexpr (PROF) return clock64();
  return 0;
}

struct Ring {  // position of a tile's first activation block in the slot ring
  int slot;
  unsigned use;
};
__device__ __forceinline__ void ring_advance(Ring& r, const ChainParams& p) {
  r.slot += p.n_act_mod;
  r.use += (unsigned)p.n_act_div;
  if (r.slot >= p.slots) { r.slot -= p.slots; ++r.use; }
}
__device__ __forceinline__ void ring_at(const Ring& base, const ChainParams& p, int blk_mod, int blk_div, int& slot,
                                        unsigned& use) {
  slot = base.slot + blk_mod;
  use = base.use + (unsigned)blk_div;
  if (slot >= p.slots) { slot -= p.slots; ++use; }
}

// ------------------------------------------------------------------------------------------------
// the kernel: warps 0..15 = epilogue, 16-17 = loaders, 18 = MMA issue, 19-20 = TMA weight producers.
// PROF = true adds the per-role cycle counters of s4g_chain_set_profile (clock reads cost the MMA warp ~150 cycles
// per job, so the product path is compiled without them).
// ------------------------------------------------------------------------------------------------
// XYZ_MLP: the IN_XYZ_MLP loader code lives in an instantiation of its own — the kernel is ~60 KB of SASS shared by
// five roles, and every extra block of rarely-run code costs the other chains instruction-cache misses.
// OUT (the chain's output mode) and GATHER (gathered vs row input) are compile-time for the same reason: a chain only
// carries the loader and the final epilogue it uses.
// TMA_IN (row input only): the input blocks are fetched by one thread with 2-D tensor copies (64 channels x 128 rows
// per box) into the 128-byte-swizzled K-major layout, instead of 64 threads x 16-byte cp.async into the interleaved one.
// EDGE (IN_GATHER_EDGE): layer 0's epilogue adds the per-group term p.term[row / K] to the shifts.  Compile-time, so the
// other chains carry none of its code.
template <bool PROF, bool XYZ_MLP, int OUT, bool GATHER, bool TMA_IN = false, bool EDGE = false>
__global__ void __launch_bounds__(kChainThreads, 1) mlp_chain_kernel(const __grid_constant__ ChainParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* slots = smem;
  uint8_t* ring = smem + (size_t)p.slots * kSlotBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(ring + (size_t)p.stages * kStageBytes);
  uint64_t* act_ready = bars;                      // [kMaxSlots]  block published (8 warp-arrivals)
  uint64_t* tm_full = act_ready + kMaxSlots;       // [4] accumulator complete
  uint64_t* tm_empty = tm_full + kAccBlocks;       // [4] accumulator drained by the epilogue warps
  uint64_t* w_full = tm_empty + kAccBlocks;        // [kMaxStages] weight chunk landed
  uint64_t* w_empty = w_full + kMaxStages;         // [kMaxStages] MMAs reading the chunk completed
  uint64_t* blk_free = w_empty + kMaxStages;       // [kMaxBlocks] last MMA reading tile-relative block b completed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(blk_free + kMaxBlocks);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);  // warp-uniform for the compiler
  const int lane = threadIdx.x & 31;
  const int tile_rows = kTileRows * p.subs;  // a tile = 1 or 2 row blocks of 128 rows (WorkerJob::sub)
  const int n_tiles = (p.P + tile_rows - 1) / tile_rows;
  const int n_my = ((int)blockIdx.x < n_tiles) ? (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;

  if (threadIdx.x == 0) {
    // one arrival per WARP (per-thread arrivals on one mbarrier serialise for hundreds of cycles).  Blocks and
    // accumulators count 16: the 16 epilogue warps of a cooperative job arrive once, the 8 warps of one
    // epilogue group with weight 2, the 2 loader warps with weight 8
    for (int s = 0; s < kMaxSlots; ++s) mbar_init(&act_ready[s], kEpiWarps);
    for (int s = 0; s < kAccBlocks; ++s) { mbar_init(&tm_full[s], 1); mbar_init(&tm_empty[s], kEpiWarps); }
    for (int s = 0; s < kMaxStages; ++s) { mbar_init(&w_full[s], 1); mbar_init(&w_empty[s], 1); }
    for (int s = 0; s < kMaxBlocks; ++s) mbar_init(&blk_free[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp) tmem_alloc(tmem_slot, 512u);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  if (warp >= kProducerWarp) {
    // ============ TMA producers: one weight chunk per MMA job, in job order; warp k takes chunks c % 2 == k ============
    const int pw = warp - kProducerWarp;
    unsigned cpar = 0;  // parity of the running chunk index
    int s = 0;
    unsigned use = 0;
    long long c_wait = 0;
    const long long t_begin = tick<PROF>();
    for (int it = 0; it < n_my; ++it) {
      const uint8_t* src = reinterpret_cast<const uint8_t*>(p.weights);
      for (int j = 0; j < p.n_mma; ++j) {
        const MmaJob job = p.mma[j];
        const unsigned bytes = (unsigned)job.n8 * (unsigned)job.k16 * 256u;  // rows * 16 k16 channels * 2 B
        if (kProducers == 1 || (int)cpar == pw) {
          const long long t0 = tick<PROF>();
          if (use > 0) mbar_wait(&w_empty[s], (use - 1) & 1);
          c_wait += tick<PROF>() - t0;
          if (elect_one()) {
            mbar_expect_tx(&w_full[s], bytes);
            bulk_g2s(ring + (size_t)s * kStageBytes, src, bytes, &w_full[s]);
          }
          __syncwarp();
        }
        cpar ^= 1u;
        src += bytes;
        if (++s == p.stages) { s = 0; ++use; }
      }
    }
    if (PROF && p.prof && lane == 0 && pw == 0) {
      p.prof[blockIdx.x * 16 + 0] = tick<PROF>() - t_begin;
      p.prof[blockIdx.x * 16 + 1] = c_wait;
    }
  } else if (warp == kMmaWarp) {
    // ===================== MMA warp (converged; one elected lane issues tcgen05.mma / commit) =====================
    // The issuing thread is the scarce resource (profiles/mma_loop.cu): everything a job needs — its table
    // entry, ring positions and the state of the (up to four) barriers it waits on — is fetched and probed
    // right after the PREVIOUS job's MMAs were issued, so those latencies overlap the tensor pipe.
    const uint32_t slots16 = smem_u32(slots) >> 4;
    const uint32_t ring16 = smem_u32(ring) >> 4;
    // descriptor high word: SBO = 128 B, version 1;  low word: (addr >> 4) | (LBO >> 4) << 16
    const uint64_t desc_hi = (uint64_t)((128u >> 4) | (1u << 14)) << 32;
    const uint32_t a_lbo16 = (uint32_t)kTileRows;  // (128 rows * 16 B) >> 4
    // swizzled input blocks: SBO = 1024 B (8 rows x 128 B), version 1, layout type 2 = SWIZZLE_128B; LBO unused
    const uint64_t swz_hi = (uint64_t)((1024u >> 4) | (1u << 14) | (2u << 29)) << 32;
    long long c_act = 0, c_tm = 0, c_w = 0;
    const long long t_begin = tick<PROF>();
    struct Next {
      MmaJob job;
      int slot, s;
      unsigned use, q, tb, wuse;
      bool ok_act, ok_tm, ok_w;
    };
    Ring base = {0, 0u};
    unsigned base_q = 0;
    int s = 0;
    unsigned wuse = 0;
    auto prepare = [&](int j) -> Next {
      Next x;
      x.job = p.mma[j];
      ring_at(base, p, x.job.blk_mod, x.job.blk_div, x.slot, x.use);
      x.q = base_q + x.job.acc;
      x.tb = x.q & (kAccBlocks - 1);
      x.s = s;
      x.wuse = wuse;
      x.ok_act = !(x.job.flags & MF_WAIT_ACT) || mbar_test(&act_ready[x.slot], x.use & 1);
      const bool need_tm = (x.job.flags & MF_FIRST_K) && x.q >= (unsigned)kAccBlocks;
      x.ok_tm = !need_tm || (mbar_test(&tm_empty[x.tb], ((x.q >> 2) - 1) & 1) &&
                             (!(x.job.flags & MF_PAIR) || mbar_test(&tm_empty[x.tb + 1], ((x.q >> 2) - 1) & 1)));
      x.ok_w = mbar_test(&w_full[s], wuse & 1);
      return x;
    };
    Next cur = {};
    if (n_my > 0) cur = prepare(0);
    for (int it = 0; it < n_my; ++it) {
      for (int j = 0; j < p.n_mma; ++j) {
        const MmaJob job = cur.job;
        const int slot = cur.slot;
        const unsigned q = cur.q, tb = cur.tb;
        const long long t0 = tick<PROF>();
        if (!cur.ok_act) mbar_wait(&act_ready[slot], cur.use & 1);
        const long long t1 = tick<PROF>();
        if (!cur.ok_tm) {
          mbar_wait(&tm_empty[tb], ((q >> 2) - 1) & 1);
          if (job.flags & MF_PAIR) mbar_wait(&tm_empty[tb + 1], ((q >> 2) - 1) & 1);
        }
        const long long t2 = tick<PROF>();
        if (!cur.ok_w) mbar_wait(&w_full[cur.s], cur.wuse & 1);
        const long long t3 = tick<PROF>();
        c_act += t1 - t0; c_tm += t2 - t1; c_w += t3 - t2;
        if (PROF && p.prof && blockIdx.x == 0 && it == 2 && lane == 0) {
          long long* tr = p.prof + 148 * 16 + j * 4;
          tr[0] = t0; tr[1] = t3;
        }
        tc_fence_after();
        // The MMA queue is shallow (an issue blocks until the previous MMA has started), so the thread-side
        // work for the NEXT job is done between this job's MMAs, while the tensor pipe is busy: all but the
        // last MMA, then fetch + probe the next job, then the last MMA and the commits.
        const uint32_t n = (uint32_t)job.n8 * 8u;
        const bool transposed = OUT == OUT_MAXPOOL && (job.flags & MF_TRANSPOSED) != 0;
        const uint32_t idesc = make_idesc(128, transposed ? kTileRows : (int)n);
        const bool swz = TMA_IN && (job.flags & MF_SWZ) != 0;
        // swizzled block: halves of 64 channels 16 KB apart, 16 channels = 32 B inside a 128-byte row
        const uint32_t a_lo = swz ? (slots16 + (uint32_t)slot * (kSlotBytes >> 4) + (uint32_t)(job.koff >> 2) * (16384u >> 4) +
                                     (uint32_t)(job.koff & 3) * 2u) | (1u << 16)
                                  : (slots16 + (uint32_t)slot * (kSlotBytes >> 4) + (uint32_t)job.koff * (2u * a_lbo16)) | (a_lbo16 << 16);
        const uint64_t a_hi = swz ? swz_hi : desc_hi;
        const uint32_t w_lo = (ring16 + (uint32_t)cur.s * (kStageBytes >> 4)) | (n << 16);  // LBO = n rows * 16 B
        // operand order is swapped BEFORE the loop: a predicated-off tcgen05.mma still costs an issue slot
        const uint32_t x0 = transposed ? w_lo : a_lo, y0 = transposed ? a_lo : w_lo;
        const uint32_t x_step = transposed ? 2u * n : (swz ? 2u : 2u * a_lbo16);  // next 16 channels = 2 K pieces
        const uint64_t x_hi = transposed ? desc_hi : a_hi;  // (a TMA_IN chain has no transposed layer)
        const uint32_t y_step = transposed ? 2u * a_lbo16 : 2u * n;
        const uint32_t d_addr = tmem_base + tb * 128u;
        const uint32_t acc0 = (job.flags & MF_FIRST_K) ? 0u : 1u;
        const int k_last = job.k16 - 1;
        if (elect_one()) {
          uint32_t x_lo = x0, y_lo = y0, acc = acc0;
#pragma unroll 1
          for (int k = 0; k < k_last; ++k) {
            umma_bf16(d_addr, x_hi | x_lo, desc_hi | y_lo, idesc, acc);
            acc = 1u;
            x_lo += x_step;
            y_lo += y_step;
          }
        }
        __syncwarp();
        // advance to the next job (possibly the first one of the CTA's next tile) and probe its barriers
        const int s_cur = cur.s;
        if (++s == p.stages) { s = 0; ++wuse; }
        int jn = j + 1;
        if (jn == p.n_mma) {
          jn = 0;
          ring_advance(base, p);
          base_q += (unsigned)p.n_acc;
        }
        if (jn != 0 || it + 1 < n_my) cur = prepare(jn);
        if (PROF && p.prof && blockIdx.x == 0 && it == 2 && lane == 0) p.prof[148 * 16 + j * 4 + 2] = tick<PROF>();
        if (elect_one()) {
          umma_bf16(d_addr, x_hi | (x0 + x_step * (uint32_t)k_last), desc_hi | (y0 + y_step * (uint32_t)k_last), idesc,
                    k_last > 0 ? 1u : acc0);
          umma_commit(&w_empty[s_cur]);                              // stage reusable once these MMAs have read it
          if (job.flags & MF_LAST_K) {                               // accumulator(s) complete
            umma_commit(&tm_full[tb]);
            if (job.flags & MF_PAIR) umma_commit(&tm_full[tb + 1]);
          }
          if (job.flags & MF_RELEASE) umma_commit(&blk_free[job.blk]);  // activation block dead
        }
        __syncwarp();
        if (PROF && p.prof && blockIdx.x == 0 && it == 2 && lane == 0) p.prof[148 * 16 + j * 4 + 3] = tick<PROF>();
      }
    }
    if (PROF && p.prof && lane == 0) {
      p.prof[blockIdx.x * 16 + 2] = tick<PROF>() - t_begin;
      p.prof[blockIdx.x * 16 + 3] = c_act;
      p.prof[blockIdx.x * 16 + 4] = c_tm;
      p.prof[blockIdx.x * 16 + 5] = c_w;
    }
  } else if (TMA_IN && GATHER && warp >= kLoadWarp0) {
    // ===================== gathered input by TMA: lane l of loader warp w fetches rows 4l..4l+3 of half w of a feature
    // block with ONE tile::gather4 copy (4 table rows -> 4 consecutive rows of the swizzled layout); the relative-xyz
    // block is computed by the 64 threads as in the cp.async path =====================
    const int lw = warp - kLoadWarp0;
    const int r = (int)threadIdx.x - kLoadWarp0 * 32;  // 0..63
    const int per_b = p.M * p.K;
    const int oob = (int)((long long)p.P / per_b) * p.N;  // first row past the feature table: zero-filled by the copy engine
    Ring base = {0, 0u};
    int jn[4] = {0, 0, 0, 0}, jn_next[4] = {0, 0, 0, 0};  // xyz block: rows r, r + 64 of each row block
    int4 g4[2], g4_next[2];                              // feature blocks: rows 4 lane .. 4 lane + 3 of each row block
    auto tile_base = [&](int jt) -> long long { return ((long long)blockIdx.x + (long long)jt * gridDim.x) * tile_rows; };
    auto load_idx = [&](int jt) {
#pragma unroll
      for (int sub = 0; sub < 2; ++sub) {
        const bool on = jt < n_my && sub < p.subs;
        const long long row4 = tile_base(jt) + sub * kTileRows + 4 * lane;
        g4_next[sub] = (on && row4 < p.P) ? __ldg(reinterpret_cast<const int4*>(p.nbr + row4)) : make_int4(-1, -1, -1, -1);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const long long row = tile_base(jt) + sub * kTileRows + r + 64 * h;
          jn_next[2 * sub + h] = (on && row < p.P) ? __ldg(p.nbr + row) : 0;
        }
      }
    };
    load_idx(0);
    for (int it = 0; it < n_my; ++it) {
#pragma unroll
      for (int q = 0; q < 4; ++q) jn[q] = jn_next[q];
      g4[0] = g4_next[0]; g4[1] = g4_next[1];
      load_idx(it + 1);
      for (int j = 0; j < p.n_ld; ++j) {
        const WorkerJob job = p.ld[j];
        int slot;
        unsigned use;
        ring_at(base, p, job.blk_mod, job.blk_div, slot, use);
        if (job.same || it >= (int)job.min_it) mbar_wait(&blk_free[job.pred], (unsigned)(job.same ? it : it - 1) & 1u);
        if (job.kind == WK_LOAD_XYZ) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const long long row = tile_base(it) + job.sub * kTileRows + r + 64 * h;
            float xa = 0.f, xb = 0.f, xc = 0.f;
            if (row < p.P) {
              const int b = (int)(row / per_b);
              const int m = (int)((row - (long long)b * per_b) / p.K);
              const float* X = p.xyz + (long long)b * 3 * p.N;
              const float* C = p.ctr + (long long)b * 3 * p.M;
              const int jq = job.sub ? jn[2 + h] : jn[h];
              xa = __fsub_rn(__ldg(X + jq), __ldg(C + m));
              xb = __fsub_rn(__ldg(X + p.N + jq), __ldg(C + p.M + m));
              xc = __fsub_rn(__ldg(X + 2 * p.N + jq), __ldg(C + 2 * p.M + m));
            }
            uint8_t* sbase = slots + (size_t)slot * kSlotBytes + (size_t)(r + 64 * h) * 16;
            __nv_bfloat162 h0 = __floats2bfloat162_rn(xa, xb), h1 = __floats2bfloat162_rn(xc, 0.f);
            *reinterpret_cast<uint4*>(sbase) =
                make_uint4(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1), 0u, 0u);
            *reinterpret_cast<uint4*>(sbase + kTileRows * 16) = make_uint4(0u, 0u, 0u, 0u);
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive_n(&act_ready[slot], kEpiWarps / kLoadWarps);
        } else {
          const bool mine = lw < ((int)job.c_count >> 6);  // warp w takes the 64-channel half w
          if (lane == 0) {
            if (mine) {
              mbar_expect_tx(&act_ready[slot], 64u * kTileRows * 2u);
              mbar_arrive_n(&act_ready[slot], kEpiWarps / kLoadWarps - 1);
            } else {
              mbar_arrive_n(&act_ready[slot], kEpiWarps / kLoadWarps);
            }
          }
          __syncwarp();
          if (mine) {
            const int4 q = job.sub ? g4[1] : g4[0];
            const long long row4 = tile_base(it) + job.sub * kTileRows + 4 * lane;
            const int t0 = (int)(row4 / per_b) * p.N;  // K % 4 == 0: the four rows belong to one cloud
            const bool valid = q.x >= 0;
            tma_gather4(slots + (size_t)slot * kSlotBytes + (size_t)lw * 16384 + (size_t)lane * 512, &p.in_map,
                        (int)job.c_begin + 64 * lw, valid ? t0 + q.x : oob, valid ? t0 + q.y : oob, valid ? t0 + q.z : oob,
                        valid ? t0 + q.w : oob, &act_ready[slot]);
          }
        }
      }
      ring_advance(base, p);
    }
  } else if (TMA_IN && !GATHER && warp >= kLoadWarp0) {
    // ===================== TMA input loader: one elected thread of loader warp 0 =====================
    if (warp == kLoadWarp0) {
      Ring base = {0, 0u};
      for (int it = 0; it < n_my; ++it) {
        const int row0 = ((int)blockIdx.x + it * (int)gridDim.x) * tile_rows;
        for (int j = 0; j < p.n_ld; ++j) {
          const WorkerJob job = p.ld[j];
          int slot;
          unsigned use;
          ring_at(base, p, job.blk_mod, job.blk_div, slot, use);
          if (job.same || it >= (int)job.min_it) mbar_wait(&blk_free[job.pred], (unsigned)(job.same ? it : it - 1) & 1u);
          if (elect_one()) {
            // rows past P are zero-filled by the copy engine and still count towards the transaction bytes
            mbar_expect_tx(&act_ready[slot], (unsigned)job.c_count * (kTileRows * 2u));
            uint8_t* dst = slots + (size_t)slot * kSlotBytes;
            for (int c = 0; c < (int)job.c_count; c += 64)
              tma_load_2d(dst + (size_t)(c >> 6) * 16384, &p.in_map, (int)job.c_begin + c, row0 + (int)job.sub * kTileRows,
                          &act_ready[slot]);
            mbar_arrive_n(&act_ready[slot], kEpiWarps - 1);
          }
          __syncwarp();
        }
        ring_advance(base, p);
      }
    }
  } else if (warp >= kLoadWarp0) {
    // ===================== loader warps: thread r stages rows r and r + 64 of every layer-0 input block =====================
    const int r = (int)threadIdx.x - kLoadWarp0 * 32;  // 0..63
    const int per_b = p.M * p.K;
    const int D = p.load_depth;
    Ring base = {0, 0u};
    // neighbour index of this thread's two rows of each row block, current / next tile (gather mode): [2 * sub + h]
    int jn[4] = {0, 0, 0, 0}, jn_next[4] = {0, 0, 0, 0};
    auto tile_row = [&](int jt, int h, int sub) -> long long {
      return ((long long)blockIdx.x + (long long)jt * gridDim.x) * tile_rows + sub * kTileRows + r + 64 * h;
    };
    auto load_nbr = [&](int jt, int h, int sub) -> int {
      if (jt >= n_my || sub >= p.subs) return 0;
      const long long row = tile_row(jt, h, sub);
      return row < p.P ? __ldg(p.nbr + row) : 0;
    };
    if constexpr (GATHER) {
#pragma unroll
      for (int q = 0; q < 4; ++q) jn_next[q] = load_nbr(0, q & 1, q >> 1);
    }
    // slots of the cp.async blocks issued and not yet published, oldest first (one commit group each)
    int pend0 = 0, pend1 = 0, pend2 = 0, npend = 0;
    auto publish_oldest = [&]() {
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive_n(&act_ready[pend0], kEpiWarps / kLoadWarps);
      pend0 = pend1; pend1 = pend2; --npend;
    };
    long long c_free = 0, c_cp = 0;
    const long long t_begin = tick<PROF>();
    for (int it = 0; it < n_my; ++it) {
      if constexpr (GATHER) {
#pragma unroll
        for (int q = 0; q < 4; ++q) { jn[q] = jn_next[q]; jn_next[q] = load_nbr(it + 1, q & 1, q >> 1); }
      }
      for (int j = 0; j < p.n_ld; ++j) {
        const WorkerJob job = p.ld[j];
        int slot;
        unsigned use;
        ring_at(base, p, job.blk_mod, job.blk_div, slot, use);
        if ((!GATHER || job.kind != WK_LOAD_XYZ) && npend == D) {  // pipeline full: the oldest block must land first
          const long long t0 = tick<PROF>();
          cp_async_wait(D - 1);
          c_cp += tick<PROF>() - t0;
          publish_oldest();
        }
        const long long tl0 = tick<PROF>();
        // slot free?  wait for the release of the block that last held it (chain_plan.cuh)
        uint64_t* fbar = &blk_free[job.pred];
        const bool need = job.same || it >= (int)job.min_it;
        const unsigned fpar = (unsigned)(job.same ? it : it - 1) & 1u;
        if (need && !__all_sync(0xffffffffu, mbar_try_wait(fbar, fpar))) {
          // never hold unpublished blocks while blocking on a slot: their consumers may be what frees it
          const long long t0 = tick<PROF>();
          if (npend) {
            cp_async_wait(0);
            while (npend) publish_oldest();
          }
          mbar_wait(fbar, fpar);
          c_free += tick<PROF>() - t0;
        }
        if (XYZ_MLP && job.kind == WK_LOAD_XYZ) {
          // the xyz layer on the CUDA cores: ReLU(W (x_j - c_m) + shift) in fp32 for this thread's two rows
          float dx[2], dy[2], dz[2];
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const long long row = tile_row(it, h, job.sub);
            dx[h] = dy[h] = dz[h] = 0.f;
            if (row < p.P) {
              const int b = (int)(row / per_b);
              const int m = (int)((row - (long long)b * per_b) / p.K);
              const float* X = p.xyz + (long long)b * 3 * p.N;
              const float* C = p.ctr + (long long)b * 3 * p.M;
              const int jq = job.sub ? jn[2 + h] : jn[h];
              dx[h] = __fsub_rn(__ldg(X + jq), __ldg(C + m));
              dy[h] = __fsub_rn(__ldg(X + p.N + jq), __ldg(C + p.M + m));
              dz[h] = __fsub_rn(__ldg(X + 2 * p.N + jq), __ldg(C + 2 * p.M + m));
            }
          }
          uint8_t* sb = slots + (size_t)slot * kSlotBytes + (size_t)r * 16;
          const bool relu = p.xyz_relu != 0;
          const int pieces = job.c_count >> 3;
#pragma unroll 2
          for (int g = 0; g < pieces; ++g) {
            float4 w[8];
#pragma unroll
            for (int e = 0; e < 8; ++e)  // constant bank, warp-uniform index
              w[e] = make_float4(p.xyz_w[(g * 8 + e) * 4], p.xyz_w[(g * 8 + e) * 4 + 1], p.xyz_w[(g * 8 + e) * 4 + 2],
                                 p.xyz_w[(g * 8 + e) * 4 + 3]);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              uint32_t pk[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float4 wa = w[2 * e], wb = w[2 * e + 1];
                const float va = fmaf(wa.z, dz[h], fmaf(wa.y, dy[h], fmaf(wa.x, dx[h], wa.w)));
                const float vb = fmaf(wb.z, dz[h], fmaf(wb.y, dy[h], fmaf(wb.x, dx[h], wb.w)));
                pk[e] = bias_act_pack(va, vb, 0.f, 0.f, relu);
              }
              *reinterpret_cast<uint4*>(sb + (size_t)g * (kTileRows * 16) + (size_t)h * (64 * 16)) =
                  make_uint4(pk[0], pk[1], pk[2], pk[3]);
            }
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive_n(&act_ready[slot], kEpiWarps / kLoadWarps);
          continue;
        }
        const long long tl1 = tick<PROF>();
        // (lane = row: an instruction touches 32 cache lines.  8 rows x 4 pieces per instruction — 8 lines, the
        // quarter-warps still conflict-free in shared memory — was measured 5 % SLOWER on the head chain, and an
        // L2 bulk prefetch of the next tile's rows changed nothing: the stall at a tile start is slot-bound.)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const long long row = tile_row(it, h, job.sub);
          const bool valid = row < p.P;
          const long long rr = valid ? row : 0;
          const int jq = job.sub ? jn[2 + h] : jn[h];
          uint8_t* sbase = slots + (size_t)slot * kSlotBytes + (size_t)(r + 64 * h) * 16;
          if (GATHER && job.kind == WK_LOAD_XYZ) {
            float xa = 0.f, xb = 0.f, xc = 0.f;
            if (valid) {
              const int b = (int)(rr / per_b);
              const int m = (int)((rr - (long long)b * per_b) / p.K);
              const float* X = p.xyz + (long long)b * 3 * p.N;
              const float* C = p.ctr + (long long)b * 3 * p.M;
              xa = __fsub_rn(__ldg(X + jq), __ldg(C + m));
              xb = __fsub_rn(__ldg(X + p.N + jq), __ldg(C + p.M + m));
              xc = __fsub_rn(__ldg(X + 2 * p.N + jq), __ldg(C + 2 * p.M + m));
            }
            __nv_bfloat162 h0 = __floats2bfloat162_rn(xa, xb), h1 = __floats2bfloat162_rn(xc, 0.f);
            *reinterpret_cast<uint4*>(sbase) =
                make_uint4(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1), 0u, 0u);
            *reinterpret_cast<uint4*>(sbase + kTileRows * 16) = make_uint4(0u, 0u, 0u, 0u);
          } else {
            const __nv_bfloat16* src;
            if constexpr (!GATHER) {
              src = reinterpret_cast<const __nv_bfloat16*>(p.in_rows) + rr * (long long)p.in_stride + job.c_begin;
            } else {
              const int b = (int)(rr / per_b);
              src = reinterpret_cast<const __nv_bfloat16*>(p.feat) + ((long long)b * p.N + jq) * p.feat_c + job.c_begin;
            }
            const int pieces = job.c_count >> 3;
#pragma unroll 4
            for (int c = 0; c < pieces; ++c) cp_async16(sbase + (size_t)c * (kTileRows * 16), src + c * 8, valid);
          }
        }
        if (PROF && p.prof && blockIdx.x == 0 && (it == 2 || it == 3) && r == 0) {  // loader timeline (chain_prof.py)
          long long* tr = p.prof + 148 * 16 + 4 * kMaxMmaJobs + 4 * kMaxEpiJobs + ((it - 2) * kMaxLoadJobs + j) * 4;
          tr[0] = tl0; tr[1] = tl1; tr[2] = tick<PROF>();
        }
        if (GATHER && job.kind == WK_LOAD_XYZ) {
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive_n(&act_ready[slot], kEpiWarps / kLoadWarps);
        } else {
          // the blocks committed before this one had this block's whole issue loop to land: publish them now,
          // not when the pipeline is full — the MMA warp starts a tile on its FIRST input block
          // (cp.async.wait_group only counts committed groups, so this does not wait for the copies just issued)
          if (npend) {
            cp_async_wait(0);
            while (npend) publish_oldest();
          }
          cp_async_commit();
          if (npend == 0) pend0 = slot; else if (npend == 1) pend1 = slot; else pend2 = slot;
          ++npend;
        }
      }
      ring_advance(base, p);
    }
    if (npend) {
      cp_async_wait(0);
      while (npend) publish_oldest();
    }
    if (PROF && p.prof && r == 0) {
      p.prof[blockIdx.x * 16 + 11] = tick<PROF>() - t_begin;
      p.prof[blockIdx.x * 16 + 8] = c_free;
      p.prof[blockIdx.x * 16 + 9] = c_cp;
    }
  } else {
    // ===================== epilogue warps: group g drains the accumulators with q % 2 == g =====================
    const int grp = warp >> 3;
    const int qd = warp & 3;              // TMEM lane quadrant this warp may read
    const int half = (warp >> 2) & 1;     // columns [64 half, 64 half + 64) of an accumulator block
    const int erow = qd * 32 + lane;      // tile row (= TMEM lane) in row-oriented epilogues
    const uint32_t lane_base = tmem_base + ((uint32_t)(qd * 32) << 16);
    Ring base = {0, 0u};
    unsigned base_q = 0;
    long long c_full = 0, c_free = 0, c_epi = 0;
    const long long t_begin = tick<PROF>();
    for (int it = 0; it < n_my; ++it) {
      const long long row0 = ((long long)blockIdx.x + (long long)it * gridDim.x) * tile_rows + erow;
      for (int j = 0; j < p.n_ep; ++j) {
        const WorkerJob job = p.ep[j];
        const long long row = row0 + (long long)job.sub * kTileRows;
        const unsigned q = base_q + job.acc;
        const bool coop = job.coop != 0;  // all 16 warps: 32 columns each; else the 8 warps of group q % 2: 64 each
        if (!coop && (int)(q & 1u) != grp) continue;
        const unsigned tb = q & (kAccBlocks - 1);
        const int c0 = coop ? 32 * (warp >> 2) : 64 * half;
        const uint32_t t_addr = lane_base + tb * 128u + (uint32_t)c0;
        const bool relu = job.relu != 0;
        if (job.kind == WK_EPI_HIDDEN || (OUT == OUT_ROWS && job.kind == WK_EPI_ROWS)) {
          const bool hidden = OUT != OUT_ROWS || job.kind == WK_EPI_HIDDEN;
          const int ncol = min(coop ? 32 : 64, (int)job.c_count - c0);  // columns of this warp: 64, 48, 32, 16 or <= 0
          const float* bias = p.bias[job.layer] + job.c_begin + c0;
          // the shifts of the first 32 columns travel while this warp waits for the accumulator
          float4 bv[8];  // the shift vectors are padded to a multiple of 128 floats: always in bounds
#pragma unroll
          for (int g = 0; g < 8; ++g) bv[g] = __ldg(reinterpret_cast<const float4*>(bias) + g);
          const long long t0 = tick<PROF>();
          mbar_wait(&tm_full[tb], (q >> 2) & 1);
          const long long t1 = tick<PROF>();
          c_full += t1 - t0;
          tc_fence_after();
          int slot = 0;
          unsigned use = 0;
          if (hidden) ring_at(base, p, job.blk_mod, job.blk_div, slot, use);
          const bool need_free = hidden && (job.same || it >= (int)job.min_it);
          const unsigned fpar = (unsigned)(job.same ? it : it - 1) & 1u;
          uint8_t* dst = slots + (size_t)slot * kSlotBytes + ((size_t)(c0 >> 3) * kTileRows + erow) * 16;
          __nv_bfloat16* orow = reinterpret_cast<__nv_bfloat16*>(p.out) + row * (long long)p.out_c + job.c_begin + c0;
          // edge chain, layer 0: this row's group term (rows past P stay without one; their groups are never emitted)
          const __nv_bfloat16* trow = nullptr;
          if constexpr (EDGE) {
            if (job.layer == 0 && row < p.P)
              trow = reinterpret_cast<const __nv_bfloat16*>(p.term) + (long long)((int)row / p.K) * p.term_c + job.c_begin + c0;
          }
          // full-width warps (64 columns, or 32 in a cooperative job): 32-column slabs, the second slab's shifts
          // travelling under its TMEM load.  Narrow layers (a multiple of 16 columns left): a compact 16-column
          // loop — the kernel's instruction footprint is what the common path pays for.
          if (ncol == 64 || ncol == 32) {
            float va[32];
            tmem_ld32_issue(t_addr, va);
            if constexpr (EDGE) add_term<8>(bv, trow);
            if (need_free) {
              mbar_wait(&blk_free[job.pred], fpar);
              c_free += tick<PROF>() - t1;
            }
            tmem_wait();
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              const uint4 pk = epi_piece_r(va + g * 8, bv[2 * g], bv[2 * g + 1], relu);
              if (hidden) *reinterpret_cast<uint4*>(dst + (size_t)g * (kTileRows * 16)) = pk;
              else if (row < p.P) *reinterpret_cast<uint4*>(orow + g * 8) = pk;
            }
            if (ncol == 64) {
              tmem_ld32_issue(t_addr + 32u, va);
#pragma unroll
              for (int g = 0; g < 8; ++g) bv[g] = __ldg(reinterpret_cast<const float4*>(bias + 32) + g);
              if constexpr (EDGE) add_term<8>(bv, trow ? trow + 32 : nullptr);
              tmem_wait();
#pragma unroll
              for (int g = 0; g < 4; ++g) {
                const uint4 pk = epi_piece_r(va + g * 8, bv[2 * g], bv[2 * g + 1], relu);
                if (hidden) *reinterpret_cast<uint4*>(dst + (size_t)(4 + g) * (kTileRows * 16)) = pk;
                else if (row < p.P) *reinterpret_cast<uint4*>(orow + 32 + g * 8) = pk;
              }
            }
          } else {
            if (need_free) mbar_wait(&blk_free[job.pred], fpar);
#pragma unroll 1
            for (int c = 0; c < ncol; c += 16) {
              float vh[16];
              tmem_ld16_issue(t_addr + (uint32_t)c, vh);
              float4 bw[4];
#pragma unroll
              for (int g = 0; g < 4; ++g) bw[g] = __ldg(reinterpret_cast<const float4*>(bias + c) + g);
              if constexpr (EDGE) add_term<4>(bw, trow ? trow + c : nullptr);
              tmem_wait();
#pragma unroll
              for (int g = 0; g < 2; ++g) {
                const uint4 pk = epi_piece_r(vh + g * 8, bw[2 * g], bw[2 * g + 1], relu);
                if (hidden) *reinterpret_cast<uint4*>(dst + (size_t)((c >> 3) + g) * (kTileRows * 16)) = pk;
                else if (row < p.P) *reinterpret_cast<uint4*>(orow + c + g * 8) = pk;
              }
            }
          }
          tc_fence_before();
          if (hidden) fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            const unsigned weight = coop ? 1u : 2u;
            if (hidden) mbar_arrive_n(&act_ready[slot], weight);
            mbar_arrive_n(&tm_empty[tb], weight);
          }
          c_epi += tick<PROF>() - t1;
          if (PROF && p.prof && blockIdx.x == 0 && it == 2 && (threadIdx.x & 255) == 0) {
            long long* tr = p.prof + 148 * 16 + 4 * kMaxMmaJobs + j * 4;
            tr[0] = t0; tr[1] = t1; tr[2] = tick<PROF>();
          }
          continue;
        }
        const long long t0 = tick<PROF>();
        mbar_wait(&tm_full[tb], (q >> 2) & 1);
        const long long t1 = tick<PROF>();
        c_full += t1 - t0;
        tc_fence_after();
        if (OUT == OUT_MAXPOOL && job.kind == WK_EPI_MAXPOOL) {
          // transposed: TMEM lane = output channel, columns = the tile's 128 positions; a group of G
          // adjacent columns is one centroid's neighbourhood (max commutes with +shift and ReLU).
          const int G = p.group;
          const int ch = job.c_begin + qd * 32 + lane;
          const float b = ch < p.out_c ? __ldg(p.bias[job.layer] + ch) : 0.f;
          __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(p.out);
          const long long n_groups = p.P / G;
          const long long tile_g0 = (((long long)blockIdx.x + (long long)it * gridDim.x) * tile_rows + job.sub * kTileRows) / G;
          float v0[32], v1[32];
          tmem_ld32_issue(t_addr, v0);
          tmem_ld32_issue(t_addr + 32u, v1);
          tmem_wait();
          auto emit = [&](float m, int col) {
            const long long gi = tile_g0 + col / G;
            if (gi < n_groups && ch < p.out_c) {
              const float t = m + b;
              out[gi * p.out_c + ch] = __float2bfloat16(relu ? fmaxf(t, 0.f) : t);
            }
          };
          if (G == 64) {
            float m = fmaxf(v0[0], v1[0]);
#pragma unroll
            for (int e = 1; e < 32; ++e) m = fmaxf(m, fmaxf(v0[e], v1[e]));
            emit(m, c0);
          } else {  // G = 32, 16 or 8: 64 / G groups in this warp's columns (compact code: the PN2_CLS levels use 64)
#pragma unroll 1
            for (int g0 = 0; g0 < 64; g0 += G) {
              float m = -3.4e38f;
#pragma unroll
              for (int e = 0; e < 32; ++e) {
                if (e >= g0 && e < g0 + G) m = fmaxf(m, v0[e]);
                if (e + 32 >= g0 && e + 32 < g0 + G) m = fmaxf(m, v1[e]);
              }
              emit(m, c0 + g0);
            }
          }
        } else if (OUT == OUT_LOGITS && half == 0) {  // WK_EPI_LOGITS: fp32, channel-first (B, out_c, n_points), bias, optional sigmoid
          const float* bias = p.bias[job.layer] + job.c_begin;
          float v[16];
          tmem_ld16_issue(t_addr, v);
          tmem_wait();
          if (row < p.P) {
            // (compact on purpose: index arithmetic hoisted, fast reciprocal — this loop is unrolled 16 times and
            // the kernel's instruction footprint is paid by every role)
            const long long bb = row / p.n_points;
            const long long n = row - bb * p.n_points;
            float* o = reinterpret_cast<float*>(p.out) + (bb * p.out_c) * p.n_points + n;
            const size_t stride = (size_t)p.n_points;
            const float4* b4 = reinterpret_cast<const float4*>(bias);
            const float4 b0 = __ldg(b4), b1 = __ldg(b4 + 1), b2 = __ldg(b4 + 2), b3 = __ldg(b4 + 3);
            const float bs[16] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w, b2.x, b2.y, b2.z, b2.w, b3.x, b3.y, b3.z, b3.w};
            const bool sig = p.sigmoid != 0;
#pragma unroll
            for (int c = 0; c < 16; ++c) {
              if (c < p.out_c) {
                float t = v[c] + bs[c];
                if (relu) t = fmaxf(t, 0.f);
                if (sig) t = __fdividef(1.f, 1.f + __expf(-t));
                o[c * stride] = t;
              }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_n(&tm_empty[tb], 2u);
        c_epi += tick<PROF>() - t1;
        if (PROF && p.prof && blockIdx.x == 0 && it == 2 && (threadIdx.x & 255) == 0) {
          long long* tr = p.prof + 148 * 16 + 4 * kMaxMmaJobs + j * 4;
          tr[0] = t0; tr[1] = t1; tr[2] = tick<PROF>();
        }
      }
      ring_advance(base, p);
      base_q += (unsigned)p.n_acc;
    }
    if (PROF && p.prof && threadIdx.x == 0) {
      p.prof[blockIdx.x * 16 + 6] = tick<PROF>() - t_begin;
      p.prof[blockIdx.x * 16 + 7] = c_full;
      p.prof[blockIdx.x * 16 + 12] = c_free;
      p.prof[blockIdx.x * 16 + 10] = c_epi;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem_base, 512u);
}

}  // namespace s4g

// ================================================================================================
// Host side: C ABI (plan in csrc/chain_plan.cu), weight packing, launch
// ================================================================================================
extern "C" s4g_chain* s4g_chain_create(int n_layers, const int* cin, const int* cout, const int* relu, int in_mode,
                                       int feat_c, int out_mode, int out_c, int group, int sigmoid) {
  s4g_chain* ch = new (std::nothrow) s4g_chain;
  if (!ch) return nullptr;
  if (s4g::plan_chain(ch, n_layers, cin, cout, relu, in_mode, feat_c, out_mode, out_c, group, sigmoid) != S4G_OK) {
    delete ch;
    return nullptr;
  }
  return ch;
}

// Same with planner decisions pinned, for host-side autotuning: slots = activation slots (0 = planner's choice),
// pairs = -1 planner's choice / 0 no N = 256 accumulator pairs / 1 pairs only, coop = -1 default policy / 0 none /
// 1 every row epilogue shared by all 16 warps / 2 the unpaired ones, subs = row blocks (128 rows) per tile: 1, or 2 =
// two tiles interleaved layer by layer.  NULL when no plan exists under the constraints.
// tma_in = 1 (row input, cin[0] a multiple of 64, not OUT_MAXPOOL): the input blocks are fetched with TMA tensor copies.
extern "C" s4g_chain* s4g_chain_create_tuned_in(int n_layers, const int* cin, const int* cout, const int* relu, int in_mode,
                                                int feat_c, int out_mode, int out_c, int group, int sigmoid, int slots,
                                                int pairs, int coop, int subs, int tma_in) {
  s4g_chain* ch = new (std::nothrow) s4g_chain;
  if (!ch) return nullptr;
  if (s4g::plan_chain(ch, n_layers, cin, cout, relu, in_mode, feat_c, out_mode, out_c, group, sigmoid, slots, pairs,
                      coop, subs, tma_in) != S4G_OK) {
    delete ch;
    return nullptr;
  }
  return ch;
}

extern "C" s4g_chain* s4g_chain_create_tuned(int n_layers, const int* cin, const int* cout, const int* relu, int in_mode,
                                             int feat_c, int out_mode, int out_c, int group, int sigmoid, int slots,
                                             int pairs, int coop, int subs) {
  return s4g_chain_create_tuned_in(n_layers, cin, cout, relu, in_mode, feat_c, out_mode, out_c, group, sigmoid, slots,
                                   pairs, coop, subs, 0);
}

extern "C" s4g_chain* s4g_chain_create_slots(int n_layers, const int* cin, const int* cout, const int* relu, int in_mode,
                                             int feat_c, int out_mode, int out_c, int group, int sigmoid, int slots) {
  return s4g_chain_create_tuned(n_layers, cin, cout, relu, in_mode, feat_c, out_mode, out_c, group, sigmoid, slots, -1, -1, 1);
}

extern "C" void s4g_chain_destroy(s4g_chain* ch) { delete ch; }

extern "C" size_t s4g_chain_weight_bytes(const s4g_chain* ch) { return ch ? ch->w_bytes : 0; }

// length (floats) of layer `layer`'s shift vector: the padded width rounded up to whole 128-column blocks
extern "C" int s4g_chain_cout_pad(const s4g_chain* ch, int layer) {
  return (ch && layer >= 0 && layer < ch->n_layers) ? (ch->cout_pad[layer] + 127) / 128 * 128 : -1;
}

// n_jobs: MMA jobs per tile; slots/stages: ring sizes; load_depth: input blocks in flight per loader
// thread; sim_cycles / mma_cycles: the planner's per-tile estimate and the tensor-pipe busy cycles in it.
extern "C" int s4g_chain_info(const s4g_chain* ch, int* n_jobs, int* slots, int* stages, int* load_depth,
                              int* smem_bytes, int* sim_cycles, int* mma_cycles) {
  S4G_CHECK_ARG(ch != nullptr, "mlp_chain: null chain");
  if (n_jobs) *n_jobs = ch->prm.n_mma;
  if (slots) *slots = ch->prm.slots;
  if (stages) *stages = ch->prm.stages;
  if (load_depth) *load_depth = ch->load_depth;
  if (smem_bytes) *smem_bytes = (int)ch->smem_bytes;
  if (sim_cycles) *sim_cycles = (int)ch->sim_cycles_per_tile;
  if (mma_cycles) *mma_cycles = (int)ch->mma_cycles_per_tile;
  return S4G_OK;
}

// Pack one layer's folded fp32 weights W[cout_real][cin_real] (row-major, host memory) into the bf16
// chunk stream the kernel consumes.  For a gathered first layer the reference's channel order
// [xyz(3) | features] (modules.py:48) becomes [features | xyz(3) | 0 x 13].
extern "C" int s4g_chain_pack_weights(const s4g_chain* ch, int layer, const float* w_host, int cout_real, int cin_real,
                                      void* packed_host) {
  S4G_CHECK_ARG(ch && w_host && packed_host, "mlp_chain: null pointer");
  S4G_CHECK_ARG(layer >= 0 && layer < ch->n_layers, "mlp_chain: bad layer");
  const s4g::ChainParams& p = ch->prm;
  __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(packed_host);
  size_t off = 0;  // in elements
  const bool gather0 = (layer == 0 && (ch->in_mode == s4g::IN_GATHER || ch->in_mode == s4g::IN_GATHER_EDGE));
  const int fc = p.feat_c;
  for (int j = 0; j < p.n_mma; ++j) {
    const s4g_chain::ChunkSrc& cs = ch->chunk[j];
    if (cs.layer == layer) {
      for (int kk = 0; kk < cs.k_count; ++kk) {
        const int c = cs.k_begin + kk;  // channel in the kernel's order
        int src_c;
        if (gather0) src_c = (c < fc) ? c + 3 : (c < fc + 3 ? c - fc : -1);
        else src_c = (c < cin_real) ? c : -1;
        for (int rr = 0; rr < cs.n_rows; ++rr) {
          const int o = cs.n_begin + rr;
          float v = 0.f;
          if (src_c >= 0 && src_c < cin_real && o < cout_real) v = w_host[(size_t)o * cin_real + src_c];
          dst[off + ((size_t)(kk >> 3) * cs.n_rows + rr) * 8 + (kk & 7)] = __float2bfloat16(v);
        }
      }
    }
    off += (size_t)cs.k_count * cs.n_rows;
  }
  return S4G_OK;
}

extern "C" int s4g_chain_set_params(s4g_chain* ch, const void* weights_dev, const float* const* bias_dev) {
  S4G_CHECK_ARG(ch && weights_dev && bias_dev, "mlp_chain: null pointer");
  S4G_CHECK_ARG(((uintptr_t)weights_dev & 15) == 0, "mlp_chain: weights must be 16-byte aligned");
  ch->prm.weights = weights_dev;
  for (int l = 0; l < ch->n_layers; ++l) {
    S4G_CHECK_ARG(((uintptr_t)bias_dev[l] & 15) == 0, "mlp_chain: shift vectors must be 16-byte aligned");
    ch->prm.bias[l] = bias_dev[l];
  }
  return S4G_OK;
}

// IN_XYZ_MLP chains: the BN-folded 3 -> cin[0] layer the loader warps evaluate in fp32.  w4_host: [cin[0]][4] fp32
// (w_x, w_y, w_z, shift) in HOST memory; it is copied into the kernel parameters.
extern "C" int s4g_chain_set_xyz_layer(s4g_chain* ch, const float* w4_host, int relu) {
  S4G_CHECK_ARG(ch && w4_host, "mlp_chain: null pointer");
  S4G_CHECK_ARG(ch->in_mode == s4g::IN_XYZ_MLP, "mlp_chain: chain was not planned with IN_XYZ_MLP");
  memcpy(ch->prm.xyz_w, w4_host, sizeof(float) * 4 * (size_t)ch->cin_pad[0]);
  ch->prm.xyz_relu = relu ? 1 : 0;
  ch->prm.xyz_set = 1;
  return S4G_OK;
}

// Optional per-CTA cycle counters (16 x int64 per CTA, >= 148 CTAs): [0] producer total, [1] producer
// waiting for a free stage; [2] MMA warp total, [3..5] waiting for activations / TMEM / weights;
// [6] epilogue warps total, [7] waiting for an accumulator, [12] for a free slot, [10] epilogue work;
// [11] loader total, [8] loader waiting for a free slot, [9] for cp.async.
extern "C" int s4g_chain_set_profile(s4g_chain* ch, void* counters_dev) {
  S4G_CHECK_ARG(ch != nullptr, "mlp_chain: null chain");
  ch->prm.prof = reinterpret_cast<long long*>(counters_dev);
  return S4G_OK;
}

namespace s4g {
template <bool PROF, bool XYZ_MLP, int OUT, bool GATHER, bool TMA_IN = false, bool EDGE = false>
static int launch_chain(const ChainParams& p, int grid, size_t smem, cudaStream_t stream) {
  auto kern = mlp_chain_kernel<PROF, XYZ_MLP, OUT, GATHER, TMA_IN, EDGE>;
  static bool attr_set[64] = {};
  if (s4g::first_use_on_device(attr_set)) {
    S4G_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  }
  kern<<<grid, kChainThreads, smem, stream>>>(p);
  return S4G_OK;
}
}  // namespace s4g

static int s4g_chain_launch(const s4g_chain* ch, s4g::ChainParams& p, cudaStream_t stream) {
  S4G_CHECK_ARG(p.weights != nullptr, "mlp_chain: s4g_chain_set_params was not called");
  if (p.P <= 0) return S4G_OK;
  const int tile_rows = s4g::kTileRows * p.subs;
  const int tiles = (p.P + tile_rows - 1) / tile_rows;
  const int grid = tiles < s4g::num_sms() ? tiles : s4g::num_sms();
  const bool gather = p.in_mode != s4g::IN_ROWS, xyz = p.in_mode == s4g::IN_XYZ_MLP, prof = p.prof != nullptr;
  const bool edge = p.in_mode == s4g::IN_GATHER_EDGE;
  S4G_CHECK_ARG(!(xyz && prof), "mlp_chain: the cycle counters are not built for IN_XYZ_MLP chains");
  S4G_CHECK_ARG(!(p.tma_in && prof), "mlp_chain: the cycle counters are not built for TMA-input chains");
  S4G_CHECK_ARG(!(edge && prof), "mlp_chain: the cycle counters are not built for edge chains");
  int rc = S4G_E_UNSUPPORTED;
  if (edge) {  // (the planner admits edge chains only as gathered max-pool chains)
    if (ch->out_mode == s4g::OUT_MAXPOOL)
      rc = p.tma_in ? s4g::launch_chain<false, false, s4g::OUT_MAXPOOL, true, true, true>(p, grid, ch->smem_bytes, stream)
                    : s4g::launch_chain<false, false, s4g::OUT_MAXPOOL, true, false, true>(p, grid, ch->smem_bytes, stream);
  } else if (p.tma_in) {
    if (ch->out_mode == s4g::OUT_ROWS && !gather) rc = s4g::launch_chain<false, false, s4g::OUT_ROWS, false, true>(p, grid, ch->smem_bytes, stream);
    if (ch->out_mode == s4g::OUT_LOGITS) rc = s4g::launch_chain<false, false, s4g::OUT_LOGITS, false, true>(p, grid, ch->smem_bytes, stream);
    if (ch->out_mode == s4g::OUT_MAXPOOL && gather) rc = s4g::launch_chain<false, false, s4g::OUT_MAXPOOL, true, true>(p, grid, ch->smem_bytes, stream);
  } else {
#define S4G_CHAIN_CASE(PROF_, XYZ_, OUT_, GATHER_)                                                                     \
  if (prof == PROF_ && xyz == XYZ_ && ch->out_mode == s4g::OUT_ && gather == GATHER_)                                  \
    rc = s4g::launch_chain<PROF_, XYZ_, s4g::OUT_, GATHER_>(p, grid, ch->smem_bytes, stream);
  S4G_CHAIN_CASE(false, false, OUT_ROWS, false)
  S4G_CHAIN_CASE(false, false, OUT_LOGITS, false)
  S4G_CHAIN_CASE(false, false, OUT_MAXPOOL, false)
  S4G_CHAIN_CASE(false, false, OUT_ROWS, true)
  S4G_CHAIN_CASE(false, false, OUT_LOGITS, true)
  S4G_CHAIN_CASE(false, false, OUT_MAXPOOL, true)
  S4G_CHAIN_CASE(true, false, OUT_ROWS, false)
  S4G_CHAIN_CASE(true, false, OUT_LOGITS, false)
  S4G_CHAIN_CASE(true, false, OUT_MAXPOOL, false)
  S4G_CHAIN_CASE(true, false, OUT_ROWS, true)
  S4G_CHAIN_CASE(true, false, OUT_LOGITS, true)
  S4G_CHAIN_CASE(true, false, OUT_MAXPOOL, true)
  S4G_CHAIN_CASE(false, true, OUT_ROWS, true)
  S4G_CHAIN_CASE(false, true, OUT_LOGITS, true)
  S4G_CHAIN_CASE(false, true, OUT_MAXPOOL, true)
#undef S4G_CHAIN_CASE
  }
  if (rc != S4G_OK) return rc == S4G_E_UNSUPPORTED ? s4g::set_error(rc, "mlp_chain: no kernel for this chain type") : rc;
  S4G_LAUNCH_CHECK("mlp_chain");
  return S4G_OK;
}

// 2-D tensor map of a bf16 row table [rows][width] (dim 0 = channels), box = 64 channels x box_rows rows, 128-byte swizzle
static int encode_rows_map(CUtensorMap* map, const void* base, long long width, long long rows, int box_rows) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    S4G_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    S4G_CHECK_ARG(fn != nullptr && qres == cudaDriverEntryPointSuccess, "mlp_chain: cuTensorMapEncodeTiled is not available");
    encode = reinterpret_cast<EncodeFn>(fn);
  }
  const cuuint64_t dims[2] = {(cuuint64_t)width, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)width * 2u};
  const cuuint32_t box[2] = {64u, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1u, 1u};
  const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  S4G_CHECK_ARG(r == CUDA_SUCCESS, "mlp_chain: cuTensorMapEncodeTiled failed");
  return S4G_OK;
}

// rows in: in_rows [P][in_stride] bf16 channel-last.  out: ROWS -> bf16 [P][out_c];
// LOGITS -> fp32 (P / n_points, out_c, n_points).
extern "C" int s4g_chain_run_rows(const s4g_chain* ch, const void* in_rows, int in_stride, long long P, void* out,
                                  int n_points, void* stream) {
  S4G_CHECK_ARG(ch && in_rows && out, "mlp_chain: null pointer");
  S4G_CHECK_ARG(ch->in_mode == s4g::IN_ROWS, "mlp_chain: chain was planned for gathered input");
  S4G_CHECK_ARG(P >= 0 && P < (1ll << 31), "mlp_chain: bad row count");
  S4G_CHECK_ARG(in_stride >= ch->cin_pad[0] && in_stride % 8 == 0 && ((uintptr_t)in_rows & 15) == 0,
                "mlp_chain: input rows must be 16-byte aligned and at least cin wide");
  if (ch->out_mode == s4g::OUT_LOGITS) S4G_CHECK_ARG(n_points > 0 && P % n_points == 0, "mlp_chain: bad n_points");
  else S4G_CHECK_ARG(((uintptr_t)out & 15) == 0, "mlp_chain: output rows must be 16-byte aligned");
  s4g::ChainParams p = ch->prm;
  p.P = (int)P;
  p.in_rows = in_rows;
  p.in_stride = in_stride;
  p.out = out;
  p.n_points = n_points > 0 ? n_points : 1;
  if (p.tma_in && P > 0) {  // box = 64 channels x 128 rows
    const int rc = encode_rows_map(&p.in_map, in_rows, in_stride, P, s4g::kTileRows);
    if (rc != S4G_OK) return rc;
  }
  return s4g_chain_launch(ch, p, (cudaStream_t)stream);
}

// gathered in (set abstraction): feat [B*N][feat_c] bf16 (or NULL when feat_c == 0), xyz (B,3,N) fp32,
// ctr (B,3,M) fp32, nbr (B,M,K) int32; term bf16 [B*M][cout[0]] of an edge chain, else NULL.
// out: MAXPOOL -> bf16 [B*M][out_c]; ROWS -> bf16 [B*M*K][out_c].
static int run_gather(const s4g_chain* ch, const void* feat, const float* xyz, const float* ctr, const int* nbr,
                      const void* term, int B, int N, int M, int K, void* out, void* stream) {
  S4G_CHECK_ARG(ch && xyz && ctr && nbr && out, "mlp_chain: null pointer");
  S4G_CHECK_ARG(ch->in_mode != s4g::IN_ROWS, "mlp_chain: chain was planned for row input");
  S4G_CHECK_ARG(ch->in_mode != s4g::IN_XYZ_MLP || ch->prm.xyz_set, "mlp_chain: s4g_chain_set_xyz_layer was not called");
  S4G_CHECK_ARG(ch->prm.feat_c == 0 || (feat != nullptr && ((uintptr_t)feat & 15) == 0), "mlp_chain: bad feature table");
  S4G_CHECK_ARG((long long)B * M * K < (1ll << 31), "mlp_chain: too many rows");
  if (ch->out_mode == s4g::OUT_MAXPOOL) S4G_CHECK_ARG(K == ch->prm.group, "mlp_chain: K != planned max-pool group");
  s4g::ChainParams p = ch->prm;
  p.P = B * M * K;
  p.feat = feat;
  p.xyz = xyz;
  p.ctr = ctr;
  p.nbr = nbr;
  p.N = N; p.M = M; p.K = K;
  p.out = out;
  p.term = term;
  if (p.tma_in && p.P > 0) {  // tile::gather4 copies: box = 64 channels x 1 row of the feature table
    S4G_CHECK_ARG(K % 4 == 0 && ((uintptr_t)nbr & 15) == 0, "mlp_chain: TMA gather needs K % 4 == 0 and 16-byte aligned indices");
    const int rc = encode_rows_map(&p.in_map, feat, ch->prm.feat_c, (long long)B * N, 1);
    if (rc != S4G_OK) return rc;
  }
  return s4g_chain_launch(ch, p, (cudaStream_t)stream);
}

extern "C" int s4g_chain_run_gather(const s4g_chain* ch, const void* feat, const float* xyz, const float* ctr,
                                    const int* nbr, int B, int N, int M, int K, void* out, void* stream) {
  S4G_CHECK_ARG(!ch || ch->in_mode != s4g::IN_GATHER_EDGE, "mlp_chain: an edge chain runs with s4g_chain_run_gather_term");
  return run_gather(ch, feat, xyz, ctr, nbr, nullptr, B, N, M, K, out, stream);
}

// An edge level (EdgeSAModule): the gathered max-pool chain whose layer 0 adds term[b * M + m] (bf16, cout[0] wide,
// 16-byte aligned rows) to the shifts of every row of centroid m's group, before the ReLU.
extern "C" int s4g_chain_run_gather_term(const s4g_chain* ch, const void* feat, const float* xyz, const float* ctr,
                                         const int* nbr, const void* term, int B, int N, int M, int K, void* out,
                                         void* stream) {
  S4G_CHECK_ARG(ch && ch->in_mode == s4g::IN_GATHER_EDGE, "mlp_chain: s4g_chain_run_gather_term needs an edge chain");
  S4G_CHECK_ARG(term != nullptr && ((uintptr_t)term & 15) == 0, "mlp_chain: the group term must be 16-byte aligned");
  return run_gather(ch, feat, xyz, ctr, nbr, term, B, N, M, K, out, stream);
}
