// Element-wise / reduction kernels of the TRAINING path (channel-last bf16 rows [P][C], C % 8 == 0), around the tcgen05
// GEMM of csrc/gemm_bf16.cu.  Together they are one shared-MLP block of the reference in training mode
// (nn_utils/conv.py:30-36,70-76: 1x1 conv -> BatchNorm with batch statistics -> ReLU, nn_utils/mlp.py:99-101 dropout) and
// its backward, plus the set-abstraction max-pool (pointnet2_utils/modules.py:243), the grouping gather / scatter
// (grouping_kernel.cu:32-54,57-96) and the interpolation scatter (interpolate_kernel.cu:243-286) in the same layout:
//
//   colstats            sum_r y, sum_r y^2 per channel (fp64 accumulation across blocks)        -> batch mean / variance
//   bn_act              z = drop(relu(y * scale + shift))                                       -> next layer's input
//   bn_act_maxpool      the same followed by the max over each group of K consecutive rows, arg-max kept (uint8)
//   bn_bwd_reduce       sum_r g, sum_r g * xhat with g = dz * relu' * drop   (dz dense, or routed through the arg-max)
//   bn_bwd_apply        dy = gamma * rstd * (g - mean(g) - xhat * mean(g * xhat))               -> bf16
//   group_rows          X0[(b,m,k)] = [feat[b, nbr] | xyz[b, nbr] - ctr[b, m] | 0]              (gather, forward)
//   group_rows_bwd      dfeat[b, nbr] += dX0[(b,m,k)]                                           (fp32 vector atomics)
//   interp_rows_bwd     dsparse[b, idx_k] += w_k * dx[(b,q)]                                    (fp32 vector atomics)
//
// Every thread owns one 16-byte piece (8 channels) of a row, so all global accesses are 16-byte vectors and adjacent
// threads touch adjacent pieces.  Dropout is a counter-based hash of (seed, row, channel): the backward recomputes the
// mask instead of storing it.
#include <cuda_bf16.h>
#include <stdlib.h>

#include "common.cuh"

namespace s4g {
namespace trn {

struct F8 { float v[8]; };

__device__ __forceinline__ F8 unpack8(const uint4 q) {
  F8 r;
  const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    r.v[2 * i] = __uint_as_float(w[i] << 16);
    r.v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
  return r;
}
__device__ __forceinline__ uint4 pack8(const F8& f) {
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __nv_bfloat162 h = __floats2bfloat162_rn(f.v[2 * i], f.v[2 * i + 1]);
    w[i] = *reinterpret_cast<uint32_t*>(&h);
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}
__device__ __forceinline__ F8 load_f8(const float* p) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  return F8{{a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w}};
}
// keep-mask bit of element (row, channel): a 32-bit mix of the linear index and the seed (murmur3 finaliser)
__device__ __forceinline__ bool keep_elem(unsigned seed, long long row, int ch, int C, unsigned thresh) {
  unsigned long long idx = (unsigned long long)row * (unsigned)C + (unsigned)ch;
  unsigned h = (unsigned)idx ^ (unsigned)(idx >> 32) * 0x9E3779B9u ^ seed;
  h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
  return h >= thresh;  // P(keep) = 1 - thresh / 2^32
}

// ---------------------------------------------------------------------------------------------- colstats
constexpr int kStatThreads = 256;
constexpr int kStatRows = 512;  // rows per block

__global__ void __launch_bounds__(kStatThreads)
colstats_kernel(const __nv_bfloat16* __restrict__ y, long long ld, long long P, int C, double* __restrict__ out) {
  extern __shared__ float s_part[];  // [row lanes][C][2]
  const int pieces = C >> 3;
  const int lanes = kStatThreads / pieces;  // row lanes per block (pieces <= 256)
  const int piece = threadIdx.x % pieces, rl = threadIdx.x / pieces;
  const long long r0 = (long long)blockIdx.x * kStatRows;
  const long long r1 = min(P, r0 + kStatRows);
  F8 s{}, q{};
  if (rl < lanes) {
    for (long long r = r0 + rl; r < r1; r += 4LL * lanes) {  // four rows in flight per thread
      uint4 raw[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const long long rr = r + (long long)u * lanes;
        raw[u] = rr < r1 ? __ldg(reinterpret_cast<const uint4*>(y + rr * ld) + piece) : make_uint4(0u, 0u, 0u, 0u);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const F8 v = unpack8(raw[u]);
#pragma unroll
        for (int e = 0; e < 8; ++e) { s.v[e] += v.v[e]; q.v[e] = fmaf(v.v[e], v.v[e], q.v[e]); }
      }
    }
    float* dst = s_part + ((size_t)rl * pieces + piece) * 16;
#pragma unroll
    for (int e = 0; e < 8; ++e) { dst[e] = s.v[e]; dst[8 + e] = q.v[e]; }
  }
  __syncthreads();
  // thread t < 2 * C: column t of the [lanes][pieces * 16] table
  for (int t = threadIdx.x; t < pieces * 16; t += kStatThreads) {
    double acc = 0.0;
    for (int l = 0; l < lanes; ++l) acc += (double)s_part[(size_t)l * pieces * 16 + t];
    const int pc = t >> 4, e = t & 15;
    atomicAdd(out + (e < 8 ? 0 : C) + pc * 8 + (e & 7), acc);
  }
}

// ---------------------------------------------------------------------------------------------- bn_act (+ maxpool)
// thread = (16-byte piece, row lane): the per-channel parameters are loaded once and reused for every row of the block's
// chunk; four rows are in flight per thread
constexpr int kEltRows = 256;  // rows per block of the element-wise kernels

__global__ void __launch_bounds__(256)
bn_act_kernel(const __nv_bfloat16* __restrict__ y, const float* __restrict__ scale, const float* __restrict__ shift,
              __nv_bfloat16* __restrict__ z, long long P, int C, int relu, unsigned seed, unsigned thresh, float keep_scale) {
  const int pieces = C >> 3;
  const int lanes = 256 / pieces;
  const int piece = threadIdx.x % pieces, rl = threadIdx.x / pieces;
  if (rl >= lanes) return;
  const long long r1 = min(P, ((long long)blockIdx.x + 1) * kEltRows);
  const F8 a = load_f8(scale + piece * 8), b = load_f8(shift + piece * 8);
  for (long long r = (long long)blockIdx.x * kEltRows + rl; r < r1; r += 4LL * lanes) {
    uint4 raw[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long rr = r + (long long)u * lanes;
      if (rr < r1) raw[u] = __ldg(reinterpret_cast<const uint4*>(y + rr * C) + piece);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long rr = r + (long long)u * lanes;
      if (rr >= r1) break;
      const F8 v = unpack8(raw[u]);
      F8 o;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        float t = fmaf(v.v[e], a.v[e], b.v[e]);
        if (relu) t = fmaxf(t, 0.f);
        if (thresh) t = keep_elem(seed, rr, piece * 8 + e, C, thresh) ? t * keep_scale : 0.f;
        o.v[e] = t;
      }
      reinterpret_cast<uint4*>(z + rr * C)[piece] = pack8(o);
    }
  }
}

__global__ void __launch_bounds__(256)
bn_act_maxpool_kernel(const __nv_bfloat16* __restrict__ y, const float* __restrict__ scale, const float* __restrict__ shift,
                      __nv_bfloat16* __restrict__ out, uint8_t* __restrict__ arg, __nv_bfloat16* __restrict__ ymax, long long G,
                      int K, int C, int relu) {
  const int pieces = C >> 3;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= G * pieces) return;
  const long long g = i / pieces;
  const int piece = (int)(i - g * pieces);
  const F8 a = load_f8(scale + piece * 8), b = load_f8(shift + piece * 8);
  F8 best, raw;  // raw: the pre-BatchNorm value at the arg-max (what the backward's reduce needs of this group)
  int bi[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { best.v[e] = -3.4e38f; raw.v[e] = 0.f; bi[e] = 0; }
  const uint4* src = reinterpret_cast<const uint4*>(y + g * K * C) + piece;
  for (int k0 = 0; k0 < K; k0 += 4) {  // four rows in flight
    uint4 rawv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (k0 + u < K) rawv[u] = __ldg(src + (size_t)(k0 + u) * pieces);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int k = k0 + u;
      if (k >= K) break;
      const F8 v = unpack8(rawv[u]);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        float t = fmaf(v.v[e], a.v[e], b.v[e]);
        if (relu) t = fmaxf(t, 0.f);
        if (t > best.v[e]) { best.v[e] = t; raw.v[e] = v.v[e]; bi[e] = k; }  // first maximum wins, like torch.max
      }
    }
  }
  reinterpret_cast<uint4*>(out + g * C)[piece] = pack8(best);
  if (ymax) reinterpret_cast<uint4*>(ymax + g * C)[piece] = pack8(raw);  // exact: raw holds bf16 values
  uint2 packed;
  packed.x = (unsigned)bi[0] | ((unsigned)bi[1] << 8) | ((unsigned)bi[2] << 16) | ((unsigned)bi[3] << 24);
  packed.y = (unsigned)bi[4] | ((unsigned)bi[5] << 8) | ((unsigned)bi[6] << 16) | ((unsigned)bi[7] << 24);
  reinterpret_cast<uint2*>(arg + g * C)[piece] = packed;
}

// ---------------------------------------------------------------------------------------------- global max-pool
// bn_act followed by the max over ALL N rows of each scene: the one group of a global set-abstraction level
// (num_centroids = 0, modules.py:93-98 + the torch.max of :106).  N is any size, so a scene's rows are split across
// CTAs (grid = chunks x B).  Per channel the result is carried as one 64-bit key, (fp32 activation in an order-preserving
// encoding) << 32 | ~row: the largest key is the largest activation at its FIRST row, the torch.max rule of
// bn_act_maxpool_kernel.  A thread keeps its running maximum as (value, row), the CTA merges its threads' keys with
// shared-memory atomicMax and the CTAs theirs with global atomicMax: a maximum does not depend on the order of the
// merges, so the result is the same bits on every run.  bn_act_segmax_finish_kernel then decodes the keys.
constexpr int kSegRows = 512;  // rows per CTA

__device__ __forceinline__ unsigned long long seg_key(float t, unsigned row) {
  const unsigned u = __float_as_uint(t);
  const unsigned o = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((unsigned long long)o << 32) | (unsigned long long)(~row);
}
__device__ __forceinline__ float seg_key_value(unsigned long long key) {
  const unsigned o = (unsigned)(key >> 32);
  return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}

__global__ void __launch_bounds__(256)
bn_act_segmax_kernel(const __nv_bfloat16* __restrict__ y, const float* __restrict__ scale, const float* __restrict__ shift,
                     long long N, int C, int relu, unsigned long long* __restrict__ keys) {
  extern __shared__ unsigned long long s_key[];  // [C]
  const int pieces = C >> 3;
  const int lanes = 256 / pieces;
  const int piece = threadIdx.x % pieces, rl = threadIdx.x / pieces;
  const long long b = blockIdx.y;
  for (int c = threadIdx.x; c < C; c += 256) s_key[c] = 0ull;  // (below every encoded activation)
  __syncthreads();
  if (rl < lanes) {
    const long long r0 = (long long)blockIdx.x * kSegRows;
    const long long r1 = min(N, r0 + kSegRows);
    const F8 a = load_f8(scale + piece * 8), sh = load_f8(shift + piece * 8);
    const __nv_bfloat16* src = y + b * N * C;
    float best[8];
    int bi[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) { best[e] = 0.f; bi[e] = -1; }
    for (long long r = r0 + rl; r < r1; r += 4LL * lanes) {  // four rows in flight, each thread's rows in order
      uint4 raw[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const long long rr = r + (long long)u * lanes;
        if (rr < r1) raw[u] = __ldg(reinterpret_cast<const uint4*>(src + rr * C) + piece);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const long long rr = r + (long long)u * lanes;
        if (rr >= r1) break;
        const F8 v = unpack8(raw[u]);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          float t = fmaf(v.v[e], a.v[e], sh.v[e]);
          if (relu) t = fmaxf(t, 0.f);
          if (bi[e] < 0 || t > best[e]) { best[e] = t; bi[e] = (int)rr; }  // first maximum wins
        }
      }
    }
#pragma unroll
    for (int e = 0; e < 8; ++e)
      if (bi[e] >= 0) atomicMax(&s_key[piece * 8 + e], seg_key(best[e], (unsigned)bi[e]));
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += 256)
    if (s_key[c]) atomicMax(keys + b * C + c, s_key[c]);
}

// keys [B][C] -> out = bf16(max activation), arg = its row inside the scene (int32), ymax = y at that row (bf16, exact)
__global__ void __launch_bounds__(256)
bn_act_segmax_finish_kernel(const unsigned long long* __restrict__ keys, const __nv_bfloat16* __restrict__ y, long long N,
                            int C, long long BP, __nv_bfloat16* __restrict__ out, int* __restrict__ arg,
                            __nv_bfloat16* __restrict__ ymax) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // (scene, piece)
  if (i >= BP) return;
  const int pieces = C >> 3;
  const long long b = i / pieces;
  const int piece = (int)(i - b * pieces);
  F8 best, raw;
  int ai[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const unsigned long long k = __ldg(keys + i * 8 + e);
    best.v[e] = seg_key_value(k);
    ai[e] = (int)~(unsigned)k;
    if (ymax) raw.v[e] = __bfloat162float(y[(b * N + ai[e]) * C + piece * 8 + e]);
  }
  reinterpret_cast<uint4*>(out)[i] = pack8(best);
  reinterpret_cast<int4*>(arg)[2 * i] = make_int4(ai[0], ai[1], ai[2], ai[3]);
  reinterpret_cast<int4*>(arg)[2 * i + 1] = make_int4(ai[4], ai[5], ai[6], ai[7]);
  if (ymax) reinterpret_cast<uint4*>(ymax)[i] = pack8(raw);
}

// d_global[b][c] += sum_n dz[b * Nq + n][c], c < C2 (dz rows ld wide): the gradient of a broadcast propagation level's
// [global | skip] rows with respect to the global feature (modules.py:131-134 expand).  CTA = (group of up to 32 pieces,
// scene); each thread sums a fixed set of rows in order, the row lanes are summed in order in shared memory: a fixed
// reduction order, no atomics, the same bits on every run.
constexpr int kSumPieces = 32;

__global__ void __launch_bounds__(256)
rows_segment_sum_kernel(const __nv_bfloat16* __restrict__ dz, long long ld, long long Nq, int C2, float* __restrict__ out) {
  __shared__ float s_part[256 * 8];  // [lanes][pieces of the CTA][8]
  const int pieces = C2 >> 3;
  const int pg = min(pieces, kSumPieces);
  const int lanes = 256 / pg;
  const int pl = threadIdx.x % pg, rl = threadIdx.x / pg;
  const int piece = blockIdx.x * pg + pl;
  const long long b = blockIdx.y;
  F8 acc{};
  if (rl < lanes && piece < pieces) {
    const __nv_bfloat16* src = dz + b * Nq * ld;
    for (long long r = rl; r < Nq; r += 4LL * lanes) {
      uint4 raw[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const long long rr = r + (long long)u * lanes;
        if (rr < Nq) raw[u] = __ldg(reinterpret_cast<const uint4*>(src + rr * ld) + piece);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (r + (long long)u * lanes >= Nq) break;
        const F8 v = unpack8(raw[u]);
#pragma unroll
        for (int e = 0; e < 8; ++e) acc.v[e] += v.v[e];
      }
    }
  }
  if (rl < lanes) {
    float* dst = s_part + ((size_t)rl * pg + pl) * 8;
#pragma unroll
    for (int e = 0; e < 8; ++e) dst[e] = acc.v[e];
  }
  __syncthreads();
  for (int t = threadIdx.x; t < pg * 8; t += 256) {
    const int c = (blockIdx.x * pg) * 8 + t;
    if (c >= C2) break;
    float s = 0.f;
    for (int l = 0; l < lanes; ++l) s += s_part[(size_t)l * pg * 8 + t];
    out[b * C2 + c] += s;
  }
}

// ---------------------------------------------------------------------------------------------- BN backward
// g of one piece: dense upstream gradient, or the pooled gradient routed to the arg-max row (K > 0)
struct Upstream {
  const __nv_bfloat16* dz;   // dense: [P][C];   pooled: [G][C]
  const uint8_t* arg;        // pooled only: [G][C]
  int K;                     // 0 = dense
  int kshift;                // log2 K when K is a power of two (every shipped configuration), else -1
  const int* arg32;          // pooled with int32 arg-max rows (the groups of a global level: K = the scene's N rows)
};
static Upstream make_upstream(const void* dz, const uint8_t* arg, int K, const int* arg32 = nullptr) {
  int sh = -1;
  if (K > 0 && (K & (K - 1)) == 0) { sh = 0; while ((1 << sh) < K) ++sh; }
  return Upstream{reinterpret_cast<const __nv_bfloat16*>(dz), arg, K, sh, arg32};
}
struct UpRaw { uint4 d; uint2 a; int k; };
// load now (raw, 16 B + 8 B), route later: keeps the loads of several rows in flight without holding converted values
__device__ __forceinline__ UpRaw upstream_load(const Upstream& u, long long row, int piece, int C) {
  UpRaw r;
  if (u.K == 0) {
    r.d = __ldg(reinterpret_cast<const uint4*>(u.dz + row * C) + piece);
    r.a = make_uint2(0u, 0u);
    r.k = -1;
  } else {
    long long g;
    if (u.kshift >= 0) {  // (a 64-bit division per row and thread was a visible part of the pooled pass: ncu, 59-63 % issue)
      g = row >> u.kshift;
      r.k = (int)(row & (long long)(u.K - 1));
    } else {
      g = row / u.K;
      r.k = (int)(row - g * u.K);
    }
    r.d = __ldg(reinterpret_cast<const uint4*>(u.dz + g * C) + piece);
    r.a = __ldg(reinterpret_cast<const uint2*>(u.arg + g * C) + piece);
  }
  return r;
}
// pooled: keep the gradient of the channels whose arg-max is this row — byte-wise compare of the 8 packed indices, the
// 8-bit masks widened to the 16-bit bf16 lanes by byte permutes (10 instructions instead of a select per channel)
__device__ __forceinline__ F8 upstream_route(const UpRaw& r) {
  uint4 d = r.d;
  if (r.k >= 0) {
    const unsigned kk = (unsigned)r.k * 0x01010101u;
    const unsigned m0 = __vcmpeq4(r.a.x, kk), m1 = __vcmpeq4(r.a.y, kk);
    d.x &= __byte_perm(m0, 0u, 0x1100);
    d.y &= __byte_perm(m0, 0u, 0x3322);
    d.z &= __byte_perm(m1, 0u, 0x1100);
    d.w &= __byte_perm(m1, 0u, 0x3322);
  }
  return unpack8(d);
}
// pooled with int32 arg-max rows (bn_act_segmax): routed at load time — the 32 bytes of indices are not kept in flight —
// so the result is a routed dense piece (k = -1) for upstream_route.  Rows < 2^31 (checked by the host): 32-bit division.
__device__ __forceinline__ UpRaw upstream_load32(const Upstream& u, long long row, int piece, int C) {
  UpRaw r;
  unsigned g, k;
  if (u.kshift >= 0) {
    g = (unsigned)row >> u.kshift;
    k = (unsigned)row & (unsigned)(u.K - 1);
  } else {
    g = (unsigned)row / (unsigned)u.K;
    k = (unsigned)row - g * (unsigned)u.K;
  }
  uint4 d = __ldg(reinterpret_cast<const uint4*>(u.dz + (long long)g * C) + piece);
  const uint4* ap = reinterpret_cast<const uint4*>(u.arg32 + (long long)g * C) + 2 * piece;
  const uint4 a0 = __ldg(ap), a1 = __ldg(ap + 1);
  // bf16 lane pairs: the low half of each word is the even channel
  d.x &= (a0.x == k ? 0x0000ffffu : 0u) | (a0.y == k ? 0xffff0000u : 0u);
  d.y &= (a0.z == k ? 0x0000ffffu : 0u) | (a0.w == k ? 0xffff0000u : 0u);
  d.z &= (a1.x == k ? 0x0000ffffu : 0u) | (a1.y == k ? 0xffff0000u : 0u);
  d.w &= (a1.z == k ? 0x0000ffffu : 0u) | (a1.w == k ? 0xffff0000u : 0u);
  r.d = d;
  r.a = make_uint2(0u, 0u);
  r.k = -1;
  return r;
}
// the upstream kinds the BatchNorm-backward kernels are compiled for
enum { kUpDenseOrArg8 = 0, kUpArg32 = 1 };
template <int UP>
__device__ __forceinline__ UpRaw upstream_load_k(const Upstream& u, long long row, int piece, int C) {
  if constexpr (UP == kUpArg32) return upstream_load32(u, row, piece, C);
  else return upstream_load(u, row, piece, C);
}

// sums = [sum_r g | sum_r g * y]; the caller turns the second into sum g * xhat = rstd * (sum g y - mean * sum g) in fp64
// (keeps mean / rstd out of the loop: 16 registers less, a third block per SM)
template <int U, int MINB, int UP = kUpDenseOrArg8>  // U rows in flight per thread, MINB resident blocks per SM
__global__ void __launch_bounds__(kStatThreads, MINB)
bn_bwd_reduce_kernel(Upstream up, const __nv_bfloat16* __restrict__ y, const float* __restrict__ scale,
                     const float* __restrict__ shift, long long P, int C, int relu, unsigned seed, unsigned thresh,
                     float keep_scale, double* __restrict__ out) {
  extern __shared__ float s_part[];
  const int pieces = C >> 3;
  const int lanes = kStatThreads / pieces;
  const int piece = threadIdx.x % pieces, rl = threadIdx.x / pieces;
  const long long r0 = (long long)blockIdx.x * kStatRows;
  const long long r1 = min(P, r0 + kStatRows);
  F8 s{}, q{};
  if (rl < lanes) {
    const F8 a = load_f8(scale + piece * 8), b = load_f8(shift + piece * 8);
    for (long long r = r0 + rl; r < r1; r += (long long)U * lanes) {
      uint4 raw[U];
      UpRaw ur[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long rr = r + (long long)u * lanes;
        if (rr < r1) {
          raw[u] = __ldg(reinterpret_cast<const uint4*>(y + rr * C) + piece);
          ur[u] = upstream_load_k<UP>(up, rr, piece, C);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long rr = r + (long long)u * lanes;
        if (rr >= r1) break;
        const F8 v = unpack8(raw[u]);
        const F8 d = upstream_route(ur[u]);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          float g = d.v[e];
          if (relu && !(fmaf(v.v[e], a.v[e], b.v[e]) > 0.f)) g = 0.f;
          if (thresh) g = keep_elem(seed, rr, piece * 8 + e, C, thresh) ? g * keep_scale : 0.f;
          s.v[e] += g;
          q.v[e] = fmaf(g, v.v[e], q.v[e]);
        }
      }
    }
    float* dst = s_part + ((size_t)rl * pieces + piece) * 16;
#pragma unroll
    for (int e = 0; e < 8; ++e) { dst[e] = s.v[e]; dst[8 + e] = q.v[e]; }
  }
  __syncthreads();
  for (int t = threadIdx.x; t < pieces * 16; t += kStatThreads) {
    double acc = 0.0;
    for (int l = 0; l < lanes; ++l) acc += (double)s_part[(size_t)l * pieces * 16 + t];
    const int pc = t >> 4, e = t & 15;
    atomicAdd(out + (e < 8 ? 0 : C) + pc * 8 + (e & 7), acc);
  }
}

// ---- the same reduction with the rows STAGED through shared memory by the copy engine ----------------------------------
// The register version above keeps 4 rows x 2 x 16 B per thread in flight, 64 KB per SM at its 24 % occupancy — about one
// bandwidth-delay product, and ncu showed it at 59-67 % of the DRAM peak with 43 % of the stalls on the loads.  Here a
// producer lane streams row tiles of both operands (dz, y: contiguous [P][C], so a tile is ONE 1-D bulk copy each) into a
// 3-stage ring (up to 192 KB in flight per SM, independent of the register file) and 16 consumer warps read them back
// with conflict-free 16-byte shared loads (thread t reads bytes [16 t, 16 t + 16) of a 4-row-lane slab).
__device__ __forceinline__ uint32_t stg_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void stg_wait(uint64_t* bar, unsigned parity) {
  unsigned ok = 0, spins = 0;
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(stg_u32(bar)), "r"(parity) : "memory");
    if (!ok && ++spins > (1u << 26)) __trap();  // a protocol bug traps instead of hanging the GPU
  }
}
constexpr int kStgConsumers = 512;
constexpr int kStgThreads = kStgConsumers + 32;  // + the producer warp
constexpr int kStgStages = 3;
constexpr int kStgRowsPerLane = 4;

__global__ void __launch_bounds__(kStgThreads, 1)
bn_bwd_reduce_staged_kernel(const __nv_bfloat16* __restrict__ dz, const __nv_bfloat16* __restrict__ y,
                            const float* __restrict__ scale, const float* __restrict__ shift, long long P, int C, int relu,
                            unsigned seed, unsigned thresh, float keep_scale, double* __restrict__ out) {
  extern __shared__ __align__(128) uint8_t stg_smem[];  // [stages][dz tile | y tile]; re-used for the final reduction
  __shared__ __align__(8) uint64_t full[kStgStages], empty[kStgStages];
  const int pieces = C >> 3;
  const int lanes = kStgConsumers / pieces;
  const int R = kStgRowsPerLane * lanes;                 // rows per tile
  const unsigned tile_bytes = (unsigned)R * (unsigned)C * 2u;  // <= 32 KB
  const long long n_tiles = (P + R - 1) / R;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kStgStages; ++s) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(stg_u32(&full[s])));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(stg_u32(&empty[s])), "r"(kStgConsumers / 32));
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (warp == kStgConsumers / 32) {
    if (lane == 0) {
      unsigned i = 0;
      for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x, ++i) {
        const unsigned s = i % kStgStages, use = i / kStgStages;
        if (use > 0) stg_wait(&empty[s], (use - 1) & 1u);
        const long long row0 = t * R;
        const unsigned bytes = (unsigned)(min((long long)R, P - row0) * C * 2);
        uint8_t* dst = stg_smem + (size_t)s * 2 * tile_bytes;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(stg_u32(&full[s])), "r"(2u * bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(stg_u32(dst)),
                     "l"(dz + row0 * C), "r"(bytes), "r"(stg_u32(&full[s])) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                         stg_u32(dst + tile_bytes)), "l"(y + row0 * C), "r"(bytes), "r"(stg_u32(&full[s])) : "memory");
      }
    }
    return;
  }
  const int piece = threadIdx.x % pieces, rl = threadIdx.x / pieces;
  const bool active = rl < lanes;
  F8 sg{}, sq{};
  const F8 a = load_f8(scale + piece * 8), b = load_f8(shift + piece * 8);
  unsigned i = 0;
  for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x, ++i) {
    const unsigned s = i % kStgStages, use = i / kStgStages;
    const long long row0 = t * R;
    const int rows = (int)min((long long)R, P - row0);
    stg_wait(&full[s], use & 1u);
    if (active) {
      const uint4* gt = reinterpret_cast<const uint4*>(stg_smem + (size_t)s * 2 * tile_bytes) + threadIdx.x;
      const uint4* yt = reinterpret_cast<const uint4*>(stg_smem + (size_t)s * 2 * tile_bytes + tile_bytes) + threadIdx.x;
      uint4 gr[kStgRowsPerLane], yr[kStgRowsPerLane];
#pragma unroll
      for (int u = 0; u < kStgRowsPerLane; ++u) {
        if (rl + u * lanes < rows) {
          gr[u] = gt[(size_t)u * lanes * pieces];
          yr[u] = yt[(size_t)u * lanes * pieces];
        }
      }
#pragma unroll
      for (int u = 0; u < kStgRowsPerLane; ++u) {
        const int rr = rl + u * lanes;
        if (rr >= rows) break;
        const F8 v = unpack8(yr[u]);
        const F8 d = unpack8(gr[u]);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          float g = d.v[e];
          if (relu && !(fmaf(v.v[e], a.v[e], b.v[e]) > 0.f)) g = 0.f;
          if (thresh) g = keep_elem(seed, row0 + rr, piece * 8 + e, C, thresh) ? g * keep_scale : 0.f;
          sg.v[e] += g;
          sq.v[e] = fmaf(g, v.v[e], sq.v[e]);
        }
      }
    }
    __syncwarp();
    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(stg_u32(&empty[s])) : "memory");
  }
  // every consumer is done with the ring (and every copy has been waited for): re-use it for the block reduction
  asm volatile("bar.sync 1, %0;" ::"n"(kStgConsumers) : "memory");
  float* s_part = reinterpret_cast<float*>(stg_smem);
  if (active) {
    float* dst = s_part + ((size_t)rl * pieces + piece) * 16;
#pragma unroll
    for (int e = 0; e < 8; ++e) { dst[e] = sg.v[e]; dst[8 + e] = sq.v[e]; }
  }
  asm volatile("bar.sync 1, %0;" ::"n"(kStgConsumers) : "memory");
  for (int t = threadIdx.x; t < pieces * 16; t += kStgConsumers) {
    double acc = 0.0;
    for (int l = 0; l < lanes; ++l) acc += (double)s_part[(size_t)l * pieces * 16 + t];
    const int pc = t >> 4, e = t & 15;
    atomicAdd(out + (e < 8 ? 0 : C) + pc * 8 + (e & 7), acc);
  }
}

// dy = coef * (g - m1 - xhat * m2) = ka * g + kb * y + kc per channel, with ka = coef, kb = -coef * rstd * m2,
// kc = coef * (rstd * m2 * mean - m1) folded by the host wrapper (coef = gamma * rstd, m1 = mean(g), m2 = mean(g * xhat))
template <int UP = kUpDenseOrArg8>
__global__ void __launch_bounds__(256, 2)
bn_bwd_apply_kernel(Upstream up, const __nv_bfloat16* __restrict__ y, const float* __restrict__ scale,
                    const float* __restrict__ shift, const float* __restrict__ ka, const float* __restrict__ kb,
                    const float* __restrict__ kc, long long P, int C, int relu, unsigned seed, unsigned thresh,
                    float keep_scale, __nv_bfloat16* __restrict__ dy) {
  const int pieces = C >> 3;
  const int lanes = 256 / pieces;
  const int piece = threadIdx.x % pieces, rl = threadIdx.x / pieces;
  if (rl >= lanes) return;
  const long long r1 = min(P, ((long long)blockIdx.x + 1) * kEltRows);
  const F8 a = load_f8(scale + piece * 8), b = load_f8(shift + piece * 8), A = load_f8(ka + piece * 8),
           Bc = load_f8(kb + piece * 8), Cc = load_f8(kc + piece * 8);
  for (long long r = (long long)blockIdx.x * kEltRows + rl; r < r1; r += 4LL * lanes) {
    uint4 raw[4];
    UpRaw ur[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long rr = r + (long long)u * lanes;
      if (rr < r1) {
        raw[u] = __ldg(reinterpret_cast<const uint4*>(y + rr * C) + piece);
        ur[u] = upstream_load_k<UP>(up, rr, piece, C);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long rr = r + (long long)u * lanes;
      if (rr >= r1) break;
      const F8 v = unpack8(raw[u]);
      const F8 d = upstream_route(ur[u]);
      F8 o;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        float g = d.v[e];
        if (relu && !(fmaf(v.v[e], a.v[e], b.v[e]) > 0.f)) g = 0.f;
        if (thresh) g = keep_elem(seed, rr, piece * 8 + e, C, thresh) ? g * keep_scale : 0.f;
        o.v[e] = fmaf(A.v[e], g, fmaf(Bc.v[e], v.v[e], Cc.v[e]));
      }
      reinterpret_cast<uint4*>(dy + rr * C)[piece] = pack8(o);
    }
  }
}

// the second pass, rows staged by the copy engine like bn_bwd_reduce_staged_kernel: y always, dz when it is dense (a pooled
// upstream gradient is G x C, K times smaller than y, and stays on the read-only path); dy leaves with 16-byte stores
// (RPL rows per thread and tile, STAGES tiles in flight, CONS consumer threads: 15 consumer warps + the producer warp = 512
// threads get 128 registers each; with 16 + 1 warps ptxas allots 96 and the five per-channel parameter vectors spill)
// DENSE / DROP are compile-time: the pooled pass (G x K rows, no dropout) carries neither the dropout hash nor the dense
// branch, the dense pass not the routing
template <int RPL, int STAGES, int CONS, bool DENSE, bool DROP, int UP = kUpDenseOrArg8>
__global__ void __launch_bounds__(CONS + 32, 1)
bn_bwd_apply_staged_kernel(Upstream up, const __nv_bfloat16* __restrict__ y, const float* __restrict__ scale,
                           const float* __restrict__ shift, const float* __restrict__ ka, const float* __restrict__ kb,
                           const float* __restrict__ kc, long long P, int C, int relu, unsigned seed, unsigned thresh,
                           float keep_scale, __nv_bfloat16* __restrict__ dy) {
  extern __shared__ __align__(128) uint8_t stg_smem[];  // [stages][y tile | dz tile]
  __shared__ __align__(8) uint64_t full[STAGES], empty[STAGES];
  const int pieces = C >> 3;
  const int lanes = CONS / pieces;
  const int R = RPL * lanes;
  const unsigned tile_bytes = (unsigned)R * (unsigned)C * 2u;
  const long long n_tiles = (P + R - 1) / R;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr bool dense = DENSE;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(stg_u32(&full[s])));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(stg_u32(&empty[s])), "r"(CONS / 32));
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (warp == CONS / 32) {
    if (lane == 0) {
      unsigned i = 0;
      for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x, ++i) {
        const unsigned s = i % STAGES, use = i / STAGES;
        if (use > 0) stg_wait(&empty[s], (use - 1) & 1u);
        const long long row0 = t * R;
        const unsigned bytes = (unsigned)(min((long long)R, P - row0) * C * 2);
        uint8_t* dst = stg_smem + (size_t)s * 2 * tile_bytes;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(stg_u32(&full[s])), "r"(dense ? 2u * bytes : bytes)
                     : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(stg_u32(dst)),
                     "l"(y + row0 * C), "r"(bytes), "r"(stg_u32(&full[s])) : "memory");
        if (dense)
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                           stg_u32(dst + tile_bytes)), "l"(up.dz + row0 * C), "r"(bytes), "r"(stg_u32(&full[s])) : "memory");
      }
    }
    return;
  }
  const int piece = threadIdx.x % pieces, rl = threadIdx.x / pieces;
  const bool active = rl < lanes;
  const F8 a = load_f8(scale + piece * 8), b = load_f8(shift + piece * 8), A = load_f8(ka + piece * 8),
           Bc = load_f8(kb + piece * 8), Cc = load_f8(kc + piece * 8);
  unsigned i = 0;
  for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x, ++i) {
    const unsigned s = i % STAGES, use = i / STAGES;
    const long long row0 = t * R;
    const int rows = (int)min((long long)R, P - row0);
    UpRaw ur[RPL];
    if (active && !dense) {  // (before the wait: these come from L2)
#pragma unroll
      for (int u = 0; u < RPL; ++u)
        if (rl + u * lanes < rows) ur[u] = upstream_load_k<UP>(up, row0 + rl + u * lanes, piece, C);
    }
    stg_wait(&full[s], use & 1u);
    if (active) {
      const uint4* yt = reinterpret_cast<const uint4*>(stg_smem + (size_t)s * 2 * tile_bytes) + threadIdx.x;
      const uint4* gt = reinterpret_cast<const uint4*>(stg_smem + (size_t)s * 2 * tile_bytes + tile_bytes) + threadIdx.x;
      uint4 yr[RPL];
#pragma unroll
      for (int u = 0; u < RPL; ++u) {
        if (rl + u * lanes < rows) {
          yr[u] = yt[(size_t)u * lanes * pieces];
          if (dense) { ur[u].d = gt[(size_t)u * lanes * pieces]; ur[u].a = make_uint2(0u, 0u); ur[u].k = -1; }
        }
      }
#pragma unroll
      for (int u = 0; u < RPL; ++u) {
        const int rr = rl + u * lanes;
        if (rr >= rows) break;
        const F8 v = unpack8(yr[u]);
        const F8 d = upstream_route(ur[u]);
        F8 o;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          float g = d.v[e];
          if (relu && !(fmaf(v.v[e], a.v[e], b.v[e]) > 0.f)) g = 0.f;
          if (DROP) g = keep_elem(seed, row0 + rr, piece * 8 + e, C, thresh) ? g * keep_scale : 0.f;
          o.v[e] = fmaf(A.v[e], g, fmaf(Bc.v[e], v.v[e], Cc.v[e]));
        }
        reinterpret_cast<uint4*>(dy + (row0 + rr) * C)[piece] = pack8(o);
      }
    }
    __syncwarp();
    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(stg_u32(&empty[s])) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------- grouping rows
// X0 row (b, m, k) = [feat[b*N + j][0..Cf) | dx dy dz 0 0 0 0 0],  j = nbr[b][m][k];  width = Cf + 8
__global__ void __launch_bounds__(256)
group_rows_kernel(const __nv_bfloat16* __restrict__ feat, const float* __restrict__ xyz, const float* __restrict__ ctr,
                  const int* __restrict__ nbr, int N, int M, int K, int Cf, long long rows, __nv_bfloat16* __restrict__ out) {
  const int pieces = (Cf >> 3) + 1;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * pieces) return;
  const long long row = i / pieces;
  const int piece = (int)(i - row * pieces);
  const long long per_b = (long long)M * K;
  const int b = (int)(row / per_b);
  const int m = (int)((row - (long long)b * per_b) / K);
  const int j = __ldg(nbr + row);
  uint4 v;
  if (piece < (Cf >> 3)) {
    v = __ldg(reinterpret_cast<const uint4*>(feat + ((long long)b * N + j) * Cf) + piece);
  } else {
    const float* X = xyz + (long long)b * 3 * N;
    const float* Cn = ctr + (long long)b * 3 * M;
    F8 r{};
    r.v[0] = __fsub_rn(__ldg(X + j), __ldg(Cn + m));
    r.v[1] = __fsub_rn(__ldg(X + N + j), __ldg(Cn + M + m));
    r.v[2] = __fsub_rn(__ldg(X + 2 * N + j), __ldg(Cn + 2 * M + m));
    v = pack8(r);
  }
  reinterpret_cast<uint4*>(out + row * (long long)(Cf + 8))[piece] = v;
}

__device__ __forceinline__ void atomic_add_f8(float* dst, const F8& v) {
  atomicAdd(reinterpret_cast<float4*>(dst), make_float4(v.v[0], v.v[1], v.v[2], v.v[3]));
  atomicAdd(reinterpret_cast<float4*>(dst) + 1, make_float4(v.v[4], v.v[5], v.v[6], v.v[7]));
}

// dfeat[b*N + nbr[row]][c] += dx[row][c]   for c < Cf;  dx rows are ld wide
__global__ void __launch_bounds__(256)
group_rows_bwd_kernel(const __nv_bfloat16* __restrict__ dx, long long ld, const int* __restrict__ nbr, int N, long long per_b,
                      int Cf, long long rows, float* __restrict__ dfeat) {
  const int pieces = Cf >> 3;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * pieces) return;
  const long long row = i / pieces;
  const int piece = (int)(i - row * pieces);
  const int b = (int)(row / per_b);
  const int j = __ldg(nbr + row);
  const F8 v = unpack8(__ldg(reinterpret_cast<const uint4*>(dx + row * ld) + piece));
  atomic_add_f8(dfeat + ((long long)b * N + j) * Cf + piece * 8, v);
}

// dsparse[b*Nk + idx[row][k]][c] += w[row][k] * dx[row][c]   for c < C2
__global__ void __launch_bounds__(256)
interp_rows_bwd_kernel(const __nv_bfloat16* __restrict__ dx, long long ld, const int* __restrict__ index,
                       const float* __restrict__ weight, int Nk, int Nq, int C2, long long rows, float* __restrict__ dsparse) {
  const int pieces = C2 >> 3;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * pieces) return;
  const long long row = i / pieces;
  const int piece = (int)(i - row * pieces);
  const long long b = row / Nq;
  const F8 v = unpack8(__ldg(reinterpret_cast<const uint4*>(dx + row * ld) + piece));
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int j = __ldg(index + row * 3 + k);
    const float w = __ldg(weight + row * 3 + k);
    F8 t;
#pragma unroll
    for (int e = 0; e < 8; ++e) t.v[e] = v.v[e] * w;
    atomic_add_f8(dsparse + (b * Nk + j) * C2 + piece * 8, t);
  }
}

// ---- the same gradient as a GATHER over the inverse of the 3-NN index -------------------------------------------------
// The scatter above issues 3 x rows x C2 fp32 atomic adds (1.26 G element-adds for 819 200 rows of 512 channels: 1.6 ms).
// The 3-NN index is geometry (fixed for the step), so it is inverted once — count, exclusive scan (caller), fill — into
// per-sparse-point lists of entries e = row * 3 + k, and every sparse row then SUMS its own list: dx rows are read three
// times in all, the result is written once (fp32 or bf16), no atomics on the gradient.
__global__ void __launch_bounds__(256)
interp_inverse_count_kernel(const int* __restrict__ index, int Nk, long long per_b, long long entries, int* __restrict__ count) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= entries) return;
  const long long b = e / per_b;  // per_b = Nq * 3
  atomicAdd(count + b * Nk + __ldg(index + e), 1);
}
__global__ void __launch_bounds__(256)
interp_inverse_fill_kernel(const int* __restrict__ index, int Nk, long long per_b, long long entries, int* __restrict__ cursor,
                           int* __restrict__ list) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= entries) return;
  const long long b = e / per_b;
  list[atomicAdd(cursor + b * Nk + __ldg(index + e), 1)] = (int)e;
}
// thread = (16-byte piece, target-row lane); out row j (+)= sum over its list of weight[e] * dx[e / DIV]
// (DIV = 3, weights: interpolation;  DIV = 1, no weights: grouping — entry e IS the gathered row (b, m, k))
template <int DIV>
__global__ void __launch_bounds__(256)
rows_bwd_gather_kernel(const __nv_bfloat16* __restrict__ dx, long long ld, const int* __restrict__ list,
                       const int* __restrict__ end, const int* __restrict__ count, const float* __restrict__ weight,
                       long long sparse_rows, int C2, int accumulate, float* __restrict__ out_f32,
                       __nv_bfloat16* __restrict__ out_bf16) {
  const int pieces = C2 >> 3;
  const int lanes = 256 / pieces;
  const int piece = threadIdx.x % pieces, rl = threadIdx.x / pieces;
  const long long j = (long long)blockIdx.x * lanes + rl;
  if (rl >= lanes || j >= sparse_rows) return;
  const int n = __ldg(count + j);
  const int* src = list + (__ldg(end + j) - n);  // end = inclusive scan of count
  F8 acc{};
  int t = 0;
  for (; t + 1 < n; t += 2) {  // two entries in flight
    const int e0 = __ldg(src + t), e1 = __ldg(src + t + 1);
    const float w0 = weight ? __ldg(weight + e0) : 1.f, w1 = weight ? __ldg(weight + e1) : 1.f;
    const F8 v0 = unpack8(__ldg(reinterpret_cast<const uint4*>(dx + (long long)(e0 / DIV) * ld) + piece));
    const F8 v1 = unpack8(__ldg(reinterpret_cast<const uint4*>(dx + (long long)(e1 / DIV) * ld) + piece));
#pragma unroll
    for (int c = 0; c < 8; ++c) acc.v[c] = fmaf(w0, v0.v[c], fmaf(w1, v1.v[c], acc.v[c]));
  }
  if (t < n) {
    const int e0 = __ldg(src + t);
    const float w0 = weight ? __ldg(weight + e0) : 1.f;
    const F8 v0 = unpack8(__ldg(reinterpret_cast<const uint4*>(dx + (long long)(e0 / DIV) * ld) + piece));
#pragma unroll
    for (int c = 0; c < 8; ++c) acc.v[c] = fmaf(w0, v0.v[c], acc.v[c]);
  }
  if (out_f32) {
    float4* o = reinterpret_cast<float4*>(out_f32 + j * C2 + piece * 8);
    if (accumulate) {  // (the row is this thread's alone: a plain read-modify-write)
      const float4 p0 = o[0], p1 = o[1];
      acc.v[0] += p0.x; acc.v[1] += p0.y; acc.v[2] += p0.z; acc.v[3] += p0.w;
      acc.v[4] += p1.x; acc.v[5] += p1.y; acc.v[6] += p1.z; acc.v[7] += p1.w;
    }
    o[0] = make_float4(acc.v[0], acc.v[1], acc.v[2], acc.v[3]);
    o[1] = make_float4(acc.v[4], acc.v[5], acc.v[6], acc.v[7]);
  }
  if (out_bf16) reinterpret_cast<uint4*>(out_bf16 + j * C2)[piece] = pack8(acc);
}

// g = dz where relu'(y * scale + shift) else 0, rows [P][C] — the pooled gradient of a max-pooled block masked ONCE on its
// G rows (y = the pre-activation at the arg-max, kept by bn_act_maxpool), so that the two passes over the G x K rows
// run without the ReLU test
__global__ void __launch_bounds__(256)
relu_mask_rows_kernel(const __nv_bfloat16* __restrict__ dz, const __nv_bfloat16* __restrict__ y, const float* __restrict__ scale,
                      const float* __restrict__ shift, long long P, int C, __nv_bfloat16* __restrict__ out) {
  const int pieces = C >> 3;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P * pieces) return;
  const int piece = (int)(i % pieces);
  const F8 a = load_f8(scale + piece * 8), b = load_f8(shift + piece * 8);
  const F8 v = unpack8(__ldg(reinterpret_cast<const uint4*>(y) + i));
  F8 d = unpack8(__ldg(reinterpret_cast<const uint4*>(dz) + i));
#pragma unroll
  for (int e = 0; e < 8; ++e)
    if (!(fmaf(v.v[e], a.v[e], b.v[e]) > 0.f)) d.v[e] = 0.f;
  reinterpret_cast<uint4*>(out)[i] = pack8(d);
}

// fp32 [rows][C] -> bf16 (gradient buffers accumulated with atomics -> the next kernel's bf16 operand)
__global__ void __launch_bounds__(256)
f32_to_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, long long n8) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n8) return;
  reinterpret_cast<uint4*>(y)[i] = pack8(load_f8(x + i * 8));
}

// BatchNorm (training) per-channel algebra in one launch instead of a dozen tiny ones.
// forward: sums -> mean, rstd, scale = gamma * rstd, shift = beta - mean * scale; running statistics updated like
// torch.nn.BatchNorm (momentum, unbiased variance).  out4c = [mean | rstd | scale | shift].
__global__ void bn_finalize_kernel(const double* __restrict__ sums, long long P, int C, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float eps, float momentum, float* __restrict__ run_mean,
                                   float* __restrict__ run_var, float* __restrict__ out4c) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double mean = sums[c] / (double)P;
  double var = sums[C + c] / (double)P - mean * mean;
  var = var > 0.0 ? var : 0.0;
  const float rstd = rsqrtf((float)var + eps);
  const float scale = gamma[c] * rstd;
  out4c[c] = (float)mean;
  out4c[C + c] = rstd;
  out4c[2 * C + c] = scale;
  out4c[3 * C + c] = beta[c] - (float)mean * scale;
  if (run_mean) {
    run_mean[c] = (1.f - momentum) * run_mean[c] + momentum * (float)mean;
    run_var[c] = (1.f - momentum) * run_var[c] + momentum * (float)(var * ((double)P / (double)(P > 1 ? P - 1 : 1)));
  }
}
// backward: sums = [sum g | sum g * y] (bn_bwd_reduce) -> dgamma += sum g xhat, dbeta += sum g, and the folded coefficients of
// dy = ka * g + kb * y + kc.  out3c = [ka | kb | kc].
__global__ void bn_bwd_finalize_kernel(const double* __restrict__ sums, long long P, int C, const float* __restrict__ gamma,
                                       const float* __restrict__ mean_rstd, float* __restrict__ dgamma,
                                       float* __restrict__ dbeta, float* __restrict__ out3c) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float mean = mean_rstd[c], rstd = mean_rstd[C + c];
  const double sgx_d = (double)rstd * (sums[C + c] - (double)mean * sums[c]);  // sum g * xhat from [sum g | sum g * y]
  const float sg = (float)sums[c], sgx = (float)sgx_d;
  const float ka = gamma[c] * rstd;
  const float m1 = (float)(sums[c] / (double)P), m2 = (float)(sgx_d / (double)P);
  out3c[c] = ka;
  out3c[C + c] = -ka * rstd * m2;
  out3c[2 * C + c] = ka * (rstd * m2 * mean - m1);
  dgamma[c] += sgx;
  dbeta[c] += sg;
}

// ---------------------------------------------------------------------------------------------- head logits
// The final biased 1x1 conv of a head (reference PointNet2_tcls.py:84-95: nn.Conv1d(C, k, 1), k <= 16) straight from
// the bf16 rows into the reference's fp32 channel-first layout (B, k, n_points), and its input gradient.  One thread
// per row; the k x C weight matrix lives in shared memory (broadcast reads).
constexpr int kMaxLogits = 16;

// Tiles of kHeadRows rows.  (First versions: one thread per row walking its 256-byte row piece by piece — every warp load
// and store touched 32 different rows, 0.11 / 0.15 ms per head for 0.03 ms of traffic.)
constexpr int kHeadRows = 128;

// forward: the h tile is staged in shared memory with coalesced 16-byte loads (row stride 2 C + 16 bytes: conflict-free
// 16-byte reads by row); thread = (row, half of the k outputs); the stores of one output j are consecutive in n
__global__ void __launch_bounds__(256)
head_logits_fwd_kernel(const __nv_bfloat16* __restrict__ h, const float* __restrict__ w, const float* __restrict__ bias,
                       float* __restrict__ out, int P, int C, int k, int n_points) {
  extern __shared__ __align__(16) uint8_t s_raw[];
  float* s_w = reinterpret_cast<float*>(s_raw);                 // [k][C]
  uint8_t* s_h = s_raw + sizeof(float) * (size_t)k * C;         // [kHeadRows][2 C + 16]
  const int pieces = C >> 3, stride = 2 * C + 16;
  for (int i = threadIdx.x; i < k * C; i += 256) s_w[i] = w[i];
  const int row0 = blockIdx.x * kHeadRows;
  const int rows = min(kHeadRows, P - row0);
  for (int i = threadIdx.x; i < rows * pieces; i += 256) {
    const int r = i / pieces, pc = i - r * pieces;
    *reinterpret_cast<uint4*>(s_h + (size_t)r * stride + pc * 16) = __ldg(reinterpret_cast<const uint4*>(h + (size_t)(row0 + r) * C) + pc);
  }
  __syncthreads();
  const int r = threadIdx.x & (kHeadRows - 1), half = threadIdx.x >> 7;  // outputs j = half, half + 2, ...
  if (r >= rows) return;
  float acc[kMaxLogits / 2];
#pragma unroll
  for (int q = 0; q < kMaxLogits / 2; ++q) acc[q] = (2 * q + half) < k ? __ldg(bias + 2 * q + half) : 0.f;
  for (int pc = 0; pc < pieces; ++pc) {
    const F8 v = unpack8(*reinterpret_cast<const uint4*>(s_h + (size_t)r * stride + pc * 16));
#pragma unroll
    for (int q = 0; q < kMaxLogits / 2; ++q) {
      const int j = 2 * q + half;
      if (j < k) {
        const float4* wj = reinterpret_cast<const float4*>(s_w + j * C + pc * 8);  // warp-uniform: broadcast
        const float4 w0 = wj[0], w1 = wj[1];
        acc[q] = fmaf(v.v[0], w0.x, fmaf(v.v[1], w0.y, fmaf(v.v[2], w0.z, fmaf(v.v[3], w0.w, acc[q]))));
        acc[q] = fmaf(v.v[4], w1.x, fmaf(v.v[5], w1.y, fmaf(v.v[6], w1.z, fmaf(v.v[7], w1.w, acc[q]))));
      }
    }
  }
  const int row = row0 + r;
  const int b = row / n_points, n = row - b * n_points;
  float* o = out + ((size_t)b * k) * n_points + n;
#pragma unroll
  for (int q = 0; q < kMaxLogits / 2; ++q)
    if (2 * q + half < k) o[(size_t)(2 * q + half) * n_points] = acc[q];
}

// dh[row][c] = sum_j dlogits[b][j][n] * w[j][c]   (bf16 rows out): the tile's k x rows gradients are staged in shared
// memory (coalesced), thread = (16-byte piece of the row, row lane) keeps its k x 8 weights in registers and stores
// 16-byte pieces next to its neighbours'
template <int KT>
__global__ void __launch_bounds__(256)
head_logits_bwd_kernel(const float* __restrict__ dl, const float* __restrict__ w, __nv_bfloat16* __restrict__ dh, int P,
                       int C, int k, int n_points) {
  __shared__ float s_g[KT][kHeadRows];
  const int pieces = C >> 3, lanes = 256 / pieces;
  const int row0 = blockIdx.x * kHeadRows;
  const int rows = min(kHeadRows, P - row0);
  for (int i = threadIdx.x; i < k * kHeadRows; i += 256) {
    const int j = i / kHeadRows, r = i - j * kHeadRows;
    float g = 0.f;
    if (r < rows) {
      const int row = row0 + r;
      const int b = row / n_points, n = row - b * n_points;
      g = __ldg(dl + ((size_t)b * k + j) * n_points + n);
    }
    s_g[j][r] = g;
  }
  const int piece = threadIdx.x % pieces, rl = threadIdx.x / pieces;
  float wr[KT][8];
#pragma unroll
  for (int j = 0; j < KT; ++j) {
    if (j < k && rl < lanes) {
      const F8 t = load_f8(w + (size_t)j * C + piece * 8);
#pragma unroll
      for (int e = 0; e < 8; ++e) wr[j][e] = t.v[e];
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) wr[j][e] = 0.f;
    }
  }
  __syncthreads();
  if (rl >= lanes) return;
  for (int r = rl; r < rows; r += lanes) {
    F8 o{};
#pragma unroll
    for (int j = 0; j < KT; ++j) {
      const float g = s_g[j][r];  // (zero for j >= k)
#pragma unroll
      for (int e = 0; e < 8; ++e) o.v[e] = fmaf(g, wr[j][e], o.v[e]);
    }
    reinterpret_cast<uint4*>(dh + (size_t)(row0 + r) * C)[piece] = pack8(o);
  }
}

// out = a + b (+ c) (+ d), bf16 rows summed in fp32, one rounding: the four heads' gradients of the per-point features
__global__ void __launch_bounds__(256)
sum_bf16_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, const uint4* __restrict__ c, const uint4* __restrict__ d,
                uint4* __restrict__ out, long long n8) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n8) return;
  const uint4 ra = __ldg(a + i), rb = __ldg(b + i);
  const uint4 rc = c ? __ldg(c + i) : make_uint4(0u, 0u, 0u, 0u), rd = d ? __ldg(d + i) : make_uint4(0u, 0u, 0u, 0u);
  const F8 fa = unpack8(ra), fb = unpack8(rb), fc = unpack8(rc), fd = unpack8(rd);
  F8 o;
#pragma unroll
  for (int e = 0; e < 8; ++e) o.v[e] = (fa.v[e] + fb.v[e]) + (fc.v[e] + fd.v[e]);
  out[i] = pack8(o);
}

// dw[j][c] += sum_row dlogits[b][j][n] * h[row][c],  dbias[j] += sum_row dlogits[b][j][n]   (fp32 atomics, k <= KT)
// thread = (16-byte piece of h, row lane); a block walks kDwTiles tiles of kHeadRows rows — the tile's k x rows gradients
// staged in shared memory (coalesced loads, broadcast reads), two rows of h in flight per thread — and reduces over its
// row lanes in shared memory at the end.  (First version: k scalar global loads per row and thread, 152 registers, one
// block per SM: 0.22 ms per head for 0.03 ms of traffic.)
constexpr int kDwTiles = 4;
template <int KT>
__global__ void __launch_bounds__(256, KT > 9 ? 1 : 2)
head_logits_dw_kernel(const float* __restrict__ dl, const __nv_bfloat16* __restrict__ h, float* __restrict__ dw,
                      float* __restrict__ dbias, int P, int C, int k, int n_points) {
  extern __shared__ float s_red[];  // [lanes][C]
  __shared__ float s_g[KT][kHeadRows];
  const int pieces = C >> 3;
  const int lanes = 256 / pieces;
  const int piece = threadIdx.x % pieces, rl = threadIdx.x / pieces;
  float acc[KT][8];
  float accb = 0.f;  // thread j < k: the bias gradient of output j
#pragma unroll
  for (int j = 0; j < KT; ++j) {
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[j][e] = 0.f;
  }
  for (int tile = 0; tile < kDwTiles; ++tile) {
    const int row0 = (blockIdx.x * kDwTiles + tile) * kHeadRows;
    if (row0 >= P) break;  // (block-uniform)
    const int rows = min(kHeadRows, P - row0);
    __syncthreads();  // the previous tile's gradients have been consumed
    for (int i = threadIdx.x; i < k * kHeadRows; i += 256) {
      const int j = i / kHeadRows, r = i - j * kHeadRows;
      float g = 0.f;
      if (r < rows) {
        const int row = row0 + r;
        const int b = row / n_points, n = row - b * n_points;
        g = __ldg(dl + ((size_t)b * k + j) * n_points + n);
      }
      s_g[j][r] = g;
    }
    __syncthreads();
    if (threadIdx.x < k) {
      float t = 0.f;
      for (int r = 0; r < rows; ++r) t += s_g[threadIdx.x][r];
      accb += t;
    }
    if (rl < lanes) {
      for (int r = rl; r < rows; r += 2 * lanes) {
        const int r1 = r + lanes;
        const bool two = r1 < rows;
        const uint4 raw0 = __ldg(reinterpret_cast<const uint4*>(h + (size_t)(row0 + r) * C) + piece);
        const uint4 raw1 = two ? __ldg(reinterpret_cast<const uint4*>(h + (size_t)(row0 + r1) * C) + piece) : make_uint4(0u, 0u, 0u, 0u);
        const F8 v0 = unpack8(raw0), v1 = unpack8(raw1);
#pragma unroll
        for (int j = 0; j < KT; ++j) {
          const float g0 = s_g[j][r], g1 = two ? s_g[j][r1] : 0.f;  // (rows j >= k hold stale or zero values: never reduced)
#pragma unroll
          for (int e = 0; e < 8; ++e) acc[j][e] = fmaf(g0, v0.v[e], fmaf(g1, v1.v[e], acc[j][e]));
        }
      }
    }
  }
  if (threadIdx.x < k) atomicAdd(dbias + threadIdx.x, accb);
#pragma unroll
  for (int j = 0; j < KT; ++j) {
    if (j < k) {  // (k is block-uniform: the barriers below are reached by every thread)
      __syncthreads();
      if (rl < lanes) {
        float* dst = s_red + (size_t)rl * C + piece * 8;
#pragma unroll
        for (int e = 0; e < 8; ++e) dst[e] = acc[j][e];
      }
      __syncthreads();
      for (int c = threadIdx.x; c < C; c += 256) {
        float t = 0.f;
        for (int l = 0; l < lanes; ++l) t += s_red[(size_t)l * C + c];
        atomicAdd(dw + (size_t)j * C + c, t);
      }
    }
  }
}

static unsigned grid_for(long long work, int threads) { return (unsigned)((work + threads - 1) / threads); }

}  // namespace trn
}  // namespace s4g

using namespace s4g::trn;
typedef __nv_bfloat16 bf16;

#define TRN_CHECK_C(C) S4G_CHECK_ARG((C) > 0 && (C) % 8 == 0 && (C) <= 2048, "train_ops: channels must be a multiple of 8, <= 2048")

extern "C" int s4g_train_colstats_bf16(const void* y, long long ld, long long P, int C, double* sums2c, void* stream) {
  S4G_CHECK_ARG(y && sums2c && P > 0 && ld >= C && ld % 8 == 0, "train_colstats: bad arguments");
  TRN_CHECK_C(C);
  cudaStream_t s = (cudaStream_t)stream;
  S4G_CUDA(cudaMemsetAsync(sums2c, 0, sizeof(double) * 2 * C, s));
  const int pieces = C >> 3, lanes = kStatThreads / pieces;
  S4G_CHECK_ARG(lanes >= 1, "train_colstats: too many channels");
  const size_t smem = (size_t)lanes * pieces * 16 * sizeof(float);
  colstats_kernel<<<grid_for(P, kStatRows), kStatThreads, smem, s>>>(reinterpret_cast<const bf16*>(y), ld, P, C, sums2c);
  S4G_LAUNCH_CHECK("train_colstats");
  return S4G_OK;
}

extern "C" int s4g_train_bn_act_bf16(const void* y, const float* scale, const float* shift, void* z, long long P, int C,
                                     int relu, unsigned seed, float drop_p, void* stream) {
  S4G_CHECK_ARG(y && scale && shift && z && P > 0 && drop_p >= 0.f && drop_p < 1.f, "train_bn_act: bad arguments");
  TRN_CHECK_C(C);
  const unsigned thresh = drop_p > 0.f ? (unsigned)((double)drop_p * 4294967296.0) : 0u;
  bn_act_kernel<<<grid_for(P, kEltRows), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const bf16*>(y), scale, shift, reinterpret_cast<bf16*>(z), P, C, relu, seed, thresh, 1.f / (1.f - drop_p));
  S4G_LAUNCH_CHECK("train_bn_act");
  return S4G_OK;
}

extern "C" int s4g_train_bn_act_maxpool_bf16(const void* y, const float* scale, const float* shift, void* out, uint8_t* arg,
                                             void* ymax, long long G, int K, int C, int relu, void* stream) {
  S4G_CHECK_ARG(y && scale && shift && out && arg && G > 0 && K > 0 && K <= 255, "train_bn_act_maxpool: bad arguments");
  TRN_CHECK_C(C);
  bn_act_maxpool_kernel<<<grid_for(G * (C >> 3), 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const bf16*>(y), scale, shift, reinterpret_cast<bf16*>(out), arg, reinterpret_cast<bf16*>(ymax), G, K, C,
      relu);
  S4G_LAUNCH_CHECK("train_bn_act_maxpool");
  return S4G_OK;
}

// upstream gradient: dz [P][C] when K == 0; pooled dz [P/K][C] + arg-max [P/K][C] when K > 0 (uint8 arg, or int32 arg32)
static int bn_bwd_reduce(const Upstream& up, const void* y, const float* scale, const float* shift, long long P, int C,
                         int relu, unsigned seed, float drop_p, double* sums2c, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  S4G_CUDA(cudaMemsetAsync(sums2c, 0, sizeof(double) * 2 * C, s));
  const int pieces = C >> 3, lanes = kStatThreads / pieces;
  S4G_CHECK_ARG(lanes >= 1, "train_bn_bwd_reduce: too many channels");
  const unsigned thresh = drop_p > 0.f ? (unsigned)((double)drop_p * 4294967296.0) : 0u;
  const void* dz = up.dz;
  const int K = up.K;
  // S4G_BWD_REDUCE_VARIANT (A/B measurements): 0 (default) = rows staged by the copy engine for dense upstream gradients,
  // 1 = registers, 2 rows in flight x 3 blocks per SM, 2 = registers, 4 x 2
  static int variant = -1;
  if (variant < 0) { const char* e = getenv("S4G_BWD_REDUCE_VARIANT"); variant = e ? atoi(e) : 0; }
  const size_t sm = (size_t)lanes * pieces * 16 * sizeof(float);
  if (up.arg32) {
    bn_bwd_reduce_kernel<4, 2, kUpArg32><<<grid_for(P, kStatRows), kStatThreads, sm, s>>>(
        up, reinterpret_cast<const bf16*>(y), scale, shift, P, C, relu, seed, thresh, 1.f / (1.f - drop_p), sums2c);
  } else if (variant == 0 && K == 0 && C <= 2048 && (((uintptr_t)dz | (uintptr_t)y) & 15) == 0) {
    const int lanes_s = kStgConsumers / pieces;
    const int R = kStgRowsPerLane * lanes_s;
    const size_t tile_bytes = (size_t)R * C * 2;
    const size_t smem = kStgStages * 2 * tile_bytes;  // (>= the 32 KB the final reduction needs)
    static bool attr[64] = {};
    if (s4g::first_use_on_device(attr)) {
      S4G_CUDA(cudaFuncSetAttribute(bn_bwd_reduce_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    }
    const long long n_tiles = (P + R - 1) / R;
    const int sms = s4g::num_sms();
    const unsigned grid = (unsigned)(n_tiles < sms ? n_tiles : sms);
    bn_bwd_reduce_staged_kernel<<<grid, kStgThreads, smem, s>>>(reinterpret_cast<const bf16*>(dz), reinterpret_cast<const bf16*>(y),
                                                                scale, shift, P, C, relu, seed, thresh, 1.f / (1.f - drop_p),
                                                                sums2c);
  } else if (variant == 1)
    bn_bwd_reduce_kernel<2, 3><<<grid_for(P, kStatRows), kStatThreads, sm, s>>>(
        up, reinterpret_cast<const bf16*>(y), scale, shift, P, C, relu, seed, thresh, 1.f / (1.f - drop_p), sums2c);
  else
    bn_bwd_reduce_kernel<4, 2><<<grid_for(P, kStatRows), kStatThreads, sm, s>>>(
        up, reinterpret_cast<const bf16*>(y), scale, shift, P, C, relu, seed, thresh, 1.f / (1.f - drop_p), sums2c);
  S4G_LAUNCH_CHECK("train_bn_bwd_reduce");
  return S4G_OK;
}

extern "C" int s4g_train_bn_bwd_reduce_bf16(const void* dz, const uint8_t* arg, int K, const void* y, const float* scale,
                                            const float* shift, long long P, int C, int relu, unsigned seed, float drop_p,
                                            double* sums2c, void* stream) {
  S4G_CHECK_ARG(dz && y && scale && shift && sums2c && P > 0 && (K == 0 || (arg && P % K == 0)),
                "train_bn_bwd_reduce: bad arguments");
  TRN_CHECK_C(C);
  return bn_bwd_reduce(make_upstream(dz, arg, K), y, scale, shift, P, C, relu, seed, drop_p, sums2c, stream);
}

extern "C" int s4g_train_bn_bwd_reduce_seg_bf16(const void* dz, const int* arg, long long N, const void* y, const float* scale,
                                                const float* shift, long long P, int C, int relu, double* sums2c,
                                                void* stream) {
  S4G_CHECK_ARG(dz && arg && y && scale && shift && sums2c && N > 0 && P > 0 && P % N == 0 && P < (1ll << 31),
                "train_bn_bwd_reduce_seg: bad arguments");
  TRN_CHECK_C(C);
  return bn_bwd_reduce(make_upstream(dz, nullptr, (int)N, arg), y, scale, shift, P, C, relu, 0u, 0.f, sums2c, stream);
}

static int bn_bwd_apply(const Upstream& up, const void* y, const float* scale, const float* shift, const float* ka,
                        const float* kb, const float* kc, long long P, int C, int relu, unsigned seed, float drop_p, void* dy,
                        void* stream) {
  const unsigned thresh = drop_p > 0.f ? (unsigned)((double)drop_p * 4294967296.0) : 0u;
  const int K = up.K;
  static int variant = -1;  // S4G_BWD_APPLY_VARIANT (A/B measurements): 0 (default) = rows staged by the copy engine, 1 = registers
  if (variant < 0) { const char* e = getenv("S4G_BWD_APPLY_VARIANT"); variant = e ? atoi(e) : 0; }
  if (variant == 0 && (((uintptr_t)up.dz | (uintptr_t)y | (uintptr_t)dy) & 15) == 0) {
    constexpr int kRpl = 4, kStages = 3, kCons = 480;
    const int pieces = C >> 3, lanes_s = kCons / pieces;
    const int R = kRpl * lanes_s;
    const size_t smem = (size_t)kStages * 2 * R * C * 2;
    static bool attr[64] = {};
    if (s4g::first_use_on_device(attr)) {
      S4G_CUDA(cudaFuncSetAttribute(bn_bwd_apply_staged_kernel<kRpl, kStages, kCons, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      S4G_CUDA(cudaFuncSetAttribute(bn_bwd_apply_staged_kernel<kRpl, kStages, kCons, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      S4G_CUDA(cudaFuncSetAttribute(bn_bwd_apply_staged_kernel<kRpl, kStages, kCons, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      S4G_CUDA(cudaFuncSetAttribute(bn_bwd_apply_staged_kernel<kRpl, kStages, kCons, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      S4G_CUDA(cudaFuncSetAttribute(bn_bwd_apply_staged_kernel<kRpl, kStages, kCons, false, false, kUpArg32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    }
    const long long n_tiles = (P + R - 1) / R;
    const int sms = s4g::num_sms();
    const unsigned grid = (unsigned)(n_tiles < sms ? n_tiles : sms);
    cudaStream_t st = (cudaStream_t)stream;
    const float ks = 1.f / (1.f - drop_p);
#define S4G_APPLY_GO(DENSE_, DROP_, ...)                                                                                   \
  bn_bwd_apply_staged_kernel<kRpl, kStages, kCons, DENSE_, DROP_, ##__VA_ARGS__><<<grid, kCons + 32, smem, st>>>(           \
      up, reinterpret_cast<const bf16*>(y), scale, shift, ka, kb, kc, P, C, relu, seed, thresh, ks, reinterpret_cast<bf16*>(dy))
    if (up.arg32) S4G_APPLY_GO(false, false, kUpArg32);  // (a pooled block has no dropout)
    else if (K == 0) { if (thresh) S4G_APPLY_GO(true, true); else S4G_APPLY_GO(true, false); }
    else { if (thresh) S4G_APPLY_GO(false, true); else S4G_APPLY_GO(false, false); }
#undef S4G_APPLY_GO
  } else if (up.arg32) {
    bn_bwd_apply_kernel<kUpArg32><<<grid_for(P, kEltRows), 256, 0, (cudaStream_t)stream>>>(
        up, reinterpret_cast<const bf16*>(y), scale, shift, ka, kb, kc, P, C, relu, seed, thresh, 1.f / (1.f - drop_p),
        reinterpret_cast<bf16*>(dy));
  } else {
    bn_bwd_apply_kernel<><<<grid_for(P, kEltRows), 256, 0, (cudaStream_t)stream>>>(
        up, reinterpret_cast<const bf16*>(y), scale, shift, ka, kb, kc, P, C, relu, seed, thresh, 1.f / (1.f - drop_p),
        reinterpret_cast<bf16*>(dy));
  }
  S4G_LAUNCH_CHECK("train_bn_bwd_apply");
  return S4G_OK;
}

extern "C" int s4g_train_bn_bwd_apply_bf16(const void* dz, const uint8_t* arg, int K, const void* y, const float* scale,
                                           const float* shift, const float* ka, const float* kb, const float* kc,
                                           long long P, int C, int relu, unsigned seed, float drop_p, void* dy, void* stream) {
  S4G_CHECK_ARG(dz && y && scale && shift && ka && kb && kc && dy && P > 0 && (K == 0 || (arg && P % K == 0)),
                "train_bn_bwd_apply: bad arguments");
  TRN_CHECK_C(C);
  return bn_bwd_apply(make_upstream(dz, arg, K), y, scale, shift, ka, kb, kc, P, C, relu, seed, drop_p, dy, stream);
}

extern "C" int s4g_train_bn_bwd_apply_seg_bf16(const void* dz, const int* arg, long long N, const void* y, const float* scale,
                                               const float* shift, const float* ka, const float* kb, const float* kc,
                                               long long P, int C, int relu, void* dy, void* stream) {
  S4G_CHECK_ARG(dz && arg && y && scale && shift && ka && kb && kc && dy && N > 0 && P > 0 && P % N == 0 && P < (1ll << 31),
                "train_bn_bwd_apply_seg: bad arguments");
  TRN_CHECK_C(C);
  return bn_bwd_apply(make_upstream(dz, nullptr, (int)N, arg), y, scale, shift, ka, kb, kc, P, C, relu, 0u, 0.f, dy, stream);
}

extern "C" int s4g_train_bn_act_segmax_bf16(const void* y, const float* scale, const float* shift, void* out, int* arg,
                                            void* ymax, unsigned long long* work, int B, long long N, int C, int relu,
                                            void* stream) {
  S4G_CHECK_ARG(y && scale && shift && out && arg && work && B > 0 && B <= 65535 && N > 0 && N < (1ll << 31),
                "train_bn_act_segmax: bad arguments");
  TRN_CHECK_C(C);
  cudaStream_t s = (cudaStream_t)stream;
  S4G_CUDA(cudaMemsetAsync(work, 0, sizeof(unsigned long long) * (size_t)B * C, s));
  const dim3 grid((unsigned)((N + kSegRows - 1) / kSegRows), (unsigned)B);
  bn_act_segmax_kernel<<<grid, 256, sizeof(unsigned long long) * (size_t)C, s>>>(reinterpret_cast<const bf16*>(y), scale,
                                                                                 shift, N, C, relu, work);
  S4G_LAUNCH_CHECK("train_bn_act_segmax");
  const long long bp = (long long)B * (C >> 3);
  bn_act_segmax_finish_kernel<<<grid_for(bp, 256), 256, 0, s>>>(work, reinterpret_cast<const bf16*>(y), N, C, bp,
                                                                reinterpret_cast<bf16*>(out), arg, reinterpret_cast<bf16*>(ymax));
  S4G_LAUNCH_CHECK("train_bn_act_segmax_finish");
  return S4G_OK;
}

extern "C" int s4g_train_rows_segment_sum_bf16(const void* dz, long long ld, int B, long long Nq, int C2, float* out,
                                               void* stream) {
  S4G_CHECK_ARG(dz && out && B > 0 && B <= 65535 && Nq > 0 && C2 > 0 && C2 % 8 == 0 && ld >= C2 && ld % 8 == 0,
                "train_rows_segment_sum: bad arguments");
  const int pieces = C2 >> 3;
  const int pg = pieces < kSumPieces ? pieces : kSumPieces;
  const dim3 grid((unsigned)((pieces + pg - 1) / pg), (unsigned)B);
  rows_segment_sum_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const bf16*>(dz), ld, Nq, C2, out);
  S4G_LAUNCH_CHECK("train_rows_segment_sum");
  return S4G_OK;
}

extern "C" int s4g_train_group_rows_bf16(const void* feat, const float* xyz, const float* ctr, const int* nbr, int B, int N,
                                         int M, int K, int Cf, void* out, void* stream) {
  S4G_CHECK_ARG(xyz && ctr && nbr && out && B > 0 && N > 0 && M > 0 && K > 0 && Cf >= 0 && Cf % 8 == 0 && (Cf == 0 || feat),
                "train_group_rows: bad arguments");
  const long long rows = (long long)B * M * K;
  group_rows_kernel<<<grid_for(rows * ((Cf >> 3) + 1), 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const bf16*>(feat), xyz, ctr, nbr, N, M, K, Cf, rows, reinterpret_cast<bf16*>(out));
  S4G_LAUNCH_CHECK("train_group_rows");
  return S4G_OK;
}

// dfeat (fp32 [B*N][Cf]) must be zeroed (or hold the gradient to add to) by the caller
extern "C" int s4g_train_group_rows_bwd(const void* dx, long long ld, const int* nbr, int B, int N, int M, int K, int Cf,
                                        float* dfeat, void* stream) {
  S4G_CHECK_ARG(dx && nbr && dfeat && B > 0 && N > 0 && M > 0 && K > 0 && Cf > 0 && Cf % 8 == 0 && ld >= Cf && ld % 8 == 0,
                "train_group_rows_bwd: bad arguments");
  const long long rows = (long long)B * M * K;
  group_rows_bwd_kernel<<<grid_for(rows * (Cf >> 3), 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const bf16*>(dx), ld, nbr, N, (long long)M * K, Cf, rows, dfeat);
  S4G_LAUNCH_CHECK("train_group_rows_bwd");
  return S4G_OK;
}

extern "C" int s4g_train_interp_rows_bwd(const void* dx, long long ld, const int* index, const float* weight, int B, int Nk,
                                         int Nq, int C2, float* dsparse, void* stream) {
  S4G_CHECK_ARG(dx && index && weight && dsparse && B > 0 && Nk > 0 && Nq > 0 && C2 > 0 && C2 % 8 == 0 && ld >= C2 && ld % 8 == 0,
                "train_interp_rows_bwd: bad arguments");
  const long long rows = (long long)B * Nq;
  interp_rows_bwd_kernel<<<grid_for(rows * (C2 >> 3), 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const bf16*>(dx), ld, index, weight, Nk, Nq, C2, rows, dsparse);
  S4G_LAUNCH_CHECK("train_interp_rows_bwd");
  return S4G_OK;
}

extern "C" int s4g_train_f32_to_bf16(const float* x, void* y, long long n, void* stream) {
  S4G_CHECK_ARG(x && y && n >= 0 && n % 8 == 0, "train_f32_to_bf16: element count must be a multiple of 8");
  if (n == 0) return S4G_OK;
  f32_to_bf16_kernel<<<grid_for(n / 8, 256), 256, 0, (cudaStream_t)stream>>>(x, reinterpret_cast<bf16*>(y), n / 8);
  S4G_LAUNCH_CHECK("train_f32_to_bf16");
  return S4G_OK;
}

extern "C" int s4g_train_bn_finalize(const double* sums2c, long long P, int C, const float* gamma, const float* beta, float eps,
                                     float momentum, float* running_mean, float* running_var, float* out4c, void* stream) {
  S4G_CHECK_ARG(sums2c && gamma && beta && out4c && P > 0 && C > 0 && (running_mean == nullptr) == (running_var == nullptr),
                "train_bn_finalize: bad arguments");
  bn_finalize_kernel<<<grid_for(C, 128), 128, 0, (cudaStream_t)stream>>>(sums2c, P, C, gamma, beta, eps, momentum,
                                                                        running_mean, running_var, out4c);
  S4G_LAUNCH_CHECK("train_bn_finalize");
  return S4G_OK;
}

extern "C" int s4g_train_bn_bwd_finalize(const double* sums2c, long long P, int C, const float* gamma, const float* mean_rstd,
                                         float* dgamma, float* dbeta, float* out3c, void* stream) {
  S4G_CHECK_ARG(sums2c && gamma && mean_rstd && dgamma && dbeta && out3c && P > 0 && C > 0, "train_bn_bwd_finalize: bad arguments");
  bn_bwd_finalize_kernel<<<grid_for(C, 128), 128, 0, (cudaStream_t)stream>>>(sums2c, P, C, gamma, mean_rstd, dgamma, dbeta, out3c);
  S4G_LAUNCH_CHECK("train_bn_bwd_finalize");
  return S4G_OK;
}

extern "C" int s4g_train_head_logits_fwd(const void* h, const float* w, const float* bias, float* out, long long P, int C, int k,
                                         int n_points, void* stream) {
  S4G_CHECK_ARG(h && w && bias && out && P > 0 && k > 0 && k <= kMaxLogits && n_points > 0 && P % n_points == 0,
                "train_head_logits_fwd: bad arguments");
  TRN_CHECK_C(C);
  S4G_CHECK_ARG(P < (1ll << 31) && C <= 512, "train_head_logits_fwd: at most 512 channels");
  const size_t smem = sizeof(float) * (size_t)k * C + (size_t)kHeadRows * (2 * C + 16);
  static bool attr[64] = {};
  if (s4g::first_use_on_device(attr))
    S4G_CUDA(cudaFuncSetAttribute(head_logits_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  head_logits_fwd_kernel<<<grid_for(P, kHeadRows), 256, smem, (cudaStream_t)stream>>>(
      reinterpret_cast<const bf16*>(h), w, bias, out, (int)P, C, k, n_points);
  S4G_LAUNCH_CHECK("train_head_logits_fwd");
  return S4G_OK;
}

extern "C" int s4g_train_head_logits_bwd(const float* dlogits, const float* w, void* dh, long long P, int C, int k, int n_points,
                                         void* stream) {
  S4G_CHECK_ARG(dlogits && w && dh && P > 0 && k > 0 && k <= kMaxLogits && n_points > 0 && P % n_points == 0,
                "train_head_logits_bwd: bad arguments");
  TRN_CHECK_C(C);
  S4G_CHECK_ARG(P < (1ll << 31), "train_head_logits_bwd: too many rows");
  const unsigned grid = grid_for(P, kHeadRows);
  cudaStream_t st = (cudaStream_t)stream;
  bf16* out = reinterpret_cast<bf16*>(dh);
  if (k <= 4) head_logits_bwd_kernel<4><<<grid, 256, 0, st>>>(dlogits, w, out, (int)P, C, k, n_points);
  else if (k <= 9) head_logits_bwd_kernel<9><<<grid, 256, 0, st>>>(dlogits, w, out, (int)P, C, k, n_points);
  else head_logits_bwd_kernel<kMaxLogits><<<grid, 256, 0, st>>>(dlogits, w, out, (int)P, C, k, n_points);
  S4G_LAUNCH_CHECK("train_head_logits_bwd");
  return S4G_OK;
}

extern "C" int s4g_train_sum_bf16(const void* a, const void* b, const void* c, const void* d, void* out, long long n,
                                  void* stream) {
  S4G_CHECK_ARG(a && b && out && n >= 0 && n % 8 == 0 && (c || !d), "train_sum_bf16: element count must be a multiple of 8");
  if (n == 0) return S4G_OK;
  sum_bf16_kernel<<<grid_for(n / 8, 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const uint4*>(a), reinterpret_cast<const uint4*>(b), reinterpret_cast<const uint4*>(c),
      reinterpret_cast<const uint4*>(d), reinterpret_cast<uint4*>(out), n / 8);
  S4G_LAUNCH_CHECK("train_sum_bf16");
  return S4G_OK;
}

extern "C" int s4g_train_head_logits_dw(const float* dlogits, const void* h, float* dw, float* dbias, long long P, int C, int k,
                                        int n_points, void* stream) {
  S4G_CHECK_ARG(dlogits && h && dw && dbias && P > 0 && k > 0 && k <= kMaxLogits && n_points > 0 && P % n_points == 0,
                "train_head_logits_dw: bad arguments");
  TRN_CHECK_C(C);
  S4G_CHECK_ARG(P < (1ll << 31), "train_head_logits_dw: too many rows");
  const size_t smem = sizeof(float) * 2048;  // lanes * C = (256 / pieces) * pieces * 8 <= 2048
  const unsigned grid = grid_for(P, kDwTiles * kHeadRows);
  cudaStream_t st = (cudaStream_t)stream;
  const bf16* hh = reinterpret_cast<const bf16*>(h);
  if (k <= 4) head_logits_dw_kernel<4><<<grid, 256, smem, st>>>(dlogits, hh, dw, dbias, (int)P, C, k, n_points);
  else if (k <= 9) head_logits_dw_kernel<9><<<grid, 256, smem, st>>>(dlogits, hh, dw, dbias, (int)P, C, k, n_points);
  else head_logits_dw_kernel<kMaxLogits><<<grid, 256, smem, st>>>(dlogits, hh, dw, dbias, (int)P, C, k, n_points);
  S4G_LAUNCH_CHECK("train_head_logits_dw");
  return S4G_OK;
}

// Inverse of an index tensor (B, E) with values in [0, T) — the 3-NN index (E = Nq * 3, T = Nk) or the ball-query
// neighbour index (E = M * K, T = N): per target (b, j) the list of entries e = b * E + i with index[e] == j.
// Step 1: count[B * T] (zeroed here).  The caller turns it into `end` = inclusive scan (int32).
extern "C" int s4g_train_index_inverse_count(const int* index, int B, int T, long long E, int* count, void* stream) {
  S4G_CHECK_ARG(index && count && B > 0 && T > 0 && E > 0 && (long long)B * E < (1ll << 31), "train_index_inverse_count: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  S4G_CUDA(cudaMemsetAsync(count, 0, sizeof(int) * (size_t)B * T, st));
  const long long entries = (long long)B * E;
  interp_inverse_count_kernel<<<grid_for(entries, 256), 256, 0, st>>>(index, T, E, entries, count);
  S4G_LAUNCH_CHECK("train_index_inverse_count");
  return S4G_OK;
}
// Step 2: cursor[B * T] = the lists' start offsets (end - count) on entry, advanced to their ends; list[B * E].
extern "C" int s4g_train_index_inverse_fill(const int* index, int B, int T, long long E, int* cursor, int* list, void* stream) {
  S4G_CHECK_ARG(index && cursor && list && B > 0 && T > 0 && E > 0, "train_index_inverse_fill: bad arguments");
  const long long entries = (long long)B * E;
  interp_inverse_fill_kernel<<<grid_for(entries, 256), 256, 0, (cudaStream_t)stream>>>(index, T, E, entries, cursor, list);
  S4G_LAUNCH_CHECK("train_index_inverse_fill");
  return S4G_OK;
}
// The scatter-add gradients as a gather: out[b * T + j][c] (+)= sum over the list of (b, j) of weight[e] * dx[e / div][c]
// (div = 3 with weights: InterpolateBackward;  div = 1, weight NULL: GroupPointsBackward).  fp32 and / or bf16 rows
// [B * T][C] (either may be NULL); accumulate != 0 adds into out_f32 (bf16 output then holds the sum as well).  The order
// inside a list is the fill's (atomic cursor): the fp32 sum may differ in its last bits between runs, like the scatter's.
extern "C" int s4g_train_rows_bwd_gather(const void* dx, long long ld, const int* list, const int* end, const int* count,
                                         const float* weight, int div, long long targets, int C, int accumulate,
                                         float* out_f32, void* out_bf16, void* stream) {
  S4G_CHECK_ARG(dx && list && end && count && (out_f32 || out_bf16) && targets > 0 && C > 0 && C % 8 == 0 && C <= 2048 &&
                    ld >= C && ld % 8 == 0 && (div == 1 || div == 3) && (!accumulate || out_f32),
                "train_rows_bwd_gather: bad arguments");
  const int lanes = 256 / (C >> 3);
  const unsigned grid = grid_for(targets, lanes);
  cudaStream_t st = (cudaStream_t)stream;
  if (div == 3)
    rows_bwd_gather_kernel<3><<<grid, 256, 0, st>>>(reinterpret_cast<const bf16*>(dx), ld, list, end, count, weight, targets, C,
                                                    accumulate, out_f32, reinterpret_cast<bf16*>(out_bf16));
  else
    rows_bwd_gather_kernel<1><<<grid, 256, 0, st>>>(reinterpret_cast<const bf16*>(dx), ld, list, end, count, weight, targets, C,
                                                    accumulate, out_f32, reinterpret_cast<bf16*>(out_bf16));
  S4G_LAUNCH_CHECK("train_rows_bwd_gather");
  return S4G_OK;
}

extern "C" int s4g_train_relu_mask_rows_bf16(const void* dz, const void* y, const float* scale, const float* shift, long long P,
                                             int C, void* out, void* stream) {
  S4G_CHECK_ARG(dz && y && scale && shift && out && P > 0, "train_relu_mask_rows: bad arguments");
  TRN_CHECK_C(C);
  relu_mask_rows_kernel<<<grid_for(P * (C >> 3), 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const bf16*>(dz), reinterpret_cast<const bf16*>(y), scale, shift, P, C, reinterpret_cast<bf16*>(out));
  S4G_LAUNCH_CHECK("train_relu_mask_rows");
  return S4G_OK;
}
