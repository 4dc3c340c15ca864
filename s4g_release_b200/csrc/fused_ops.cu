// Feature-propagation front end of the fused path (channel-last bf16 features):
//   * three_nn_weights: the reference's PointSearch (interpolate_kernel.cu:33-81) fused with the
//     inverse-squared-distance weights of FeatureInterpolator.forward (pointnet2_utils/modules.py:115-120):
//     w_k = (1/max(d2_k,1e-10)) / sum_k(1/max(d2_k,1e-10)), int32 indices;
//   * interp_concat: InterpolateForward (interpolate_kernel.cu:139-181) + the channel concat of
//     modules.py:124-127 ("interpolated first, then the dense skip feature") written once, as the bf16
//     row matrix the MLP chain consumes.
#include <cuda_bf16.h>

#include "common.cuh"
#include "grid.cuh"

namespace s4g {

constexpr int kNnwThreads = 256;
constexpr int kNnwTile = 2048;

__global__ void __launch_bounds__(kNnwThreads)
three_nn_weights_kernel(const float* __restrict__ query, const float* __restrict__ key, int Nq, int Nk,
                        int* __restrict__ index, float* __restrict__ weight) {
  __shared__ float4 s_key[kNnwTile];
  const int b = blockIdx.y;
  const int i = blockIdx.x * kNnwThreads + threadIdx.x;
  const bool valid = i < Nq;
  const float* Q = query + (size_t)b * 3 * Nq;
  const float* KX = key + (size_t)b * 3 * Nk;
  const float* KY = KX + Nk;
  const float* KZ = KY + Nk;
  const int iq = valid ? i : Nq - 1;
  const float x1 = Q[iq], y1 = Q[Nq + iq], z1 = Q[2 * Nq + iq];
  const float inf = __int_as_float(0x7f800000);
  float d0 = inf, d1 = inf, d2 = inf;
  int i0 = -1, i1 = -1, i2 = -1;
  for (int base = 0; base < Nk; base += kNnwTile) {
    const int n = min(kNnwTile, Nk - base);
    __syncthreads();
    for (int k = threadIdx.x; k < n; k += kNnwThreads)
      s_key[k] = make_float4(__ldg(KX + base + k), __ldg(KY + base + k), __ldg(KZ + base + k), 0.f);
    __syncthreads();
#pragma unroll 4
    for (int k = 0; k < n; ++k) {
      const float4 p = s_key[k];
      const float d = sqdist(__fsub_rn(x1, p.x), __fsub_rn(y1, p.y), __fsub_rn(z1, p.z));
      if (d < d2) {
        const int j = base + k;
        if (d < d1) {
          d2 = d1; i2 = i1;
          if (d < d0) { d1 = d0; i1 = i0; d0 = d; i0 = j; }
          else { d1 = d; i1 = j; }
        } else { d2 = d; i2 = j; }
      }
    }
  }
  if (valid) {
    // the reference's distances when fewer than three are finite; its index -1 (weight 1/inf = 0) is written as 0
    three_nn_reference_tail(d0, d1, d2, i0, i1, i2, inf);
    const float v0 = __fdiv_rn(1.0f, fmaxf(d0, 1e-10f));
    const float v1 = __fdiv_rn(1.0f, fmaxf(d1, 1e-10f));
    const float v2 = __fdiv_rn(1.0f, fmaxf(d2, 1e-10f));
    const float norm = __fadd_rn(__fadd_rn(v0, v1), v2);
    int* oi = index + ((size_t)b * Nq + i) * 3;
    float* ow = weight + ((size_t)b * Nq + i) * 3;
    oi[0] = max(i0, 0); oi[1] = max(i1, 0); oi[2] = max(i2, 0);
    ow[0] = __fdiv_rn(v0, norm); ow[1] = __fdiv_rn(v1, norm); ow[2] = __fdiv_rn(v2, norm);
  }
}

// One warp per kInterpRows consecutive query rows of one cloud (blockIdx.y = cloud: no 64-bit divisions); the 3 x 4
// neighbour indices / weights of the rows are one coalesced load by 12 lanes and travel by shuffle; per 16-byte piece
// (8 bf16 channels) the 3 x 4 gathered loads of all rows are issued before any arithmetic, so 12 requests per lane are
// in flight.  (r1 kernel: one row per warp, index arithmetic in 64 bit per lane — 24.7 % of the HBM peak with 61 % of the
// issue slots busy at the finest level, profiles/r02/ncu_geometry.txt.)
constexpr int kInterpRows = 4;

__device__ __forceinline__ uint32_t interp_pair(uint32_t a, uint32_t b, uint32_t c, float w0, float w1, float w2, bool relu) {
  // bf16 -> fp32 is a 16-bit shift; fma(in2,w2, fma(in1,w1, in0*w0)) as interpolate_kernel.cu:167-174
  const float x = __fmaf_rn(__uint_as_float(c << 16), w2, __fmaf_rn(__uint_as_float(b << 16), w1, __fmul_rn(__uint_as_float(a << 16), w0)));
  const float y = __fmaf_rn(__uint_as_float(c & 0xffff0000u), w2,
                            __fmaf_rn(__uint_as_float(b & 0xffff0000u), w1, __fmul_rn(__uint_as_float(a & 0xffff0000u), w0)));
  __nv_bfloat162 h = __floats2bfloat162_rn(x, y);
  uint32_t r = *reinterpret_cast<uint32_t*>(&h);
  if (relu) asm("max.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(r), "r"(0u));
  return r;
}

__global__ void __launch_bounds__(256)
interp_concat_kernel(const __nv_bfloat16* __restrict__ sparse, const int* __restrict__ index,
                     const float* __restrict__ weight, const __nv_bfloat16* __restrict__ dense, int Nk, int Nq,
                     int C2, int C1, __nv_bfloat16* __restrict__ out, int relu) {
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  const int row0 = (blockIdx.x * 8 + (threadIdx.x >> 5)) * kInterpRows;
  if (row0 >= Nq) return;
  const int n_rows = min(kInterpRows, Nq - row0);
  const size_t q0 = (size_t)b * Nq + row0;  // first (batch-global) query row of this warp
  int my_i = 0;
  float my_w = 0.f;
  if (lane < 3 * n_rows) {
    my_i = __ldg(index + q0 * 3 + lane);
    my_w = __ldg(weight + q0 * 3 + lane);
  }
  const uint4* src[kInterpRows][3];
  float w[kInterpRows][3];
#pragma unroll
  for (int r = 0; r < kInterpRows; ++r)
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int j = __shfl_sync(0xffffffffu, my_i, 3 * r + k);  // rows past n_rows read index 0 (valid) and are not stored
      w[r][k] = __shfl_sync(0xffffffffu, my_w, 3 * r + k);
      src[r][k] = reinterpret_cast<const uint4*>(sparse + ((size_t)b * Nk + j) * C2);
    }
  const int width = C2 + C1;
  for (int c = lane; c < C2 / 8; c += 32) {
    uint4 v[kInterpRows][3];
#pragma unroll
    for (int r = 0; r < kInterpRows; ++r)
#pragma unroll
      for (int k = 0; k < 3; ++k) v[r][k] = __ldg(src[r][k] + c);
#pragma unroll
    for (int r = 0; r < kInterpRows; ++r) {
      if (r < n_rows) {
        uint4 o;
        o.x = interp_pair(v[r][0].x, v[r][1].x, v[r][2].x, w[r][0], w[r][1], w[r][2], relu);
        o.y = interp_pair(v[r][0].y, v[r][1].y, v[r][2].y, w[r][0], w[r][1], w[r][2], relu);
        o.z = interp_pair(v[r][0].z, v[r][1].z, v[r][2].z, w[r][0], w[r][1], w[r][2], relu);
        o.w = interp_pair(v[r][0].w, v[r][1].w, v[r][2].w, w[r][0], w[r][1], w[r][2], relu);
        reinterpret_cast<uint4*>(out + (q0 + r) * width)[c] = o;
      }
    }
  }
  if (C1 > 0) {
    for (int c = lane; c < C1 / 8; c += 32) {
      uint4 d[kInterpRows];
#pragma unroll
      for (int r = 0; r < kInterpRows; ++r)
        if (r < n_rows) d[r] = __ldg(reinterpret_cast<const uint4*>(dense + (q0 + r) * C1) + c);
#pragma unroll
      for (int r = 0; r < kInterpRows; ++r)
        if (r < n_rows) reinterpret_cast<uint4*>(out + (q0 + r) * width + C2)[c] = d[r];
    }
  }
}

// fp32 channel-first (B,C,N) -> bf16 channel-last [B*N][C] and back (interface <-> fused-path layout)
__global__ void __launch_bounds__(256)
gather_xyz_kernel(const float* __restrict__ xyz, const int* __restrict__ index, int N, int M, float* __restrict__ out) {
  const int b = blockIdx.y;
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  const int j = index[(size_t)b * M + m];
  const float* X = xyz + (size_t)b * 3 * N;
  float* O = out + (size_t)b * 3 * M;
  O[m] = __ldg(X + j);
  O[M + m] = __ldg(X + N + j);
  O[2 * M + m] = __ldg(X + 2 * N + j);
}

// Global set-abstraction level (num_centroids = 0, modules.py:93-98): the gathered max-pool chain pools a scene's N
// points as P partial groups; this kernel reduces the P partial rows of each scene.  Max is exact and ignores order and
// repeated rows, so the result equals the one N-wide group of the reference bit for bit.  One lane per 16-byte piece
// (8 channels) of a row; the 8 warps of a block split the rows and meet in shared memory.
constexpr int kSegWarps = 8;

__device__ __forceinline__ uint32_t max_bf16x2(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("max.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}

__device__ __forceinline__ uint4 max_bf16x8(uint4 a, uint4 b) {
  return make_uint4(max_bf16x2(a.x, b.x), max_bf16x2(a.y, b.y), max_bf16x2(a.z, b.z), max_bf16x2(a.w, b.w));
}

__global__ void __launch_bounds__(32 * kSegWarps)
rows_segment_max_kernel(const uint4* __restrict__ in, int P, int C8, uint4* __restrict__ out) {
  __shared__ uint4 s_part[kSegWarps][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.y;
  const int c = blockIdx.x * 32 + lane;
  const uint32_t ninf = 0xff80ff80u;  // bf16 -inf pair
  uint4 m = make_uint4(ninf, ninf, ninf, ninf);
  if (c < C8) {
    const uint4* src = in + (size_t)b * P * C8 + c;
#pragma unroll 4
    for (int r = warp; r < P; r += kSegWarps) m = max_bf16x8(m, __ldg(src + (size_t)r * C8));
  }
  s_part[warp][lane] = m;
  __syncthreads();
  if (warp == 0 && c < C8) {
#pragma unroll
    for (int w = 1; w < kSegWarps; ++w) m = max_bf16x8(m, s_part[w][lane]);
    out[(size_t)b * C8 + c] = m;
  }
}

// Broadcast feature propagation (num_fp_neighbours = 0, modules.py:131-134): the single global feature of a scene is
// repeated on every dense row, followed by the dense skip feature — [broadcast | skip], the reference's order.  One
// thread per 16-byte piece of an output row.
__global__ void __launch_bounds__(256)
broadcast_concat_kernel(const uint4* __restrict__ sparse, const uint4* __restrict__ dense, int Nq, int C2_8, int C1_8,
                        uint4* __restrict__ out) {
  const int b = blockIdx.y;
  const int w8 = C2_8 + C1_8;
  const int n = Nq * w8;
  uint4* O = out + (size_t)b * n;
  for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
    const int q = i / w8, c = i - q * w8;
    O[i] = c < C2_8 ? __ldg(sparse + (size_t)b * C2_8 + c) : __ldg(dense + ((size_t)b * Nq + q) * C1_8 + (c - C2_8));
  }
}

// Input rows of PN2_LOCAL's grasp-evaluation head (PointNet2_local.forward_modules; reference :131-147): row (b, f, s) of [B*F*S][C + 48] is the
// point feature of point f followed by the 12 candidate values [R0..R8 t0..t2] repeated 4 times, the order of
// torch.cat([per_point, frames.repeat(1, 4, 1, 1)], 1).  12 values x 2 repeats = 24 bf16 = three 16-byte pieces, so the
// 48 candidate channels are those three pieces twice.  Phase 1: one thread per row reads its 12 fp32 values (coalesced
// across neighbouring (f, s)), in the given mode makes the translation relative to the point and writes it back to the
// caller's frames (the reference's in-place update, :135), and stages the three bf16 pieces in shared memory.  Phase 2:
// the block writes its rows, which are contiguous in the output, one thread per 16-byte piece.
constexpr int kEvalRows = 256;

__global__ void __launch_bounds__(kEvalRows)
local_eval_rows_kernel(const uint4* __restrict__ feat, int N, int C8, float* frames, const float* __restrict__ points,
                       const float* __restrict__ R, const float* __restrict__ t, int F, int S, long long rows,
                       uint4* __restrict__ out) {
  __shared__ uint4 s_cand[kEvalRows][3];
  __shared__ long long s_src[kEvalRows];  // the row's point-feature row b * N + f
  const long long r0 = (long long)blockIdx.x * kEvalRows;
  const int nrows = (int)min((long long)kEvalRows, rows - r0);
  const long long FS = (long long)F * S;
  if ((int)threadIdx.x < nrows) {
    const long long r = r0 + threadIdx.x;
    const long long b = r / FS, fs = r - b * FS;
    s_src[threadIdx.x] = b * N + fs / S;
    float v[12];
    if (frames != nullptr) {  // given: frames (B, 12, F, S); points (B, 3, N)
      float* fr = frames + b * 12 * FS + fs;
#pragma unroll
      for (int k = 0; k < 9; ++k) v[k] = fr[k * FS];
      const int f = (int)(fs / S);
      const float* p = points + b * 3 * N + f;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        v[9 + k] = __fsub_rn(fr[(9 + k) * FS], __ldg(p + (size_t)k * N));
        fr[(9 + k) * FS] = v[9 + k];
      }
    } else {  // self: R (B, 9, N), t (B, 3, N); F = N, S = 1
#pragma unroll
      for (int k = 0; k < 9; ++k) v[k] = __ldg(R + (b * 9 + k) * N + fs);
#pragma unroll
      for (int k = 0; k < 3; ++k) v[9 + k] = __ldg(t + (b * 3 + k) * N + fs);
    }
    uint32_t h[12];
#pragma unroll
    for (int k = 0; k < 12; k += 2) {
      const __nv_bfloat162 pr = __floats2bfloat162_rn(v[k], v[k + 1]);
      h[k / 2] = *reinterpret_cast<const uint32_t*>(&pr);
    }
    // bf16 pairs: piece 0 = v0..v7, piece 1 = v8..v11 v0..v3, piece 2 = v4..v11
    s_cand[threadIdx.x][0] = make_uint4(h[0], h[1], h[2], h[3]);
    s_cand[threadIdx.x][1] = make_uint4(h[4], h[5], h[0], h[1]);
    s_cand[threadIdx.x][2] = make_uint4(h[2], h[3], h[4], h[5]);
  }
  __syncthreads();
  const int w8 = C8 + 6;
  const int n = nrows * w8;
  uint4* O = out + r0 * w8;
  for (int i = threadIdx.x; i < n; i += kEvalRows) {
    const int q = i / w8, c = i - q * w8;
    uint4 val;
    if (c < C8)
      val = __ldg(feat + s_src[q] * C8 + c);
    else
      val = s_cand[q][(c - C8) % 3];
    O[i] = val;
  }
}

}  // namespace s4g

extern "C" int s4g_rows_segment_max_bf16(const void* in, int B, int P, int C, void* out, void* stream) {
  S4G_CHECK_ARG(in && out, "rows_segment_max: null pointer");
  S4G_CHECK_ARG(B >= 0 && B <= 65535 && P > 0 && C > 0 && C % 8 == 0, "rows_segment_max: bad shape (C %% 8 == 0)");
  S4G_CHECK_ARG(((uintptr_t)in & 15) == 0 && ((uintptr_t)out & 15) == 0, "rows_segment_max: rows must be 16-byte aligned");
  if (B == 0) return S4G_OK;
  const int C8 = C / 8;
  const dim3 grid((unsigned)((C8 + 31) / 32), (unsigned)B);
  s4g::rows_segment_max_kernel<<<grid, 32 * s4g::kSegWarps, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const uint4*>(in), P, C8, reinterpret_cast<uint4*>(out));
  S4G_LAUNCH_CHECK("rows_segment_max");
  return S4G_OK;
}

extern "C" int s4g_broadcast_concat_bf16(const void* sparse, const void* dense, int B, int Nq, int C2, int C1, void* out,
                                         void* stream) {
  S4G_CHECK_ARG(sparse && out, "broadcast_concat: null pointer");
  S4G_CHECK_ARG(C2 > 0 && C2 % 8 == 0 && C1 >= 0 && C1 % 8 == 0, "broadcast_concat: channel counts must be multiples of 8");
  S4G_CHECK_ARG(C1 == 0 || dense != nullptr, "broadcast_concat: dense feature missing");
  S4G_CHECK_ARG(B >= 0 && B <= 65535 && Nq > 0 && (long long)Nq * ((C2 + C1) / 8) < (1ll << 31),
                "broadcast_concat: bad shape");
  S4G_CHECK_ARG(((uintptr_t)sparse & 15) == 0 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)dense & 15) == 0,
                "broadcast_concat: feature rows must be 16-byte aligned");
  if (B == 0) return S4G_OK;
  const long long pieces = (long long)Nq * ((C2 + C1) / 8);
  const dim3 grid((unsigned)std::min<long long>((pieces + 255) / 256, 1024), (unsigned)B);
  s4g::broadcast_concat_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const uint4*>(sparse), reinterpret_cast<const uint4*>(dense), Nq, C2 / 8, C1 / 8,
      reinterpret_cast<uint4*>(out));
  S4G_LAUNCH_CHECK("broadcast_concat");
  return S4G_OK;
}

extern "C" int s4g_local_eval_rows_bf16(const void* feat, int B, int N, int C, float* frames, const float* points,
                                        int F, int S, const float* R, const float* t, void* out, void* stream) {
  S4G_CHECK_ARG(feat && out, "local_eval_rows: null pointer");
  S4G_CHECK_ARG(frames ? points != nullptr : (R && t), "local_eval_rows: frames need points; without frames R and t");
  S4G_CHECK_ARG(B >= 0 && N > 0 && C > 0 && C % 8 == 0, "local_eval_rows: bad shape (C %% 8 == 0)");
  S4G_CHECK_ARG(frames ? (F >= 1 && F <= N && S >= 1) : (F == N && S == 1),
                "local_eval_rows: bad candidate shape (given: 1 <= F <= N, S >= 1; self: F = N, S = 1)");
  S4G_CHECK_ARG(((uintptr_t)feat & 15) == 0 && ((uintptr_t)out & 15) == 0,
                "local_eval_rows: feature and output rows must be 16-byte aligned");
  const long long rows = (long long)B * F * S;
  S4G_CHECK_ARG((rows + s4g::kEvalRows - 1) / s4g::kEvalRows < (1ll << 31), "local_eval_rows: too many rows");
  if (rows == 0) return S4G_OK;
  const unsigned grid = (unsigned)((rows + s4g::kEvalRows - 1) / s4g::kEvalRows);
  s4g::local_eval_rows_kernel<<<grid, s4g::kEvalRows, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const uint4*>(feat), N, C / 8, frames, points, R, t, F, S, rows, reinterpret_cast<uint4*>(out));
  S4G_LAUNCH_CHECK("local_eval_rows");
  return S4G_OK;
}

extern "C" int s4g_three_nn_weights_f32_i32(const float* query, const float* key, int B, int Nq, int Nk, int* index,
                                            float* weight, void* stream) {
  S4G_CHECK_ARG(query && key && index && weight, "three_nn_weights: null pointer");
  S4G_CHECK_ARG(Nk >= 3, "three_nn_weights: num_key < 3");
  S4G_CHECK_ARG(B >= 0 && B <= 65535 && Nq > 0, "three_nn_weights: bad shape");
  if (B == 0) return S4G_OK;
  if (Nk >= s4g::kGridKnnMinKeys)
    return s4g::three_nn_grid<1>(query, key, B, Nq, Nk, index, weight, (cudaStream_t)stream);
  dim3 grid((Nq + s4g::kNnwThreads - 1) / s4g::kNnwThreads, B);
  s4g::three_nn_weights_kernel<<<grid, s4g::kNnwThreads, 0, (cudaStream_t)stream>>>(query, key, Nq, Nk, index, weight);
  S4G_LAUNCH_CHECK("three_nn_weights");
  return S4G_OK;
}

extern "C" int s4g_interp_concat_act_bf16(const void* sparse, const int* index, const float* weight, const void* dense,
                                          int B, int Nk, int Nq, int C2, int C1, int relu, void* out, void* stream) {
  S4G_CHECK_ARG(sparse && index && weight && out, "interp_concat: null pointer");
  S4G_CHECK_ARG(C2 > 0 && C2 % 8 == 0 && C1 >= 0 && C1 % 8 == 0, "interp_concat: channel counts must be multiples of 8");
  S4G_CHECK_ARG(C1 == 0 || dense != nullptr, "interp_concat: dense feature missing");
  S4G_CHECK_ARG(B >= 0 && B <= 65535 && Nq > 0 && Nk > 0, "interp_concat: bad shape");
  S4G_CHECK_ARG(((uintptr_t)sparse & 15) == 0 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)dense & 15) == 0,
                "interp_concat: feature rows must be 16-byte aligned");
  if (B == 0) return S4G_OK;
  const dim3 grid((unsigned)((Nq + 8 * s4g::kInterpRows - 1) / (8 * s4g::kInterpRows)), (unsigned)B);
  s4g::interp_concat_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const __nv_bfloat16*>(sparse), index, weight, reinterpret_cast<const __nv_bfloat16*>(dense), Nk,
      Nq, C2, C1, reinterpret_cast<__nv_bfloat16*>(out), relu);
  S4G_LAUNCH_CHECK("interp_concat");
  return S4G_OK;
}

extern "C" int s4g_interp_concat_bf16(const void* sparse, const int* index, const float* weight, const void* dense,
                                      int B, int Nk, int Nq, int C2, int C1, void* out, void* stream) {
  return s4g_interp_concat_act_bf16(sparse, index, weight, dense, B, Nk, Nq, C2, C1, 0, out, stream);
}

extern "C" int s4g_gather_xyz_f32_i32(const float* xyz, const int* index, int B, int N, int M, float* out,
                                      void* stream) {
  S4G_CHECK_ARG(xyz && index && out, "gather_xyz: null pointer");
  S4G_CHECK_ARG(B >= 0 && B <= 65535 && N > 0 && M > 0, "gather_xyz: bad shape");
  if (B == 0) return S4G_OK;
  dim3 grid((M + 255) / 256, B);
  s4g::gather_xyz_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(xyz, index, N, M, out);
  S4G_LAUNCH_CHECK("gather_xyz");
  return S4G_OK;
}
