// a8: per-joint softmax + expectation of voxel-centre coordinates
// (utils/op.py:83-96).  HBM-bound: one pass over the logits with an online softmax
// (running max + rescaled sums), warp-shuffle reduction, cross-CTA combine through a
// tiny workspace.  The softmaxed volume (reference output #3) is written by a second
// elementwise pass only when the caller asks for it.
#include "common.cuh"

namespace sceneego {

constexpr int SA_THREADS = 256;
constexpr int SA_MAX_SPLITS = 64;
constexpr float kLog2e = 1.4426950408889634f;

struct SaAcc { float m, s, sx, sy, sz; };

__device__ __forceinline__ void sa_merge(SaAcc& a, const SaAcc& b) {
  const float m = fmaxf(a.m, b.m);
  const float fa = (a.m == -INFINITY) ? 0.f : exp2f((a.m - m) * kLog2e);
  const float fb = (b.m == -INFINITY) ? 0.f : exp2f((b.m - m) * kLog2e);
  a.s = a.s * fa + b.s * fb;
  a.sx = a.sx * fa + b.sx * fb;
  a.sy = a.sy * fa + b.sy * fb;
  a.sz = a.sz * fa + b.sz * fb;
  a.m = m;
}

// grid: (splits, B*J).  Each CTA reduces `chunk` consecutive voxels of one joint volume.
template <bool kSoftmax, bool kAxis>
__global__ void __launch_bounds__(SA_THREADS) softargmax_partial_kernel(
    const float* __restrict__ logits, int N, int V, int log2v, int chunk, float mult, const float* __restrict__ axis,
    const float* __restrict__ coords, float* __restrict__ partial) {
  extern __shared__ float s_axis[];  // 3*V when kAxis
  if (kAxis) {
    for (int i = threadIdx.x; i < 3 * V; i += SA_THREADS) s_axis[i] = axis[i];
    __syncthreads();
  }
  const int bj = blockIdx.y;
  const int begin = blockIdx.x * chunk;
  const int end = min(N, begin + chunk);
  const float4* src = reinterpret_cast<const float4*>(logits + (size_t)bj * N);
  SaAcc a{-INFINITY, 0.f, 0.f, 0.f, 0.f};
  if (!kSoftmax) a.m = 0.f;
  for (int i4 = begin / 4 + threadIdx.x; i4 < end / 4; i4 += SA_THREADS * 4) {
    float4 v[4];
    int idx[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      idx[u] = i4 + u * SA_THREADS;
      v[u] = (idx[u] < end / 4) ? __ldcs(src + idx[u]) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    }
    if (kSoftmax) {
      float mx = a.m;
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (idx[u] < end / 4)
          mx = fmaxf(mx, fmaxf(fmaxf(v[u].x * mult, v[u].y * mult), fmaxf(v[u].z * mult, v[u].w * mult)));
      if (mx > a.m) {
        const float f = (a.m == -INFINITY) ? 0.f : exp2f((a.m - mx) * kLog2e);
        a.s *= f; a.sx *= f; a.sy *= f; a.sz *= f;
        a.m = mx;
      }
      // every logit this thread has seen is -inf: their weights are 0, but exp2f(-inf - -inf) would make them NaN
      if (a.m == -INFINITY) continue;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (idx[u] >= end / 4) continue;
      const float e[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
      float w[4];
#pragma unroll
      for (int q = 0; q < 4; ++q)
        w[q] = kSoftmax ? exp2f((e[q] * mult - a.m) * kLog2e) : fmaxf(e[q] * mult, 0.f);
      const int n0 = idx[u] * 4;
      if (kAxis) {  // V % 4 == 0: the four voxels share x and y
        // power-of-two sides (64, 128): shifts instead of three runtime integer divisions per float4
        const int z0 = log2v >= 0 ? (n0 & (V - 1)) : n0 % V;
        const int y = log2v >= 0 ? ((n0 >> log2v) & (V - 1)) : (n0 / V) % V;
        const int x = log2v >= 0 ? (n0 >> (2 * log2v)) : n0 / (V * V);
        const float ws = (w[0] + w[1]) + (w[2] + w[3]);
        a.s += ws;
        a.sx = fmaf(ws, s_axis[x], a.sx);
        a.sy = fmaf(ws, s_axis[V + y], a.sy);
#pragma unroll
        for (int q = 0; q < 4; ++q) a.sz = fmaf(w[q], s_axis[2 * V + z0 + q], a.sz);
      } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float* c = coords + (size_t)(n0 + q) * 3;
          a.s += w[q];
          a.sx = fmaf(w[q], c[0], a.sx);
          a.sy = fmaf(w[q], c[1], a.sy);
          a.sz = fmaf(w[q], c[2], a.sz);
        }
      }
    }
  }
  // warp reduce, then one warp combines the 8 warps
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    SaAcc b;
    b.m = __shfl_xor_sync(0xffffffffu, a.m, o);
    b.s = __shfl_xor_sync(0xffffffffu, a.s, o);
    b.sx = __shfl_xor_sync(0xffffffffu, a.sx, o);
    b.sy = __shfl_xor_sync(0xffffffffu, a.sy, o);
    b.sz = __shfl_xor_sync(0xffffffffu, a.sz, o);
    if (kSoftmax) sa_merge(a, b);
    else { a.s += b.s; a.sx += b.sx; a.sy += b.sy; a.sz += b.sz; }
  }
  __shared__ SaAcc s_part[SA_THREADS / 32];
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) {
    SaAcc t = s_part[0];
    for (int w = 1; w < SA_THREADS / 32; ++w) {
      if (kSoftmax) sa_merge(t, s_part[w]);
      else { t.s += s_part[w].s; t.sx += s_part[w].sx; t.sy += s_part[w].sy; t.sz += s_part[w].sz; }
    }
    float* o = partial + ((size_t)bj * gridDim.x + blockIdx.x) * 5;
    o[0] = t.m; o[1] = t.s; o[2] = t.sx; o[3] = t.sy; o[4] = t.sz;
  }
}

// one thread per (b, j): combine the splits, write the keypoint and (max, 1/sum) for pass 2
template <bool kSoftmax>
__global__ void softargmax_combine_kernel(const float* __restrict__ partial, int splits, int BJ,
                                          float* __restrict__ kp, float* __restrict__ stats) {
  const int bj = blockIdx.x * blockDim.x + threadIdx.x;
  if (bj >= BJ) return;
  const float* p = partial + (size_t)bj * splits * 5;
  SaAcc t{p[0], p[1], p[2], p[3], p[4]};
  for (int s = 1; s < splits; ++s) {
    SaAcc b{p[5 * s], p[5 * s + 1], p[5 * s + 2], p[5 * s + 3], p[5 * s + 4]};
    if (kSoftmax) sa_merge(t, b);
    else { t.s += b.s; t.sx += b.sx; t.sy += b.sy; t.sz += b.sz; }
  }
  const float inv = kSoftmax ? 1.0f / t.s : 1.0f;
  kp[3 * bj + 0] = t.sx * inv;
  kp[3 * bj + 1] = t.sy * inv;
  kp[3 * bj + 2] = t.sz * inv;
  stats[2 * bj] = t.m;
  stats[2 * bj + 1] = inv;
}

template <bool kSoftmax>
__global__ void __launch_bounds__(256) softmax_write_kernel(const float* __restrict__ logits, int N4, float mult,
                                                           const float* __restrict__ stats,
                                                           float* __restrict__ out) {
  const int bj = blockIdx.y;
  const float m = stats[2 * bj], inv = stats[2 * bj + 1];
  const float4* src = reinterpret_cast<const float4*>(logits) + (size_t)bj * N4;
  float4* dst = reinterpret_cast<float4*>(out) + (size_t)bj * N4;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N4; i += gridDim.x * blockDim.x) {
    const float4 v = __ldcs(src + i);
    float4 o;
    if (kSoftmax) {
      o.x = exp2f((v.x * mult - m) * kLog2e) * inv;
      o.y = exp2f((v.y * mult - m) * kLog2e) * inv;
      o.z = exp2f((v.z * mult - m) * kLog2e) * inv;
      o.w = exp2f((v.w * mult - m) * kLog2e) * inv;
    } else {
      o.x = fmaxf(v.x * mult, 0.f); o.y = fmaxf(v.y * mult, 0.f);
      o.z = fmaxf(v.z * mult, 0.f); o.w = fmaxf(v.w * mult, 0.f);
    }
    __stcs(dst + i, o);
  }
}

static int sa_splits(int BJ, int N, int* chunk_out) {
  // ~6 CTAs of 256 threads are resident per SM: aim for >= 8 full waves so the last partial wave costs little
  // (one CTA per joint volume left 960 CTAs = 1.08 waves at B = 64: the tail doubled the time)
  int splits = (48 * kNumSMs + BJ - 1) / BJ;
  if (splits < 1) splits = 1;
  if (splits > SA_MAX_SPLITS) splits = SA_MAX_SPLITS;
  const int unit = SA_THREADS * 16;  // elements one CTA iteration covers
  int chunk = ((N + splits - 1) / splits + unit - 1) / unit * unit;
  splits = (N + chunk - 1) / chunk;
  *chunk_out = chunk;
  return splits;
}

}  // namespace sceneego

using namespace sceneego;

extern "C" size_t sceneego_softargmax_workspace_bytes(int batch, int joints, int /*volume_size*/) {
  return (size_t)batch * joints * (SA_MAX_SPLITS * 5 + 2) * sizeof(float);
}

extern "C" int sceneego_softargmax3d_f32(const float* d_logits, int batch, int joints, int V, float mult,
                                         int softmax, const float* d_axis, const float* d_coords,
                                         float* d_kp, float* d_vol_out, void* d_ws, void* stream) {
  SE_REQUIRE(d_logits && d_kp && d_ws, "softargmax: null argument");
  SE_REQUIRE((d_axis != nullptr) != (d_coords != nullptr), "softargmax: exactly one of d_axis / d_coords");
  SE_REQUIRE(batch > 0 && joints > 0 && (long long)batch * joints <= 65535, "softargmax: bad batch/joints");
  SE_REQUIRE(V > 0 && V % 4 == 0 && V <= 1024, "softargmax: volume_size must be a multiple of 4");
  const int N = V * V * V, BJ = batch * joints;
  int chunk;
  const int splits = sa_splits(BJ, N, &chunk);
  float* partial = (float*)d_ws;
  float* stats = partial + (size_t)BJ * SA_MAX_SPLITS * 5;
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(splits, BJ);
  const size_t smem = d_axis ? 3 * V * sizeof(float) : 0;
  int log2v = -1;
  for (int k = 0; k < 12; ++k) if ((1 << k) == V) log2v = k;
  if (softmax) {
    if (d_axis) softargmax_partial_kernel<true, true><<<grid, SA_THREADS, smem, st>>>(d_logits, N, V, log2v, chunk, mult, d_axis, nullptr, partial);
    else softargmax_partial_kernel<true, false><<<grid, SA_THREADS, 0, st>>>(d_logits, N, V, log2v, chunk, mult, nullptr, d_coords, partial);
    softargmax_combine_kernel<true><<<(BJ + 127) / 128, 128, 0, st>>>(partial, splits, BJ, d_kp, stats);
  } else {
    if (d_axis) softargmax_partial_kernel<false, true><<<grid, SA_THREADS, smem, st>>>(d_logits, N, V, log2v, chunk, mult, d_axis, nullptr, partial);
    else softargmax_partial_kernel<false, false><<<grid, SA_THREADS, 0, st>>>(d_logits, N, V, log2v, chunk, mult, nullptr, d_coords, partial);
    softargmax_combine_kernel<false><<<(BJ + 127) / 128, 128, 0, st>>>(partial, splits, BJ, d_kp, stats);
  }
  SE_CUDA_LAUNCH_CHECK("softargmax");
  if (d_vol_out) {
    dim3 g2(min(256, (N / 4 + 255) / 256), BJ);
    if (softmax) softmax_write_kernel<true><<<g2, 256, 0, st>>>(d_logits, N / 4, mult, stats, d_vol_out);
    else softmax_write_kernel<false><<<g2, 256, 0, st>>>(d_logits, N / 4, mult, stats, d_vol_out);
    SE_CUDA_LAUNCH_CHECK("softmax_write");
  }
  return SCENEEGO_OK;
}
