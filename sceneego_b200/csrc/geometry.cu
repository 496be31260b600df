// Camera tables, depth-map voxelisation (a4/a5) and fused unprojection (a1-a3, a6).
// All kernels here are HBM-bound byte/float work: coalesced, vectorised, no tensor cores.
#include "common.cuh"
#include <math.h>

namespace sceneego {

// ---------------------------------------------------------------------------
// a4: unit ray per pixel, fp64, bit-identical to the NumPy reference
// (utils/fisheye/FishEyeCalibrated.py:42-50).  No FMA contraction anywhere.
// ---------------------------------------------------------------------------
__global__ void ray_table_kernel(CalibDev cal, double* __restrict__ ray) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  if (x >= cal.width) return;
  const double xc = __dsub_rn((double)x, cal.cx);
  const double yc = __dsub_rn((double)y, cal.cy);
  const double r2 = __dadd_rn(__dmul_rn(xc, xc), __dmul_rn(yc, yc));
  const double d = sqrt(r2);
  double z = 0.0;  // np.polyval: y = y*x + c, highest power first
#pragma unroll
  for (int i = 6; i >= 0; --i) z = __dadd_rn(__dmul_rn(z, d), cal.c2w[i]);
  const double nz = -z;
  const double norm = sqrt(__dadd_rn(r2, __dmul_rn(nz, nz)));
  double* o = ray + ((size_t)y * cal.width + x) * 3;
  o[0] = __ddiv_rn(xc, norm);
  o[1] = __ddiv_rn(yc, norm);
  o[2] = __ddiv_rn(nz, norm);
}

// ---------------------------------------------------------------------------
// a3: voxel centre -> pixel (Scaramuzza W2C polynomial), fp32 like the reference
// (utils/fisheye/FishEyeCalibrated.py:147-174).  Shared by the table builder and
// by the fused gather kernel.
// ---------------------------------------------------------------------------
struct W2CF32 {
  float a[11];
  float cx, cy;
};

__device__ __forceinline__ bool project_voxel(const W2CF32& k, float X, float Y, float Z, float& px, float& py) {
  const float z = __fmul_rn(Z, -1.0f);
  const float r = sqrtf(__fadd_rn(__fmul_rn(X, X), __fmul_rn(Y, Y)));
  if (r == 0.0f) { px = k.cx; py = k.cy; return false; }
  const float theta = atanf(__fdiv_rn(z, r));
  const float inv = __fdiv_rn(1.0f, r);
  float rho = k.a[0];
  float t = 1.0f;
#pragma unroll
  for (int i = 1; i < 11; ++i) {
    t = __fmul_rn(t, theta);
    rho = __fadd_rn(rho, __fmul_rn(t, k.a[i]));
  }
  px = __fadd_rn(__fmul_rn(__fmul_rn(X, inv), rho), k.cx);
  py = __fadd_rn(__fmul_rn(__fmul_rn(Y, inv), rho), k.cy);
  return true;
}

__device__ __forceinline__ void normalise_px(float px, float py, int hm_h, int hm_w, float& gx, float& gy) {
  // utils/op.py:179-180: g = 2 * (p / [W,H] - 0.5)
  gx = __fmul_rn(2.0f, __fsub_rn(__fdiv_rn(px, (float)hm_w), 0.5f));
  gy = __fmul_rn(2.0f, __fsub_rn(__fdiv_rn(py, (float)hm_h), 0.5f));
}

static W2CF32 make_w2c(const sceneego_calib_t* c) {
  W2CF32 k;
  for (int i = 0; i < 11; ++i) k.a[i] = (float)c->w2c[i];
  k.cx = (float)c->cx;
  k.cy = (float)c->cy;
  return k;
}

__global__ void project_voxels_kernel(W2CF32 k, int V, float lo, float step, int hm_h, int hm_w,
                                      float* __restrict__ px_out, float* __restrict__ grid_out,
                                      int* __restrict__ status) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= V * V * V) return;
  const int z = n % V, y = (n / V) % V, x = n / (V * V);
  float px, py;
  const bool ok = project_voxel(k, voxel_coord(lo, step, x), voxel_coord(lo, step, y),
                                voxel_coord(0.0f, step, z), px, py);
  if (!ok && status) atomicExch(status, 1);
  if (px_out) { px_out[2 * n] = px; px_out[2 * n + 1] = py; }
  if (grid_out) {
    float gx, gy;
    normalise_px(px, py, hm_h, hm_w, gx, gy);
    grid_out[2 * n] = gx;
    grid_out[2 * n + 1] = gy;
  }
}

// Arbitrary points (N,3) -> pixels (N,2): FishEyeCameraCalibrated.world2camera_pytorch.
__global__ void world2camera_kernel(W2CF32 k, const float* __restrict__ pts, int n_pts, float* __restrict__ px_out,
                                    int* __restrict__ status) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n_pts) return;
  float px, py;
  const bool ok = project_voxel(k, pts[3 * n], pts[3 * n + 1], pts[3 * n + 2], px, py);
  if (!ok && status) atomicExch(status, 1);
  px_out[2 * n] = px;
  px_out[2 * n + 1] = py;
}

// Generic F.grid_sample(bilinear, zeros, align_corners=True) on an NCHW f32 image with a grid
// shared by the batch (utils/op.py:194-214 called on a materialised feature map).  One thread =
// one sample point, looping over channels; consecutive points are neighbours in the image.
__global__ void __launch_bounds__(256) grid_sample_kernel(const float* __restrict__ img, const float* __restrict__ grid,
                                                         int64_t grid_batch_stride, int C, int H, int W, int N,
                                                         float* __restrict__ out) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (n >= N) return;
  const float2 g = reinterpret_cast<const float2*>(grid + (size_t)b * grid_batch_stride)[n];
  const float ix = __fmul_rn(__fdiv_rn(__fadd_rn(g.x, 1.0f), 2.0f), (float)(W - 1));
  const float iy = __fmul_rn(__fdiv_rn(__fadd_rn(g.y, 1.0f), 2.0f), (float)(H - 1));
  const float x0f = floorf(ix), y0f = floorf(iy);
  const float wx1 = ix - x0f, wy1 = iy - y0f, wx0 = (x0f + 1.0f) - ix, wy0 = (y0f + 1.0f) - iy;
  // clamped before the conversion: far outside (|g| ~ 1e30) (int) saturates at INT_MAX and x0 + 1 would overflow,
  // which the compiler may fold into a bounds test that passes; a clamped corner keeps both taps outside
  const int x0 = (int)fminf(fmaxf(x0f, -2.0f), (float)W), y0 = (int)fminf(fmaxf(y0f, -2.0f), (float)H);
  float wt[4];
  int off[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const int X = x0 + (t & 1), Y = y0 + (t >> 1);
    const bool inb = X >= 0 && X < W && Y >= 0 && Y < H;
    wt[t] = inb ? ((t & 1) ? wx1 : wx0) * ((t >> 1) ? wy1 : wy0) : 0.f;
    off[t] = inb ? Y * W + X : 0;
  }
  const float* ib = img + (size_t)b * C * H * W;
  for (int c = 0; c < C; ++c) {
    const float* pl = ib + (size_t)c * H * W;
    const float v = __ldg(pl + off[0]) * wt[0] + __ldg(pl + off[1]) * wt[1] + __ldg(pl + off[2]) * wt[2] +
                    __ldg(pl + off[3]) * wt[3];
    __stcs(out + ((size_t)b * C + c) * N + n, v);
  }
}

// ---------------------------------------------------------------------------
// a1: 1x1 Conv2d 256 -> 32 (+bias), NCHW f32 in, channel-last f32 out.  HBM-bound (4.2 MB read per frame).
// One CTA = 128 pixels x 32 output channels; each thread owns a 4 pixel x 4 channel register tile, so one
// LDS.128 of inputs and one of weights feed 16 FMAs (the first version: 9 shared loads per 8 FMAs, 1.3 TB/s).
// K is streamed through shared memory in chunks of 32 channels; the next chunk's global loads are in flight
// while the current one is multiplied.  Same accumulation order as a sequential dot product (k ascending, fmaf).
// ---------------------------------------------------------------------------
constexpr int FC_PIX = 128, FC_KC = 32, FC_CO = 32;

__global__ void __launch_bounds__(256) feature_conv1x1_kernel(const float* __restrict__ feat,
                                                             const float* __restrict__ weight,
                                                             const float* __restrict__ bias,
                                                             float* __restrict__ out, int cin, int hw) {
  __shared__ __align__(16) float s_in[FC_KC][FC_PIX];     // [k][pixel]
  __shared__ __align__(16) float s_w[FC_KC][FC_CO];       // [k][co]
  const int b = blockIdx.y;
  const int pix0 = blockIdx.x * FC_PIX;
  const int tid = threadIdx.x;
  const int cg = tid & 7;          // channels 4*cg .. 4*cg+3
  const int pg = tid >> 3;         // pixels   4*pg .. 4*pg+3
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const float* fb = feat + (size_t)b * cin * hw;
  const bool vec = (hw % 4 == 0) && (pix0 + FC_PIX <= hw);
  float4 rin[4];
  float rw[4];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = tid + 256 * i;                   // float4 index inside the [32][128] chunk
      const int kk = e >> 5, p4 = (e & 31) * 4;
      const float* src = fb + (size_t)(k0 + kk) * hw + pix0 + p4;
      if (vec) rin[i] = __ldcs(reinterpret_cast<const float4*>(src));
      else {
        rin[i].x = pix0 + p4 + 0 < hw ? src[0] : 0.f; rin[i].y = pix0 + p4 + 1 < hw ? src[1] : 0.f;
        rin[i].z = pix0 + p4 + 2 < hw ? src[2] : 0.f; rin[i].w = pix0 + p4 + 3 < hw ? src[3] : 0.f;
      }
      // weight element kk = e / 32, co = e % 32: lanes walk co, so the shared-memory store below is conflict-free
      // (the 32 KB weight matrix is L2-resident; its strided 4-byte reads do not matter)
      rw[i] = weight[(size_t)(e & 31) * cin + k0 + (e >> 5)];
    }
  };
  fetch(0);
  for (int k0 = 0; k0 < cin; k0 += FC_KC) {
    __syncthreads();                                 // the previous chunk has been consumed
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = tid + 256 * i;
      *reinterpret_cast<float4*>(&s_in[e >> 5][(e & 31) * 4]) = rin[i];
      s_w[e >> 5][e & 31] = rw[i];
    }
    __syncthreads();
    if (k0 + FC_KC < cin) fetch(k0 + FC_KC);
#pragma unroll 8
    for (int kk = 0; kk < FC_KC; ++kk) {
      const float4 x = *reinterpret_cast<const float4*>(&s_in[kk][4 * pg]);
      const float4 w = *reinterpret_cast<const float4*>(&s_w[kk][4 * cg]);
      const float xs[4] = {x.x, x.y, x.z, x.w}, ws[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(xs[i], ws[j], acc[i][j]);
    }
  }
  const float4 bv = make_float4(bias[4 * cg], bias[4 * cg + 1], bias[4 * cg + 2], bias[4 * cg + 3]);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int p = pix0 + 4 * pg + i;
    if (p < hw)
      *reinterpret_cast<float4*>(out + ((size_t)b * hw + p) * FC_CO + 4 * cg) =
          make_float4(acc[i][0] + bv.x, acc[i][1] + bv.y, acc[i][2] + bv.z, acc[i][3] + bv.w);
  }
}

// Output #2 of the reference forward: nearest upsample + pad, materialised only on request.
// Pure write bandwidth (168 MB per frame).  One CTA = one (frame, channel, source row): the
// up/h identical output rows are built once in registers (one float4 per thread) and stored
// up/h times with streaming stores.
__global__ void __launch_bounds__(320) upsample_pad_kernel(const float* __restrict__ in, float* __restrict__ out, int c,
                                                          int h, int w, int up, int pad) {
  const int W = up + 2 * pad;
  const int sy = blockIdx.x;
  const int bc = blockIdx.y;
  const int b = bc / c, ch = bc % c;
  const int rows = up / h;                       // output rows fed by one source row
  const float* src = in + (((size_t)b * h + sy) * w) * c + ch;
  for (int x4 = threadIdx.x * 4; x4 < W; x4 += blockDim.x * 4) {
    float v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int x = x4 + i - pad;
      v[i] = (x >= 0 && x < up) ? __ldg(src + (size_t)(int)(((long long)x * w) / up) * c) : 0.f;
    }
    const float4 o = make_float4(v[0], v[1], v[2], v[3]);
    float* dst = out + ((size_t)bc * up + (size_t)sy * rows) * W + x4;
    for (int r = 0; r < rows; ++r) __stcs(reinterpret_cast<float4*>(dst + (size_t)r * W), o);
  }
}

// ---------------------------------------------------------------------------
// a2/a3/a6: fused (projection +) bilinear gather.
// One thread = one voxel, all 32 channels.  The x16-upsampled, zero-padded image of the
// reference is never materialised: tap (X,Y) of the virtual img_h x img_w plane maps to
// source cell (Y*h/img_h, (X-pad)*w/up).  Channel-last f32 source rows are read as float4
// (8 x 16 B per tap); consecutive voxels (z fastest) project to neighbouring pixels, so
// the 512 KB per-frame source stays in L1/L2.  Stores: f32 NCDHW (128 B per warp per
// channel) and/or bf16 planar padded (512 B per warp per channel group).
// ---------------------------------------------------------------------------
// The two halves of unproject_kernel for unproject_cameras_kernel below.  A voxel's geometry: its projection, the four
// bilinear taps of the virtual image plane and their weights, taps that share a source cell merged (cell -1 = nothing
// to fetch); frame-invariant for one camera.  Same steps, in the same order, as unproject_kernel, which keeps its own
// inline copy: calling these helpers from it moved its register allocation (fused form).
template <bool kProject>
__device__ __forceinline__ void unproject_taps(const float* __restrict__ grid, const W2CF32& cam, int n, int vx, int vy,
                                               int vz, int h, int w, float lo, float step, int img_h, int img_w,
                                               int up_shift_y, int up_shift_x, int (&cell)[4], float (&wt)[4]) {
  float gx, gy;
  if (kProject) {
    float px, py;
    project_voxel(cam, voxel_coord(lo, step, vx), voxel_coord(lo, step, vy), voxel_coord(0.0f, step, vz), px, py);
    normalise_px(px, py, img_h, img_w, gx, gy);
  } else {
    const float2 g = reinterpret_cast<const float2*>(grid)[n];
    gx = g.x; gy = g.y;
  }
  // ATen grid_sampler_2d, align_corners=True: ix = ((g+1)/2)*(W-1)
  const float ix = __fmul_rn(__fdiv_rn(__fadd_rn(gx, 1.0f), 2.0f), (float)(img_w - 1));
  const float iy = __fmul_rn(__fdiv_rn(__fadd_rn(gy, 1.0f), 2.0f), (float)(img_h - 1));
  const float x0f = floorf(ix), y0f = floorf(iy);
  const float wx1 = ix - x0f, wy1 = iy - y0f;
  const float wx0 = (x0f + 1.0f) - ix, wy0 = (y0f + 1.0f) - iy;
  const int x0 = (int)fminf(fmaxf(x0f, -2.0f), (float)img_w), y0 = (int)fminf(fmaxf(y0f, -2.0f), (float)img_h);   // as in grid_sample_kernel
  const int pad = (img_w - img_h) / 2;

  // The image plane is the 16x nearest-upsampled source, so the four bilinear taps usually (88 % of the
  // voxels at V = 64) fall into ONE source cell: taps are merged per source cell and each distinct
  // 128-byte cell is fetched once (the gather is L2-bandwidth-bound otherwise).
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const int X = x0 + (t & 1), Y = y0 + (t >> 1);
    wt[t] = ((t & 1) ? wx1 : wx0) * ((t >> 1) ? wy1 : wy0);
    const bool inb = (X >= 0) && (X < img_w) && (Y >= 0) && (Y < img_h);   // zeros padding
    const int xs = X - pad;
    cell[t] = -1;
    if (inb && xs >= 0 && xs < img_h) {                                    // outside: ConstantPad2d zeros
      // nearest source cell: Y * h / img_h.  The 64-bit divisions here (eight per voxel, ~100 instructions each)
      // were what bounded the kernel; 1024 / 64 is a power of two, otherwise the 32-bit quotient is exact too
      // (Y * h < 2^31, checked on the host)
      const int sy = up_shift_y >= 0 ? (Y >> up_shift_y) : (int)((unsigned)(Y * h) / (unsigned)img_h);
      const int sx = up_shift_x >= 0 ? (xs >> up_shift_x) : (int)((unsigned)(xs * w) / (unsigned)img_h);
      cell[t] = sy * w + sx;
    }
  }
#pragma unroll
  for (int t = 1; t < 4; ++t)
#pragma unroll
    for (int u = 0; u < t; ++u)
      if (cell[t] >= 0 && cell[t] == cell[u]) { wt[u] += wt[t]; cell[t] = -1; }
}

// One frame of one voxel: the merged taps applied to frame b's 32 channels, stored in every requested form.
__device__ __forceinline__ void unproject_frame(const float* __restrict__ feat, int b, int h, int w, int n, int N, int vx,
                                                int vy, int vz, const int (&cell)[4], const float (&wt)[4],
                                                float* __restrict__ out_f32, __nv_bfloat16* __restrict__ out_bf16,
                                                const sceneego_vol_layout_t& lay, int extra_zero_planes) {
  constexpr int C = 32;
  float acc[C];
#pragma unroll
  for (int c = 0; c < C; ++c) acc[c] = 0.f;
  const float* fb = feat + (size_t)b * h * w * C;
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    if (cell[t] >= 0) {
      // 256-bit loads (sm_100): a warp's lanes fall into ~6 distinct 128-byte source cells, and every load
      // instruction costs one L1 wavefront per distinct cell whatever its width -- the L1 data pipe, not DRAM,
      // bounds this kernel (ncu: 80 % of peak with 128-bit loads), so half as many instructions for the same bytes
      const float* src = fb + (size_t)cell[t] * C;
      const float w_t = wt[t];
#pragma unroll
      for (int q = 0; q < C / 8; ++q) {
        float v[8];
        asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
                     : "l"(src + 8 * q));
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[8 * q + i] = fmaf(v[i], w_t, acc[8 * q + i]);
      }
    }
  }
  if (out_f32) {
    float* o = out_f32 + (size_t)b * C * N + n;
#pragma unroll
    for (int c = 0; c < C; ++c) __stcs(o + (size_t)c * N, acc[c]);
  }
  if (out_bf16) {
    const int64_t cell0 = vol_cell(lay, b, vx, vy, vz, 0, C / 8);
#pragma unroll
    for (int g = 0; g < C / 8; ++g) {
      *reinterpret_cast<uint4*>(out_bf16 + (cell0 + (int64_t)g * lay.plane_stride) * 8) =
          make_uint4(act_pack2(acc[8 * g + 0], acc[8 * g + 1]), act_pack2(acc[8 * g + 2], acc[8 * g + 3]),
                     act_pack2(acc[8 * g + 4], acc[8 * g + 5]), act_pack2(acc[8 * g + 6], acc[8 * g + 7]));
    }
    // scene-occupancy plane(s) behind the features: cleared here, set by voxelize_kernel
    if (lay.s2d) {
      // one cell per 2x2x2 block holds the block's 8 occupancy values: the even-even-even voxel clears it
      if (extra_zero_planes > 0 && ((vx | vy | vz) & 1) == 0)
        *reinterpret_cast<uint4*>(out_bf16 + (vol_scene_elem(lay, b, vx, vy, vz, C / 8) & ~(int64_t)7)) = make_uint4(0, 0, 0, 0);
    } else {
      for (int g = C / 8; g < C / 8 + extra_zero_planes; ++g)
        *reinterpret_cast<uint4*>(out_bf16 + (cell0 + (int64_t)g * lay.plane_stride) * 8) = make_uint4(0, 0, 0, 0);
    }
  }
}

template <bool kProject>
__global__ void __launch_bounds__(128) unproject_kernel(const float* __restrict__ feat, const float* __restrict__ grid,
                                                       W2CF32 cam, int h, int w, int V, float lo, float step,
                                                       int img_h, int img_w, float* __restrict__ out_f32,
                                                       __nv_bfloat16* __restrict__ out_bf16,
                                                       sceneego_vol_layout_t lay, int extra_zero_planes,
                                                       int up_shift_y, int up_shift_x, int log2v, int batch,
                                                       int frames_per_thread) {
  constexpr int C = 32;
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  const int N = V * V * V;
  if (n >= N) return;
  // power-of-two sides: shifts instead of runtime integer divisions
  const int vz = log2v >= 0 ? (n & (V - 1)) : n % V;
  const int vy = log2v >= 0 ? ((n >> log2v) & (V - 1)) : (n / V) % V;
  const int vx = log2v >= 0 ? (n >> (2 * log2v)) : n / (V * V);
  float gx, gy;
  if (kProject) {
    float px, py;
    project_voxel(cam, voxel_coord(lo, step, vx), voxel_coord(lo, step, vy), voxel_coord(0.0f, step, vz), px, py);
    normalise_px(px, py, img_h, img_w, gx, gy);
  } else {
    const float2 g = reinterpret_cast<const float2*>(grid)[n];
    gx = g.x; gy = g.y;
  }
  // ATen grid_sampler_2d, align_corners=True: ix = ((g+1)/2)*(W-1)
  const float ix = __fmul_rn(__fdiv_rn(__fadd_rn(gx, 1.0f), 2.0f), (float)(img_w - 1));
  const float iy = __fmul_rn(__fdiv_rn(__fadd_rn(gy, 1.0f), 2.0f), (float)(img_h - 1));
  const float x0f = floorf(ix), y0f = floorf(iy);
  const float wx1 = ix - x0f, wy1 = iy - y0f;
  const float wx0 = (x0f + 1.0f) - ix, wy0 = (y0f + 1.0f) - iy;
  const int x0 = (int)fminf(fmaxf(x0f, -2.0f), (float)img_w), y0 = (int)fminf(fmaxf(y0f, -2.0f), (float)img_h);   // as in grid_sample_kernel
  const int pad = (img_w - img_h) / 2;

  // The image plane is the 16x nearest-upsampled source, so the four bilinear taps usually (88 % of the
  // voxels at V = 64) fall into ONE source cell: taps are merged per source cell and each distinct
  // 128-byte cell is fetched once (the gather is L2-bandwidth-bound otherwise).
  int cell[4];
  float wt[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const int X = x0 + (t & 1), Y = y0 + (t >> 1);
    wt[t] = ((t & 1) ? wx1 : wx0) * ((t >> 1) ? wy1 : wy0);
    const bool inb = (X >= 0) && (X < img_w) && (Y >= 0) && (Y < img_h);   // zeros padding
    const int xs = X - pad;
    cell[t] = -1;
    if (inb && xs >= 0 && xs < img_h) {                                    // outside: ConstantPad2d zeros
      // nearest source cell: Y * h / img_h.  The 64-bit divisions here (eight per voxel, ~100 instructions each)
      // were what bounded the kernel; 1024 / 64 is a power of two, otherwise the 32-bit quotient is exact too
      // (Y * h < 2^31, checked on the host)
      const int sy = up_shift_y >= 0 ? (Y >> up_shift_y) : (int)((unsigned)(Y * h) / (unsigned)img_h);
      const int sx = up_shift_x >= 0 ? (xs >> up_shift_x) : (int)((unsigned)(xs * w) / (unsigned)img_h);
      cell[t] = sy * w + sx;
    }
  }
#pragma unroll
  for (int t = 1; t < 4; ++t)
#pragma unroll
    for (int u = 0; u < t; ++u)
      if (cell[t] >= 0 && cell[t] == cell[u]) { wt[u] += wt[t]; cell[t] = -1; }
  // the voxel's geometry (projection, taps, weights) is frame-invariant: it is computed once and applied to
  // `frames_per_thread` frames (it was two thirds of the kernel's instructions when every frame recomputed it)
  for (int b = blockIdx.y * frames_per_thread; b < min(batch, (int)(blockIdx.y + 1) * frames_per_thread); ++b) {
  float acc[C];
#pragma unroll
  for (int c = 0; c < C; ++c) acc[c] = 0.f;
  const float* fb = feat + (size_t)b * h * w * C;
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    if (cell[t] >= 0) {
      // 256-bit loads (sm_100): a warp's lanes fall into ~6 distinct 128-byte source cells, and every load
      // instruction costs one L1 wavefront per distinct cell whatever its width -- the L1 data pipe, not DRAM,
      // bounds this kernel (ncu: 80 % of peak with 128-bit loads), so half as many instructions for the same bytes
      const float* src = fb + (size_t)cell[t] * C;
      const float w_t = wt[t];
#pragma unroll
      for (int q = 0; q < C / 8; ++q) {
        float v[8];
        asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
                     : "l"(src + 8 * q));
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[8 * q + i] = fmaf(v[i], w_t, acc[8 * q + i]);
      }
    }
  }
  if (out_f32) {
    float* o = out_f32 + (size_t)b * C * N + n;
#pragma unroll
    for (int c = 0; c < C; ++c) __stcs(o + (size_t)c * N, acc[c]);
  }
  if (out_bf16) {
    const int64_t cell0 = vol_cell(lay, b, vx, vy, vz, 0, C / 8);
#pragma unroll
    for (int g = 0; g < C / 8; ++g) {
      *reinterpret_cast<uint4*>(out_bf16 + (cell0 + (int64_t)g * lay.plane_stride) * 8) =
          make_uint4(act_pack2(acc[8 * g + 0], acc[8 * g + 1]), act_pack2(acc[8 * g + 2], acc[8 * g + 3]),
                     act_pack2(acc[8 * g + 4], acc[8 * g + 5]), act_pack2(acc[8 * g + 6], acc[8 * g + 7]));
    }
    // scene-occupancy plane(s) behind the features: cleared here, set by voxelize_kernel
    if (lay.s2d) {
      // one cell per 2x2x2 block holds the block's 8 occupancy values: the even-even-even voxel clears it
      if (extra_zero_planes > 0 && ((vx | vy | vz) & 1) == 0)
        *reinterpret_cast<uint4*>(out_bf16 + (vol_scene_elem(lay, b, vx, vy, vz, C / 8) & ~(int64_t)7)) = make_uint4(0, 0, 0, 0);
    } else {
      for (int g = C / 8; g < C / 8 + extra_zero_planes; ++g)
        *reinterpret_cast<uint4*>(out_bf16 + (cell0 + (int64_t)g * lay.plane_stride) * 8) = make_uint4(0, 0, 0, 0);
    }
  }
  }   // frames
}

// A camera per frame: frame b is seen through camera frame_camera[b] (grid row frame_camera[b] of the stacked (K,N,2)
// tables, or coefficient set frame_camera[b] of `cams`).  The block's frame range is taken in `frame_order` (NULL =
// identity; the host passes a stable sort by camera, so frames that share a camera are adjacent) and a thread
// recomputes the voxel's geometry only when the camera changes between consecutive frames of its range; the camera is
// uniform over the block, so the change is too.  Outputs go to the frame's own slot.
struct W2CSet {
  W2CF32 k[SCENEEGO_MAX_CAMERAS];
};

template <bool kProject>
__global__ void __launch_bounds__(128) unproject_cameras_kernel(const float* __restrict__ feat,
                                                               const float* __restrict__ grids,
                                                               const __grid_constant__ W2CSet cams,
                                                               const int* __restrict__ frame_camera,
                                                               const int* __restrict__ frame_order, int h, int w, int V,
                                                               float lo, float step, int img_h, int img_w,
                                                               float* __restrict__ out_f32,
                                                               __nv_bfloat16* __restrict__ out_bf16,
                                                               sceneego_vol_layout_t lay, int extra_zero_planes,
                                                               int up_shift_y, int up_shift_x, int log2v, int batch,
                                                               int frames_per_thread) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  const int N = V * V * V;
  if (n >= N) return;
  const int vz = log2v >= 0 ? (n & (V - 1)) : n % V;
  const int vy = log2v >= 0 ? ((n >> log2v) & (V - 1)) : (n / V) % V;
  const int vx = log2v >= 0 ? (n >> (2 * log2v)) : n / (V * V);
  int cell[4];
  float wt[4];
  int cur = -1;
  for (int p = blockIdx.y * frames_per_thread; p < min(batch, (int)(blockIdx.y + 1) * frames_per_thread); ++p) {
    const int b = frame_order ? __ldg(frame_order + p) : p;
    const int k = __ldg(frame_camera + b);
    if (k != cur) {
      cur = k;
      unproject_taps<kProject>(kProject ? grids : grids + (size_t)k * N * 2, cams.k[k], n, vx, vy, vz, h, w, lo, step, img_h, img_w,
                               up_shift_y, up_shift_x, cell, wt);
    }
    unproject_frame(feat, b, h, w, n, N, vx, vy, vz, cell, wt, out_f32, out_bf16, lay, extra_zero_planes);
  }
}

// ---------------------------------------------------------------------------
// a5: back-project every pixel of the (nearest-resized, padded) depth map and scatter
// occupancy.  fp64, round-half-even, exactly the NumPy order of
// network/voxel_net_depth.py:199-217.  One thread = one pixel of the img_h x img_w plane,
// row-major, so depth, ray table (24 B / pixel, L2 resident across frames) and the
// zero-padding test are all coalesced.  The scatter is a benign same-value race.
// ---------------------------------------------------------------------------
// Nearest-neighbour index maps exactly as OpenCV builds them (resizeNN): src = min(cvFloor(dst * ifx), n_src - 1)
// with ifx = 1.0 / ((double)n_dst / n_src) evaluated in fp64 on the host -- NOT floor(dst * n_src / n_dst) in exact
// arithmetic, which differs from cv2 for 115 source sizes below 1400 (e.g. 26 -> 1280).  Two maps are composed:
// the model's resize to img_h x img_h (network/voxel_net_depth.py:197) after the dataset's optional resize of the
// raw map to pre_h x pre_w (dataset/demo_dataset.py:86-88, dataset/test_dataset.py:138-140); identity when equal.
struct NearestMaps {
  double ify1, ifx1;   // img_h grid -> (pre_h, pre_w) grid
  double ify0, ifx0;   // (pre_h, pre_w) grid -> raw (h, w) grid
  int pre_h, pre_w;
  float clamp_max;     // depth_map[depth_map > clamp_max] = clamp_max (demo_dataset.py:91); +inf = off
};

// One occupied voxel into the planar bf16 V2V input (three storage forms, include/sceneego_b200.h).
__device__ __forceinline__ void set_occupied(__nv_bfloat16* __restrict__ occ, const sceneego_vol_layout_t& lay, int b, int x,
                                             int y, int z, int channel, int V) {
  const __nv_bfloat16 one = act_from_float(1.0f);
  if (lay.zwin) {
    // z-window plane: entry e of cell (x,y,zc) is occ[x][y][zc-3+e] -> this voxel is entry e of the cells zc = z+3-e
    const int64_t base = ((int64_t)(channel >> 3) * lay.plane_stride + vol_pos(lay, b, x, y, 0)) * 8;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int zc = z + 3 - e;
      if (zc >= 0 && zc < V) occ[base + (int64_t)zc * 8 + e] = one;
    }
  } else {
    occ[vol_scene_elem(lay, b, x, y, z, channel >> 3) + (lay.s2d ? 0 : (channel & 7))] = one;
  }
}

// Round-to-nearest arithmetic of one precision, never contracted to FMA: the quantisation below is instantiated in
// fp64 (depth maps; float64 clouds) and in fp32 (float32 clouds, which NumPy and torch keep in float32 when a Python
// float is added or multiplied in).
template <typename T> struct RnOps;
template <> struct RnOps<double> {
  static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
  static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
  static __device__ __forceinline__ double div(double a, double b) { return __ddiv_rn(a, b); }
  static __device__ __forceinline__ double round_even(double a) { return rint(a); }
};
template <> struct RnOps<float> {
  static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
  static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
  static __device__ __forceinline__ float div(float a, float b) { return __fdiv_rn(a, b); }
  static __device__ __forceinline__ float round_even(float a) { return rintf(a); }
};

// kPow2Side: 0 = divide by the cuboid side; 1 = the side is a power of two (x / 2^k == x * 2^-k exactly); 2 = the side AND
// the volume size are powers of two: (x * V) * 2^-k == x * (V * 2^-k) exactly (both are exponent shifts), one multiply
//
// One camera-space point -> its voxel, point_cloud_to_voxel_numpy (network/voxel_net_depth.py:207-222) in the
// reference's order: q_xy = ((p + s/2) * V) / s, q_z = (p_z * V) / s, round half-to-even, kept iff 0 <= q <= V-1 on all
// three axes (-0.0 passes, as in NumPy; NaN / inf fail every comparison).  half = s/2, Vd = V, hi = V-1 in precision T.
// voxelize_kernel keeps its own inline copy of the same fp64 steps: calling this helper from it changed that kernel's
// SASS (its instruction count moved by up to 32 per instantiation in each form of the call tried).
template <int kPow2Side, typename T>
__device__ __forceinline__ bool quantize_point(T x, T y, T z, T half, T Vd, T side, T inv_side, T hi, int& ix, int& iy,
                                               int& iz) {
  using R = RnOps<T>;
  const T mul = kPow2Side == 2 ? R::mul(Vd, inv_side) : Vd;     // exact: a power of two either way
  T qx = R::mul(R::add(x, half), mul);
  T qy = R::mul(R::add(y, half), mul);
  T qz = R::mul(z, mul);
  if (kPow2Side == 2) {
  } else if (kPow2Side == 1) {   // x / 2^k == x * 2^-k exactly (no divide on the hot path)
    qx = R::mul(qx, inv_side); qy = R::mul(qy, inv_side); qz = R::mul(qz, inv_side);
  } else {
    qx = R::div(qx, side); qy = R::div(qy, side); qz = R::div(qz, side);
  }
  qx = R::round_even(qx); qy = R::round_even(qy); qz = R::round_even(qz);
  if (qx >= T(0) && qx <= hi && qy >= T(0) && qy <= hi && qz >= T(0) && qz <= hi) {
    ix = (int)qx; iy = (int)qy; iz = (int)qz;
    return true;
  }
  return false;
}

template <int kPow2Side>
__global__ void __launch_bounds__(256) voxelize_kernel(const float* __restrict__ depth, int h, int w, NearestMaps nm,
                                                      const double* __restrict__ ray, int img_h, int img_w, int V,
                                                      double side, double inv_side, float* __restrict__ occ_f32,
                                                      __nv_bfloat16* __restrict__ occ_bf16,
                                                      sceneego_vol_layout_t lay, int channel, int batch, int frames_per_block,
                                                      int cols) {
  // threads cover the `cols` source columns only (img_h: the network's squash-and-pad of voxel_net_depth.py:197-198;
  // img_w: the dataset's pixel-for-pixel product of dataset/real_depth_utils.py:31-33); the zero-padded columns
  // (np.pad, :198) all land on the zero-depth voxel, which one thread of the launch sets when there is any padding
  const int xs = blockIdx.x * blockDim.x + threadIdx.x;
  const int Y = blockIdx.y;
  const int pad = (img_w - cols) / 2;
  const int X = xs + pad;
  const bool in_src = xs < cols;
  const bool in_img = in_src;
  // cv2.resize(INTER_NEAREST), model side then dataset side
  int sy = (int)floor(__dmul_rn((double)Y, nm.ify1));
  int sx = (int)floor(__dmul_rn((double)(in_src ? xs : 0), nm.ifx1));
  sy = sy < nm.pre_h - 1 ? sy : nm.pre_h - 1;
  sx = sx < nm.pre_w - 1 ? sx : nm.pre_w - 1;
  sy = (int)floor(__dmul_rn((double)sy, nm.ify0));
  sx = (int)floor(__dmul_rn((double)sx, nm.ifx0));
  sy = sy < h - 1 ? sy : h - 1;
  sx = sx < w - 1 ? sx : w - 1;
  // the pixel's ray is frame-invariant: fetched once for the `frames_per_block` frames this block covers
  // (the 31.5 MB table is L2-resident, but at one fetch per frame its L2 traffic, not the depth map, bounds the kernel)
  double r0 = 0.0, r1 = 0.0, r2 = 0.0;
  if (in_src) {
    const double* r = ray + ((size_t)Y * img_w + X) * 3;
    r0 = r[0]; r1 = r[1]; r2 = r[2];
  }
  const double half = side / 2;             // cuboid_side / 2
  const double Vd = (double)V;
  const double hi = (double)(V - 1);
  // every zero-depth pixel (all the padded columns, everything outside the image circle) lands on
  // ray*0 -> q = (rint((0+s/2)*V/s), same, 0)
  const double q0 = rint(kPow2Side ? __dmul_rn(__dmul_rn(half, Vd), inv_side) : __ddiv_rn(__dmul_rn(half, Vd), side));
  const bool q0_in = q0 >= 0.0 && q0 <= hi;
  const int b_begin = blockIdx.z * frames_per_block;
  // all depth values of this pixel first (up to 8 independent loads in flight), then the arithmetic: one load per
  // loop iteration behind a block-wide barrier left the kernel latency-bound at 0.9 TB/s
  constexpr int kMaxFpb = 8;
  float dvs[kMaxFpb];
#pragma unroll
  for (int f = 0; f < kMaxFpb; ++f) {
    dvs[f] = 0.f;
    if (f < frames_per_block && b_begin + f < batch && in_src) {
      const float t = __ldcs(depth + ((size_t)(b_begin + f) * h + sy) * w + sx);
      dvs[f] = t > nm.clamp_max ? nm.clamp_max : t;          // NaN compares false and stays, like NumPy's mask
    }
  }
#pragma unroll
  for (int f = 0; f < kMaxFpb; ++f) {
    const int b = b_begin + f;
    if (f >= frames_per_block || b >= batch) break;         // uniform over the block
    const float dv = dvs[f];
    int ix = -1, iy = 0, iz = 0;
    const bool zero = in_img && (dv == 0.0f);
    if (in_img && !zero) {
      const double d = (double)dv;
      const double mul = kPow2Side == 2 ? __dmul_rn(Vd, inv_side) : Vd;     // exact: a power of two either way
      double qx = __dmul_rn(__dadd_rn(__dmul_rn(r0, d), half), mul);
      double qy = __dmul_rn(__dadd_rn(__dmul_rn(r1, d), half), mul);
      double qz = __dmul_rn(__dmul_rn(r2, d), mul);
      if (kPow2Side == 2) {
      } else if (kPow2Side == 1) {   // x / 2^k == x * 2^-k exactly (no fp64 divide on the hot path)
        qx = __dmul_rn(qx, inv_side); qy = __dmul_rn(qy, inv_side); qz = __dmul_rn(qz, inv_side);
      } else {
        qx = __ddiv_rn(qx, side); qy = __ddiv_rn(qy, side); qz = __ddiv_rn(qz, side);
      }
      qx = rint(qx); qy = rint(qy); qz = rint(qz);
      if (qx >= 0.0 && qx <= hi && qy >= 0.0 && qy <= hi && qz >= 0.0 && qz <= hi) {
        ix = (int)qx; iy = (int)qy; iz = (int)qz;
      }
    }
    // one thread per block writes the zero-depth voxel when any pixel of the block has zero depth (a per-warp vote
    // instead of the block-wide one made 8x more writers hammer the same voxel: 3.6 -> 4.6 us); block (0,0,z) also
    // does it for the padded columns
    const bool any_zero = __syncthreads_or(zero ? 1 : 0) != 0 || (pad > 0 && blockIdx.x == 0 && blockIdx.y == 0);
    if (any_zero && threadIdx.x == 0 && q0_in) {
      const int c = (int)q0;
      if (occ_f32) occ_f32[(((size_t)b * V + c) * V + c) * V] = 1.0f;
      if (occ_bf16) set_occupied(occ_bf16, lay, b, c, c, 0, channel, V);
    }
    if (ix >= 0) {
      if (occ_f32) occ_f32[(((size_t)b * V + ix) * V + iy) * V + iz] = 1.0f;
      if (occ_bf16) set_occupied(occ_bf16, lay, b, ix, iy, iz, channel, V);
    }
  }
}

// A camera per frame: frame b back-projects through ray table frame_camera[b] of the stacked (K, img_h, img_w, 3) tables.
// The block's frames are taken in `frame_order` (NULL = identity; a stable sort by camera from the host), and the
// pixel's ray is reloaded only when the camera changes, so a table is still fetched once per block and camera run.  The
// fp64 steps are voxelize_kernel's (quantize_point performs them in the same order: ray * depth, + s/2, * V, / s).
// Eight blocks per SM on the power-of-two paths (32 registers, as voxelize_kernel gets): the frame order and the camera
// ids add two dependent loads in front of the ray's, and occupancy is what hides them.
template <int kPow2Side>
__global__ void __launch_bounds__(256, kPow2Side ? 8 : 1) voxelize_cameras_kernel(const float* __restrict__ depth, int h, int w,
                                                              NearestMaps nm, const double* __restrict__ rays,
                                                              const int* __restrict__ frame_camera,
                                                              const int* __restrict__ frame_order, int img_h, int img_w,
                                                              int V, double side, double inv_side,
                                                              float* __restrict__ occ_f32,
                                                              __nv_bfloat16* __restrict__ occ_bf16,
                                                              sceneego_vol_layout_t lay, int channel, int batch,
                                                              int frames_per_block, int cols) {
  const int xs = blockIdx.x * blockDim.x + threadIdx.x;
  const int Y = blockIdx.y;
  const int pad = (img_w - cols) / 2;
  const int X = xs + pad;
  const bool in_src = xs < cols;
  int sy = (int)floor(__dmul_rn((double)Y, nm.ify1));
  int sx = (int)floor(__dmul_rn((double)(in_src ? xs : 0), nm.ifx1));
  sy = sy < nm.pre_h - 1 ? sy : nm.pre_h - 1;
  sx = sx < nm.pre_w - 1 ? sx : nm.pre_w - 1;
  sy = (int)floor(__dmul_rn((double)sy, nm.ify0));
  sx = (int)floor(__dmul_rn((double)sx, nm.ifx0));
  sy = sy < h - 1 ? sy : h - 1;
  sx = sx < w - 1 ? sx : w - 1;
  const double half = side / 2;
  const double Vd = (double)V;
  const double hi = (double)(V - 1);
  const double q0 = rint(kPow2Side ? __dmul_rn(__dmul_rn(half, Vd), inv_side) : __ddiv_rn(__dmul_rn(half, Vd), side));
  const bool q0_in = q0 >= 0.0 && q0 <= hi;
  const int b_begin = blockIdx.z * frames_per_block;
  constexpr int kMaxFpb = 8;
  int fb[kMaxFpb], fk[kMaxFpb];
  float dvs[kMaxFpb];
#pragma unroll
  for (int f = 0; f < kMaxFpb; ++f) {
    dvs[f] = 0.f;
    fb[f] = -1; fk[f] = 0;
    if (f < frames_per_block && b_begin + f < batch) {
      fb[f] = frame_order ? __ldg(frame_order + b_begin + f) : b_begin + f;
      fk[f] = __ldg(frame_camera + fb[f]);
      if (in_src) {
        const float t = __ldcs(depth + ((size_t)fb[f] * h + sy) * w + sx);
        dvs[f] = t > nm.clamp_max ? nm.clamp_max : t;          // NaN compares false and stays, like NumPy's mask
      }
    }
  }
  int cur = -1;
  double r0 = 0.0, r1 = 0.0, r2 = 0.0;
#pragma unroll
  for (int f = 0; f < kMaxFpb; ++f) {
    const int b = fb[f];
    if (b < 0) break;                                        // uniform over the block
    if (fk[f] != cur) {                                      // uniform over the block as well
      cur = fk[f];
      if (in_src) {
        const double* r = rays + ((size_t)cur * img_h * img_w + (size_t)Y * img_w + X) * 3;
        r0 = r[0]; r1 = r[1]; r2 = r[2];
      }
    }
    const float dv = dvs[f];
    int ix = -1, iy = 0, iz = 0;
    const bool zero = in_src && (dv == 0.0f);
    if (in_src && !zero) {
      const double d = (double)dv;
      if (!quantize_point<kPow2Side>(__dmul_rn(r0, d), __dmul_rn(r1, d), __dmul_rn(r2, d), half, Vd, side, inv_side, hi,
                                     ix, iy, iz))
        ix = -1;
    }
    const bool any_zero = __syncthreads_or(zero ? 1 : 0) != 0 || (pad > 0 && blockIdx.x == 0 && blockIdx.y == 0);
    if (any_zero && threadIdx.x == 0 && q0_in) {
      const int c = (int)q0;
      if (occ_f32) occ_f32[(((size_t)b * V + c) * V + c) * V] = 1.0f;
      if (occ_bf16) set_occupied(occ_bf16, lay, b, c, c, 0, channel, V);
    }
    if (ix >= 0) {
      if (occ_f32) occ_f32[(((size_t)b * V + ix) * V + iy) * V + iz] = 1.0f;
      if (occ_bf16) set_occupied(occ_bf16, lay, b, ix, iy, iz, channel, V);
    }
  }
}

// ---------------------------------------------------------------------------
// point_cloud_to_voxel_numpy / point_cloud_to_voxel_pytorch over a ragged batch of camera-space clouds: frame b owns
// points [offsets[b], offsets[b+1]).  One grid-stride loop over ALL points of the batch (the host does not know the
// per-frame counts without a synchronisation, and a flat loop keeps every block busy however ragged the batch is); a
// thread finds its frame by a binary search over `offsets` only when its point leaves the frame it was in.
// Scatter: consecutive points of a cloud usually land in the same voxel (neighbouring pixels of a depth map, a wall,
// the thousands of zero-depth points at (0,0,0)), so the lanes of a warp that target the same voxel elect one writer
// (match.any): same-address stores serialise in L2, which is what voxelize_kernel's block vote on the zero-depth voxel
// avoids as well.  Stores of 1.0 by different warps to one voxel are a benign race.
// ---------------------------------------------------------------------------
template <int kPow2Side, typename T>
__global__ void __launch_bounds__(256) voxelize_points_kernel(const T* __restrict__ pts,
                                                             const int64_t* __restrict__ offsets, int batch, int V,
                                                             T half, T Vd, T side, T inv_side, T hi,
                                                             float* __restrict__ occ) {
  const int64_t begin = offsets[0], end = offsets[batch];
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;                 // a multiple of 32: warps stay whole
  const int64_t vol = (int64_t)V * V * V;
  int b = -1;
  int64_t f_lo = 0, f_hi = -1;                                            // [f_lo, f_hi): points of frame b
  for (int64_t base = begin + (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < end; base += stride) {
    const int64_t i = base + lane;
    long long key = -1;
    if (i < end) {
      if (i >= f_hi || i < f_lo) {
        int lo = 0, hi_b = batch;                                          // last b with offsets[b] <= i
        while (hi_b - lo > 1) {
          const int mid = (lo + hi_b) >> 1;
          if (__ldg(offsets + mid) <= i) lo = mid; else hi_b = mid;
        }
        b = lo;
        f_lo = __ldg(offsets + b);
        f_hi = __ldg(offsets + b + 1);
      }
      const T* p = pts + 3 * i;
      int ix, iy, iz;
      if (quantize_point<kPow2Side>(__ldcs(p), __ldcs(p + 1), __ldcs(p + 2), half, Vd, side, inv_side, hi, ix, iy, iz))
        key = (long long)b * vol + ((int64_t)ix * V + iy) * V + iz;
    }
    const unsigned peers = __match_any_sync(0xffffffffu, (unsigned long long)key);
    if (key >= 0 && lane == __ffs(peers) - 1) occ[key] = 1.0f;
  }
}

// ---------------------------------------------------------------------------
// One world-space scan shared by `batch` frames, each with its own camera pose: frame b's cloud is
// c_k = ((A[k,0]*x + A[k,1]*y) + A[k,2]*z) + t[k] for the (3,4) block [A|t] of cam_from_world[b] (NumPy's order for
// `A[k,0]*x + A[k,1]*y + A[k,2]*z + t[k]`, every operation rounded, no FMA), then quantised by quantize_point like
// voxelize_points_kernel.  The transformed clouds are never written: a thread loads a scan point once and evaluates it
// for every frame of its block's frame tile (blockIdx.y), whose poses sit in shared memory.
// kScanFrameTile = 32 frames per tile: the scan is read once per tile, i.e. 24 bytes (fp64) or 12 bytes (fp32) per point
// against 32 transforms and quantisations.  The arithmetic dominates at that ratio (B = 64 on a B200 reads the scan at
// 0.1-0.3 TB/s, DESIGN section 7), so a larger tile would save little traffic while leaving fewer (point block, frame
// tile) pairs to spread a small scan over.
// Scatter: per frame (uniform over the warp), lanes that hit the same voxel elect one writer, as in
// voxelize_points_kernel: a dense scan puts many points into one voxel.
// ---------------------------------------------------------------------------
constexpr int kScanFrameTile = 32;

template <int kPow2Side, typename T>
__global__ void __launch_bounds__(256) voxelize_scan_kernel(const T* __restrict__ pts, int64_t n,
                                                           const T* __restrict__ cam_from_world, int batch, int V,
                                                           T half, T Vd, T side, T inv_side, T hi,
                                                           float* __restrict__ occ) {
  using R = RnOps<T>;
  __shared__ T pose[kScanFrameTile][12];
  const int b0 = blockIdx.y * kScanFrameTile;
  const int nf = min(kScanFrameTile, batch - b0);
  for (int e = threadIdx.x; e < nf * 12; e += blockDim.x) pose[e / 12][e % 12] = cam_from_world[(int64_t)b0 * 12 + e];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;                 // a multiple of 32: warps stay whole
  const int64_t vol = (int64_t)V * V * V;
  for (int64_t base = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < n; base += stride) {
    const int64_t i = base + lane;
    T x = T(0), y = T(0), z = T(0);
    if (i < n) {
      const T* p = pts + 3 * i;
      x = __ldg(p); y = __ldg(p + 1); z = __ldg(p + 2);
    }
    for (int f = 0; f < nf; ++f) {                                         // uniform over the block
      const T* P = pose[f];
      long long key = -1;
      if (i < n) {
        const T c0 = R::add(R::add(R::add(R::mul(P[0], x), R::mul(P[1], y)), R::mul(P[2], z)), P[3]);
        const T c1 = R::add(R::add(R::add(R::mul(P[4], x), R::mul(P[5], y)), R::mul(P[6], z)), P[7]);
        const T c2 = R::add(R::add(R::add(R::mul(P[8], x), R::mul(P[9], y)), R::mul(P[10], z)), P[11]);
        int ix, iy, iz;
        if (quantize_point<kPow2Side>(c0, c1, c2, half, Vd, side, inv_side, hi, ix, iy, iz))
          key = (long long)(b0 + f) * vol + ((int64_t)ix * V + iy) * V + iz;
      }
      const unsigned peers = __match_any_sync(0xffffffffu, (unsigned long long)key);
      if (key >= 0 && lane == __ffs(peers) - 1) occ[key] = 1.0f;
    }
  }
}

// ---------------------------------------------------------------------------
// z-window occupancy plane from a plain f32 occupancy grid (the marching stem's input, include/sceneego_b200.h):
// cell (x,y,z) of plane channel/8 = occ[x][y][z-3 .. z+4] as eight 16-bit values.  voxelize_kernel can scatter into
// that form directly (set_occupied: eight 2-byte stores and their bounds checks per occupied pixel), but the
// voxelisation is bound by instruction issue and the plane then has to be cleared beforehand by the unprojection
// (4.2 MB of its 21 MB per frame).  One store per pixel into a plain grid plus this pass (1 MB read, 4.2 MB written,
// every real cell: no clearing anywhere) is cheaper on both sides.  The grid is SELF-CLEANING: a block reads its rows
// into shared memory, zeroes the entries that were set, and leaves the grid all-zero for the next batch.
// One block = OE_K x `rows` (x,y) rows of one frame, one thread per OE_K voxels.
// ---------------------------------------------------------------------------
constexpr int OE_K = 4;       // row groups per thread: four loads in flight per thread (the pass is latency-, not bandwidth-bound)
__global__ void __launch_bounds__(256) occ_expand_zwin_kernel(float* __restrict__ occ, __nv_bfloat16* __restrict__ vol,
                                                             sceneego_vol_layout_t lay, int plane, int V, int rows) {
  extern __shared__ float s_row[];                       // OE_K x rows x (V + 8): three zeros before, five after each row
  const int z = threadIdx.x, r = threadIdx.y;
  const int b = blockIdx.y;
  const int n_rows = V * V;
  float v[OE_K];
  int row[OE_K];
#pragma unroll
  for (int k = 0; k < OE_K; ++k) {
    row[k] = (blockIdx.x * OE_K + k) * rows + r;         // x * V + y
    v[k] = row[k] < n_rows ? occ[((size_t)b * n_rows + row[k]) * V + z] : 0.f;
  }
#pragma unroll
  for (int k = 0; k < OE_K; ++k) {
    float* srow = s_row + (k * rows + r) * (V + 8);
    srow[z + 3] = v[k];
    if (z < 3) srow[z] = 0.f;
    if (z < 5) srow[V + 3 + z] = 0.f;
    if (v[k] != 0.f) occ[((size_t)b * n_rows + row[k]) * V + z] = 0.f;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < OE_K; ++k) {
    if (row[k] >= n_rows) continue;
    const float* srow = s_row + (k * rows + r) * (V + 8);
    const int x = row[k] / V, y = row[k] - x * V;
    const uint4 cell = make_uint4(act_pack2(srow[z], srow[z + 1]), act_pack2(srow[z + 2], srow[z + 3]),
                                  act_pack2(srow[z + 4], srow[z + 5]), act_pack2(srow[z + 6], srow[z + 7]));
    *reinterpret_cast<uint4*>(vol + ((int64_t)plane * lay.plane_stride + vol_pos(lay, b, x, y, z)) * 8) = cell;
  }
}

// ---------------------------------------------------------------------------
// with_intersection (network/voxel_net_depth.py:257-260): volumes = cat([volumes, volumes * scene, scene]).
// In place on the planar bf16 V2V input: feature planes [0, C/8) -> planes [C/8, 2C/8) multiplied by the
// occupancy value stored in channel 2C (exact: scene is 0 or 1).  One thread = one voxel.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) intersect_kernel(__nv_bfloat16* __restrict__ vol, sceneego_vol_layout_t lay, int c8) {
  const int S = lay.side;
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (n >= S * S * S) return;
  const int z = n % S, y = (n / S) % S, x = n / (S * S);
  const int64_t pos = vol_pos(lay, b, x, y, z);
  const float sc = act_to_float(vol[((int64_t)(2 * c8) * lay.plane_stride + pos) * 8]);
  for (int g = 0; g < c8; ++g) {
    const uint4 in = *reinterpret_cast<const uint4*>(vol + ((int64_t)g * lay.plane_stride + pos) * 8);
    const uint32_t h[4] = {in.x, in.y, in.z, in.w};
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 t = act_unpack2(h[j]);
      o[j] = act_pack2(t.x * sc, t.y * sc);
    }
    *reinterpret_cast<uint4*>(vol + ((int64_t)(c8 + g) * lay.plane_stride + pos) * 8) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// ---------------------------------------------------------------------------
// layout conversions (scene_volumes= input path; tests)
// ---------------------------------------------------------------------------
__global__ void pack_volume_kernel(const float* __restrict__ in, int c, int c_offset, __nv_bfloat16* __restrict__ out,
                                   sceneego_vol_layout_t lay) {
  const int S = lay.s2d ? 2 * lay.side : lay.side;
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (n >= S * S * S) return;
  const int z = n % S, y = (n / S) % S, x = n / (S * S);
  for (int ch = 0; ch < c; ++ch) {
    const int oc = ch + c_offset;
    const __nv_bfloat16 v = act_from_float(in[((size_t)b * c + ch) * S * S * S + n]);
    if (lay.zwin && oc >= 32) {   // z-window occupancy plane: this thread writes its whole cell = occ[x][y][z-3 .. z+4]
      if (oc == 32) {
        __align__(16) __nv_bfloat16 cell[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int zz = z - 3 + e;
          cell[e] = act_from_float((zz >= 0 && zz < S) ? in[((size_t)b * c + ch) * S * S * S + (n - z + zz)] : 0.f);
        }
        *reinterpret_cast<uint4*>(out + ((int64_t)4 * lay.plane_stride + vol_pos(lay, b, x, y, z)) * 8) = *reinterpret_cast<const uint4*>(cell);
      }
      continue;
    }
    if (lay.s2d) {   // stem input: 32 feature channels (4 groups) + the occupancy channel (index 32)
      if (oc < 32) out[vol_cell(lay, b, x, y, z, oc >> 3, 4) * 8 + (oc & 7)] = v;
      else if (oc == 32) out[vol_scene_elem(lay, b, x, y, z, 4)] = v;
    } else {
      out[(vol_cell(lay, b, x, y, z, oc >> 3, 0)) * 8 + (oc & 7)] = v;
    }
  }
}

__global__ void unpack_volume_kernel(const __nv_bfloat16* __restrict__ in, sceneego_vol_layout_t lay, int c,
                                     float* __restrict__ out) {
  const int S = lay.s2d ? 2 * lay.side : lay.side;
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (n >= S * S * S) return;
  const int z = n % S, y = (n / S) % S, x = n / (S * S);
  for (int ch = 0; ch < c; ++ch) {
    int64_t e;
    if (lay.zwin && ch >= 32) e = ((int64_t)4 * lay.plane_stride + vol_pos(lay, b, x, y, z)) * 8 + 3;   // entry 3 = the voxel itself
    else if (lay.s2d) e = ch < 32 ? vol_cell(lay, b, x, y, z, ch >> 3, 4) * 8 + (ch & 7) : vol_scene_elem(lay, b, x, y, z, 4);
    else e = vol_cell(lay, b, x, y, z, ch >> 3, 0) * 8 + (ch & 7);
    out[((size_t)b * c + ch) * S * S * S + n] = act_to_float(in[e]);
  }
}

}  // namespace sceneego

using namespace sceneego;

extern "C" int64_t sceneego_vol_layout_make_s2d(int full_side, int batch, sceneego_vol_layout_t* out) {
  if (full_side <= 0 || (full_side & 1)) return SCENEEGO_E_INVALID;
  const int64_t rc = sceneego_vol_layout_make(full_side / 2, 2, batch, out);
  if (rc > 0) out->s2d = 1;
  return rc;
}

extern "C" int64_t sceneego_vol_layout_make_zwin(int side, int batch, sceneego_vol_layout_t* out) {
  const int64_t rc = sceneego_vol_layout_make(side, 3, batch, out);
  if (rc > 0) out->zwin = 1;
  return rc;
}

extern "C" int64_t sceneego_vol_layout_make(int side, int pad, int batch, sceneego_vol_layout_t* out) {
  if (side <= 0 || pad < 0 || batch <= 0 || !out) return SCENEEGO_E_INVALID;
  sceneego_vol_layout_t L;
  L.s2d = 0; L.zwin = 0;
  L.side = side;
  L.pad = pad;
  L.pitch_y = side + pad;
  L.pitch_x = L.pitch_y * L.pitch_y;
  // guard: largest tap offset of a (2*pad+1)^3 stencil, rounded up to 8 positions (128 B)
  const int g = pad * (L.pitch_x + L.pitch_y + 1);
  L.guard = (g + 7) / 8 * 8;
  L.frame_pitch = ((L.guard + side * L.pitch_x) + 7) / 8 * 8;
  // slack after the last frame: one trailing guard + the widest CTA work item (1024 positions)
  L.plane_stride = (int64_t)batch * L.frame_pitch + L.guard + 1024 + 8;
  *out = L;
  return L.plane_stride;
}

extern "C" int sceneego_ray_table_f64(const sceneego_calib_t* calib, double* d_ray, void* stream) {
  SE_REQUIRE(calib && d_ray, "ray_table: null argument");
  SE_REQUIRE(calib->width > 0 && calib->height > 0, "ray_table: bad image size");
  dim3 grid((calib->width + 255) / 256, calib->height);
  ray_table_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(to_dev(calib), d_ray);
  SE_CUDA_LAUNCH_CHECK("ray_table");
  return SCENEEGO_OK;
}

extern "C" int sceneego_project_voxels_f32(const sceneego_calib_t* calib, int V, float side, int hm_h, int hm_w,
                                           float* d_px, float* d_grid, int32_t* d_status, void* stream) {
  SE_REQUIRE(calib && (d_px || d_grid), "project_voxels: null argument");
  SE_REQUIRE(V >= 2 && V <= 512, "project_voxels: volume_size out of range");
  const float step = (float)((double)side / (V - 1));
  const float lo = (float)(-(double)side / 2);
  const int N = V * V * V;
  project_voxels_kernel<<<(N + 255) / 256, 256, 0, (cudaStream_t)stream>>>(make_w2c(calib), V, lo, step, hm_h, hm_w,
                                                                           d_px, d_grid, d_status);
  SE_CUDA_LAUNCH_CHECK("project_voxels");
  return SCENEEGO_OK;
}

// the CUDA-core form (any cin that is a multiple of 32; csrc/feature_conv.cu holds the entry point and the tensor-core form)
namespace sceneego {
int launch_feature_conv1x1_simt(const float* d_feat, const float* d_weight, const float* d_bias, float* d_out, int batch,
                                int cin, int cout, int h, int w, cudaStream_t st) {
  SE_REQUIRE(cout == FC_CO && cin % FC_KC == 0 && batch > 0, "feature_conv1x1: need cout == 32, cin %% 32 == 0");
  dim3 grid((h * w + FC_PIX - 1) / FC_PIX, batch);
  feature_conv1x1_kernel<<<grid, 256, 0, st>>>(d_feat, d_weight, d_bias, d_out, cin, h * w);
  SE_CUDA_LAUNCH_CHECK("feature_conv1x1");
  return SCENEEGO_OK;
}
}  // namespace sceneego

extern "C" int sceneego_features_upsample_pad_f32(const float* d_in, float* d_out, int batch, int c, int h, int w,
                                                  int up, int pad, void* stream) {
  SE_REQUIRE(d_in && d_out && batch > 0, "features_upsample_pad: null argument");
  SE_REQUIRE((up + 2 * pad) % 4 == 0, "features_upsample_pad: output width must be a multiple of 4");
  SE_REQUIRE((long long)batch * c <= 65535, "features_upsample_pad: batch*c too large for one launch");
  SE_REQUIRE(up % h == 0, "features_upsample_pad: up must be a multiple of h (src = dst * h / up)");
  dim3 grid(h, batch * c);
  upsample_pad_kernel<<<grid, 320, 0, (cudaStream_t)stream>>>(d_in, d_out, c, h, w, up, pad);
  SE_CUDA_LAUNCH_CHECK("features_upsample_pad");
  return SCENEEGO_OK;
}

// d_frame_camera == NULL: one camera (d_grid, or calibs[0] when d_grid is NULL) for the whole batch
static int unproject_impl(const float* d_feat, const float* d_grid, const sceneego_calib_t* calibs, int n_cameras,
                          const int32_t* d_frame_camera, const int32_t* d_frame_order, int batch, int h, int w, int c,
                          int V, float side, int img_h, int img_w, float* d_out_f32, void* d_out_bf16,
                          const sceneego_vol_layout_t* lay, int extra_zero_planes, void* stream) {
  SE_REQUIRE(d_feat && (d_grid || calibs) && (d_out_f32 || d_out_bf16), "unproject: null argument");
  SE_REQUIRE(c == 32, "unproject: 32 feature channels expected (process_features output)");
  SE_REQUIRE(!d_out_bf16 || (lay && (lay->s2d ? 2 * lay->side : lay->side) == V), "unproject: bf16 output needs a matching layout");
  SE_REQUIRE(batch > 0 && batch <= 65535 && img_w >= img_h, "unproject: bad batch / image plane");
  const int N = V * V * V;
  const int fpt = batch >= 32 ? 4 : batch >= 8 ? 2 : 1;       // frames per thread (grid.y stays >= 8 blocks deep)
  dim3 grid((N + 127) / 128, (batch + fpt - 1) / fpt);
  sceneego_vol_layout_t L = lay ? *lay : sceneego_vol_layout_t{};
  const float step = (float)((double)side / (V - 1));
  const float lo = (float)(-(double)side / 2);
  SE_REQUIRE(h > 0 && w > 0 && (long long)img_w * (h > w ? h : w) < (1ll << 31), "unproject: image plane too large");
  auto shift_of = [](int num, int den) {       // log2(num / den) when that ratio is an exact power of two, else -1
    if (den <= 0 || num % den) return -1;
    const int r = num / den;
    for (int k = 0; k < 31; ++k) if ((1 << k) == r) return k;
    return -1;
  };
  const int sh_y = shift_of(img_h, h), sh_x = shift_of(img_h, w), log2v = shift_of(V, 1);
  cudaStream_t st = (cudaStream_t)stream;
  __nv_bfloat16* o16 = (__nv_bfloat16*)d_out_bf16;
  if (d_frame_camera) {
    W2CSet cams{};
    if (!d_grid)
      for (int k = 0; k < n_cameras; ++k) cams.k[k] = make_w2c(calibs + k);
    if (d_grid)
      unproject_cameras_kernel<false><<<grid, 128, 0, st>>>(d_feat, d_grid, cams, d_frame_camera, d_frame_order, h, w, V,
                                                            lo, step, img_h, img_w, d_out_f32, o16, L,
                                                            extra_zero_planes, sh_y, sh_x, log2v, batch, fpt);
    else
      unproject_cameras_kernel<true><<<grid, 128, 0, st>>>(d_feat, nullptr, cams, d_frame_camera, d_frame_order, h, w, V,
                                                           lo, step, img_h, img_w, d_out_f32, o16, L,
                                                           extra_zero_planes, sh_y, sh_x, log2v, batch, fpt);
  } else {
    W2CF32 cam = calibs ? make_w2c(calibs) : W2CF32{};
    if (d_grid)
      unproject_kernel<false><<<grid, 128, 0, st>>>(d_feat, d_grid, cam, h, w, V, lo, step, img_h, img_w, d_out_f32, o16,
                                                    L, extra_zero_planes, sh_y, sh_x, log2v, batch, fpt);
    else
      unproject_kernel<true><<<grid, 128, 0, st>>>(d_feat, nullptr, cam, h, w, V, lo, step, img_h, img_w, d_out_f32, o16,
                                                   L, extra_zero_planes, sh_y, sh_x, log2v, batch, fpt);
  }
  SE_CUDA_LAUNCH_CHECK("unproject");
  return SCENEEGO_OK;
}

extern "C" int sceneego_unproject_f32(const float* d_feat, const float* d_grid, const sceneego_calib_t* calib,
                                      int batch, int h, int w, int c, int V, float side, int img_h, int img_w,
                                      float* d_out_f32, void* d_out_bf16, const sceneego_vol_layout_t* lay,
                                      int extra_zero_planes, void* stream) {
  return unproject_impl(d_feat, d_grid, calib, 1, nullptr, nullptr, batch, h, w, c, V, side, img_h, img_w, d_out_f32,
                        d_out_bf16, lay, extra_zero_planes, stream);
}

extern "C" int sceneego_unproject_cameras_f32(const float* d_feat, const float* d_grids, const sceneego_calib_t* calibs,
                                              int n_cameras, const int32_t* d_frame_camera,
                                              const int32_t* d_frame_order, int batch, int h, int w, int c, int V,
                                              float side, int img_h, int img_w, float* d_out_f32, void* d_out_bf16,
                                              const sceneego_vol_layout_t* lay, int extra_zero_planes, void* stream) {
  SE_REQUIRE(n_cameras >= 1 && n_cameras <= SCENEEGO_MAX_CAMERAS, "unproject_cameras: n_cameras must be in [1, %d]",
             SCENEEGO_MAX_CAMERAS);
  SE_REQUIRE(d_frame_camera, "unproject_cameras: null frame_camera");
  return unproject_impl(d_feat, d_grids, calibs, n_cameras, d_frame_camera, d_frame_order, batch, h, w, c, V, side,
                        img_h, img_w, d_out_f32, d_out_bf16, lay, extra_zero_planes, stream);
}

// d_frame_camera != NULL: d_ray holds one table per camera, frame b uses table d_frame_camera[b]
static int voxelize_impl(const float* d_depth, int batch, int h, int w, int pre_h, int pre_w, float clamp_max,
                         const double* d_ray, int img_h, int img_w, int V, double side, float* d_occ_f32,
                         void* d_occ_bf16, const sceneego_vol_layout_t* lay, int channel, void* stream,
                         bool direct = false, const int32_t* d_frame_camera = nullptr,
                         const int32_t* d_frame_order = nullptr) {
  SE_REQUIRE(d_depth && d_ray && (d_occ_f32 || d_occ_bf16), "voxelize: null argument");
  SE_REQUIRE(batch > 0 && batch <= 65535 && h > 0 && w > 0 && pre_h > 0 && pre_w > 0 && img_w >= img_h, "voxelize: bad shape");
  SE_REQUIRE(!d_occ_bf16 || (lay && (lay->s2d ? 2 * lay->side : lay->side) == V && channel >= 0), "voxelize: bf16 output needs a matching layout");
  SE_REQUIRE(!d_occ_bf16 || !(lay->s2d || lay->zwin) || channel % 8 == 0, "voxelize: s2d / z-window occupancy follows whole channel groups");
  // several frames per block so that a pixel's ray is fetched once for all of them (grid.z <= 65535 either way)
  const int fpb = batch >= 32 ? 8 : batch >= 8 ? 4 : 1;
  const int cols = direct ? img_w : img_h;                            // source columns only
  dim3 grid((cols + 255) / 256, img_h, (batch + fpb - 1) / fpb);
  sceneego_vol_layout_t L = lay ? *lay : sceneego_vol_layout_t{};
  NearestMaps nm;
  // OpenCV: inv_scale = (double)dsize / ssize; ifx = 1. / inv_scale
  nm.ify1 = 1.0 / ((double)img_h / (double)pre_h);
  nm.ifx1 = 1.0 / ((double)cols / (double)pre_w);
  nm.ify0 = (h == pre_h && w == pre_w) ? 1.0 : 1.0 / ((double)pre_h / (double)h);
  nm.ifx0 = (h == pre_h && w == pre_w) ? 1.0 : 1.0 / ((double)pre_w / (double)w);
  nm.pre_h = pre_h; nm.pre_w = pre_w; nm.clamp_max = clamp_max;
  int e2 = 0;
  const bool pow2 = side > 0 && frexp(side, &e2) == 0.5;       // side == 2^(e2-1): divide == exact multiply
  const bool pow2_v = V > 0 && (V & (V - 1)) == 0;
  cudaStream_t st = (cudaStream_t)stream;
  __nv_bfloat16* o16 = (__nv_bfloat16*)d_occ_bf16;
  const int path = pow2 && pow2_v ? 2 : pow2 ? 1 : 0;
  const double inv = pow2 ? 1.0 / side : 0.0;
  if (d_frame_camera) {
    if (path == 2)
      voxelize_cameras_kernel<2><<<grid, 256, 0, st>>>(d_depth, h, w, nm, d_ray, d_frame_camera, d_frame_order, img_h,
                                                       img_w, V, side, inv, d_occ_f32, o16, L, channel, batch, fpb, cols);
    else if (path == 1)
      voxelize_cameras_kernel<1><<<grid, 256, 0, st>>>(d_depth, h, w, nm, d_ray, d_frame_camera, d_frame_order, img_h,
                                                       img_w, V, side, inv, d_occ_f32, o16, L, channel, batch, fpb, cols);
    else
      voxelize_cameras_kernel<0><<<grid, 256, 0, st>>>(d_depth, h, w, nm, d_ray, d_frame_camera, d_frame_order, img_h,
                                                       img_w, V, side, inv, d_occ_f32, o16, L, channel, batch, fpb, cols);
  } else {
    if (path == 2)
      voxelize_kernel<2><<<grid, 256, 0, st>>>(d_depth, h, w, nm, d_ray, img_h, img_w, V, side, inv, d_occ_f32, o16, L,
                                               channel, batch, fpb, cols);
    else if (path == 1)
      voxelize_kernel<1><<<grid, 256, 0, st>>>(d_depth, h, w, nm, d_ray, img_h, img_w, V, side, inv, d_occ_f32, o16, L,
                                               channel, batch, fpb, cols);
    else
      voxelize_kernel<0><<<grid, 256, 0, st>>>(d_depth, h, w, nm, d_ray, img_h, img_w, V, side, inv, d_occ_f32, o16, L,
                                               channel, batch, fpb, cols);
  }
  SE_CUDA_LAUNCH_CHECK("voxelize");
  return SCENEEGO_OK;
}

extern "C" int sceneego_voxelize_depth_f64(const float* d_depth, int batch, int h, int w, const double* d_ray,
                                           int img_h, int img_w, int V, double side, float* d_occ_f32,
                                           void* d_occ_bf16, const sceneego_vol_layout_t* lay, int channel,
                                           void* stream) {
  return voxelize_impl(d_depth, batch, h, w, h, w, INFINITY, d_ray, img_h, img_w, V, side, d_occ_f32, d_occ_bf16, lay,
                       channel, stream);
}

extern "C" int sceneego_voxelize_depth_raw_f64(const float* d_depth_raw, int batch, int h, int w, int pre_h, int pre_w,
                                               float clamp_max, const double* d_ray, int img_h, int img_w, int V,
                                               double side, float* d_occ_f32, void* d_occ_bf16,
                                               const sceneego_vol_layout_t* lay, int channel, void* stream) {
  return voxelize_impl(d_depth_raw, batch, h, w, pre_h, pre_w, clamp_max, d_ray, img_h, img_w, V, side, d_occ_f32,
                       d_occ_bf16, lay, channel, stream);
}

extern "C" int sceneego_voxelize_depth_cameras_f64(const float* d_depth, int batch, int h, int w, int pre_h, int pre_w,
                                                   float clamp_max, const double* d_rays, int n_cameras,
                                                   const int32_t* d_frame_camera, const int32_t* d_frame_order,
                                                   int img_h, int img_w, int V, double side, float* d_occ_f32,
                                                   void* d_occ_bf16, const sceneego_vol_layout_t* lay, int channel,
                                                   void* stream) {
  SE_REQUIRE(n_cameras >= 1 && n_cameras <= SCENEEGO_MAX_CAMERAS, "voxelize_cameras: n_cameras must be in [1, %d]",
             SCENEEGO_MAX_CAMERAS);
  SE_REQUIRE(d_frame_camera, "voxelize_cameras: null frame_camera");
  return voxelize_impl(d_depth, batch, h, w, pre_h, pre_w, clamp_max, d_rays, img_h, img_w, V, side, d_occ_f32,
                       d_occ_bf16, lay, channel, stream, false, d_frame_camera, d_frame_order);
}

extern "C" int sceneego_voxelize_depth_dataset_f64(const float* d_depth_raw, int batch, int h, int w, int pre_h, int pre_w,
                                                   float clamp_max, const double* d_ray, int V, double side,
                                                   float* d_occ_f32, void* stream) {
  // dataset/real_depth_utils.py:29-43: the (pre_h, pre_w) map times the (pre_h, pre_w) ray table, pixel for pixel
  return voxelize_impl(d_depth_raw, batch, h, w, pre_h, pre_w, clamp_max, d_ray, pre_h, pre_w, V, side, d_occ_f32,
                       nullptr, nullptr, 0, stream, true);
}

// quantize_point's operands in the points' precision and which kPow2Side path applies
template <typename T>
struct PointQuant {
  T half, Vd, s, inv, hi;
  int path;
  PointQuant(int V, double side) {
    // fp32 clouds: NumPy / torch turn the Python float s/2 and the ints V, V-1 into float32 operands; s/2 is formed in
    // fp64 first, like the reference's `s / 2`
    half = (T)(side / 2); Vd = (T)V; s = (T)side; hi = (T)(V - 1);
    int e2 = 0;
    const bool pow2 = frexp(side, &e2) == 0.5;                  // side == 2^(e2-1): divide == exact multiply
    const bool pow2_v = (V & (V - 1)) == 0;
    inv = pow2 ? (T)(1.0 / side) : T(0);
    path = pow2 && pow2_v ? 2 : pow2 ? 1 : 0;
  }
};

template <typename T>
static void launch_voxelize_points(const T* d_points, const int64_t* d_offsets, int batch, int V, double side,
                                   float* d_occ, int blocks, cudaStream_t st) {
  const PointQuant<T> q(V, side);
  if (q.path == 2)
    voxelize_points_kernel<2, T><<<blocks, 256, 0, st>>>(d_points, d_offsets, batch, V, q.half, q.Vd, q.s, q.inv, q.hi, d_occ);
  else if (q.path == 1)
    voxelize_points_kernel<1, T><<<blocks, 256, 0, st>>>(d_points, d_offsets, batch, V, q.half, q.Vd, q.s, q.inv, q.hi, d_occ);
  else
    voxelize_points_kernel<0, T><<<blocks, 256, 0, st>>>(d_points, d_offsets, batch, V, q.half, q.Vd, q.s, q.inv, q.hi, d_occ);
}

template <typename T>
static void launch_voxelize_scan(const T* d_points, int64_t n, const T* d_pose, int batch, int V, double side,
                                 float* d_occ, dim3 grid, cudaStream_t st) {
  const PointQuant<T> q(V, side);
  if (q.path == 2)
    voxelize_scan_kernel<2, T><<<grid, 256, 0, st>>>(d_points, n, d_pose, batch, V, q.half, q.Vd, q.s, q.inv, q.hi, d_occ);
  else if (q.path == 1)
    voxelize_scan_kernel<1, T><<<grid, 256, 0, st>>>(d_points, n, d_pose, batch, V, q.half, q.Vd, q.s, q.inv, q.hi, d_occ);
  else
    voxelize_scan_kernel<0, T><<<grid, 256, 0, st>>>(d_points, n, d_pose, batch, V, q.half, q.Vd, q.s, q.inv, q.hi, d_occ);
}

extern "C" int sceneego_voxelize_points(const void* d_points, int points_is_f64, const int64_t* d_offsets, int batch,
                                        int volume_size, double cuboid_side, float* d_occ_f32, void* stream) {
  SE_REQUIRE(volume_size > 0 && cuboid_side > 0 && batch >= 0, "voxelize_points: need volume_size > 0, cuboid_side > 0, batch >= 0");
  SE_REQUIRE(volume_size <= 4096 && (double)batch * volume_size * volume_size * volume_size < 4.0e18,
             "voxelize_points: occupancy grid too large");
  SE_REQUIRE(d_points && d_offsets && d_occ_f32, "voxelize_points: null argument");
  if (batch == 0) return SCENEEGO_OK;
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
    set_error("voxelize_points: %s", cudaGetErrorString(cudaGetLastError()));
    return SCENEEGO_E_CUDA;
  }
  const int blocks = 8 * sms;                                   // 2048 resident threads per SM, one wave
  if (points_is_f64)
    launch_voxelize_points((const double*)d_points, d_offsets, batch, volume_size, cuboid_side, d_occ_f32, blocks,
                           (cudaStream_t)stream);
  else
    launch_voxelize_points((const float*)d_points, d_offsets, batch, volume_size, cuboid_side, d_occ_f32, blocks,
                           (cudaStream_t)stream);
  SE_CUDA_LAUNCH_CHECK("voxelize_points");
  return SCENEEGO_OK;
}

extern "C" int sceneego_voxelize_scan(const void* d_points, int points_is_f64, int64_t n_points,
                                      const void* d_cam_from_world, int batch, int volume_size, double cuboid_side,
                                      float* d_occ_f32, void* stream) {
  SE_REQUIRE(volume_size > 0 && cuboid_side > 0 && batch >= 0 && n_points >= 0,
             "voxelize_scan: need volume_size > 0, cuboid_side > 0, batch >= 0, n_points >= 0");
  SE_REQUIRE(volume_size <= 4096 && (double)batch * volume_size * volume_size * volume_size < 4.0e18,
             "voxelize_scan: occupancy grid too large");
  SE_REQUIRE(n_points <= INT64_MAX / 3 - 256, "voxelize_scan: too many points");
  SE_REQUIRE(batch <= 65535LL * kScanFrameTile, "voxelize_scan: batch too large");
  SE_REQUIRE(d_points && d_cam_from_world && d_occ_f32, "voxelize_scan: null argument");
  if (batch == 0 || n_points == 0) return SCENEEGO_OK;
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
    set_error("voxelize_scan: %s", cudaGetErrorString(cudaGetLastError()));
    return SCENEEGO_E_CUDA;
  }
  // (point blocks, frame tiles): one resident wave of 2048 threads per SM over the point blocks of each tile, fewer
  // when the scan is small; a block strides over the scan
  const int64_t need = (n_points + 255) / 256;
  const dim3 grid((unsigned)(need < 8LL * sms ? need : 8LL * sms), (unsigned)((batch + kScanFrameTile - 1) / kScanFrameTile));
  if (points_is_f64)
    launch_voxelize_scan((const double*)d_points, n_points, (const double*)d_cam_from_world, batch, volume_size,
                         cuboid_side, d_occ_f32, grid, (cudaStream_t)stream);
  else
    launch_voxelize_scan((const float*)d_points, n_points, (const float*)d_cam_from_world, batch, volume_size,
                         cuboid_side, d_occ_f32, grid, (cudaStream_t)stream);
  SE_CUDA_LAUNCH_CHECK("voxelize_scan");
  return SCENEEGO_OK;
}

extern "C" int sceneego_occ_expand_zwin_bf16(float* d_occ_f32, void* d_vol, const sceneego_vol_layout_t* lay, int batch,
                                             int channel, void* stream) {
  SE_REQUIRE(d_occ_f32 && d_vol && lay && batch > 0, "occ_expand_zwin: bad argument");
  SE_REQUIRE(lay->zwin == 1 && channel % 8 == 0, "occ_expand_zwin: needs a z-window layout and a plane-aligned channel");
  const int V = lay->side;
  SE_REQUIRE(V >= 8 && V <= 256, "occ_expand_zwin: side must be in [8, 256]");
  const int rows = 256 / V > 0 ? 256 / V : 1;
  dim3 block((unsigned)V, (unsigned)rows), grid((unsigned)((V * V + rows * OE_K - 1) / (rows * OE_K)), (unsigned)batch);
  occ_expand_zwin_kernel<<<grid, block, (size_t)OE_K * rows * (V + 8) * sizeof(float), (cudaStream_t)stream>>>(
      d_occ_f32, (__nv_bfloat16*)d_vol, *lay, channel / 8, V, rows);
  SE_CUDA_LAUNCH_CHECK("occ_expand_zwin");
  return SCENEEGO_OK;
}

extern "C" int sceneego_intersect_bf16(void* d_vol, const sceneego_vol_layout_t* lay, int batch, int c, void* stream) {
  SE_REQUIRE(d_vol && lay && batch > 0 && batch <= 65535 && c > 0 && c % 8 == 0, "intersect: bad argument");
  SE_REQUIRE(lay->s2d == 0, "intersect: plain planar layout only (the 65-channel stem does not use space-to-depth)");
  const int N = lay->side * lay->side * lay->side;
  intersect_kernel<<<dim3((N + 255) / 256, batch), 256, 0, (cudaStream_t)stream>>>((__nv_bfloat16*)d_vol, *lay, c / 8);
  SE_CUDA_LAUNCH_CHECK("intersect");
  return SCENEEGO_OK;
}

extern "C" int sceneego_pack_volume_bf16(const float* d_in, int batch, int c, int c_offset, void* d_out,
                                         const sceneego_vol_layout_t* lay, void* stream) {
  SE_REQUIRE(d_in && d_out && lay && batch > 0 && batch <= 65535, "pack_volume: bad argument");
  const int S = lay->s2d ? 2 * lay->side : lay->side;
  SE_REQUIRE(!(lay->s2d || lay->zwin) || c + c_offset <= 33, "pack_volume: an s2d / z-window volume holds 32 feature channels + occupancy");
  const int N = S * S * S;
  pack_volume_kernel<<<dim3((N + 255) / 256, batch), 256, 0, (cudaStream_t)stream>>>(d_in, c, c_offset,
                                                                                      (__nv_bfloat16*)d_out, *lay);
  SE_CUDA_LAUNCH_CHECK("pack_volume");
  return SCENEEGO_OK;
}

extern "C" int sceneego_unpack_volume_f32(const void* d_in, const sceneego_vol_layout_t* lay, int batch, int c,
                                          float* d_out, void* stream) {
  SE_REQUIRE(d_in && d_out && lay && batch > 0 && batch <= 65535, "unpack_volume: bad argument");
  const int Sfull = lay->s2d ? 2 * lay->side : lay->side;
  SE_REQUIRE(!(lay->s2d || lay->zwin) || c <= 33, "unpack_volume: an s2d / z-window volume holds 32 feature channels + occupancy");
  const int N = Sfull * Sfull * Sfull;
  unpack_volume_kernel<<<dim3((N + 255) / 256, batch), 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)d_in,
                                                                                        *lay, c, d_out);
  SE_CUDA_LAUNCH_CHECK("unpack_volume");
  return SCENEEGO_OK;
}

extern "C" int sceneego_world2camera_f32(const sceneego_calib_t* calib, const float* d_points, int n_points,
                                         float* d_px, int32_t* d_status, void* stream) {
  SE_REQUIRE(calib && d_points && d_px && n_points > 0, "world2camera: bad argument");
  world2camera_kernel<<<(n_points + 255) / 256, 256, 0, (cudaStream_t)stream>>>(make_w2c(calib), d_points, n_points,
                                                                                d_px, d_status);
  SE_CUDA_LAUNCH_CHECK("world2camera");
  return SCENEEGO_OK;
}

extern "C" int sceneego_grid_sample_f32(const float* d_img, const float* d_grid, int64_t grid_batch_stride, int batch,
                                        int c, int h, int w, int n_points, float* d_out, void* stream) {
  SE_REQUIRE(d_img && d_grid && d_out, "grid_sample: null argument");
  SE_REQUIRE(batch > 0 && batch <= 65535 && c > 0 && h > 1 && w > 1 && n_points > 0, "grid_sample: bad shape");
  grid_sample_kernel<<<dim3((n_points + 255) / 256, batch), 256, 0, (cudaStream_t)stream>>>(
      d_img, d_grid, grid_batch_stride, c, h, w, n_points, d_out);
  SE_CUDA_LAUNCH_CHECK("grid_sample");
  return SCENEEGO_OK;
}
