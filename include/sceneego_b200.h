/*
 * sceneego_b200 -- C-ABI of the B200-native SceneEgo volumetric lifting stage.
 *
 * The reference (jianwang-mpi/SceneEgo) is pure Python: it has no FFI of its
 * own, its boundary is the nn.Module `VoxelNetwork_depth` and four functions of
 * `utils/op.py`.  Each entry point below replaces the torch / NumPy call site
 * cited next to it; the Python mirror in `sceneego_b200/` binds them with
 * ctypes (see INTEGRATION.md for the stub a reference maintainer would add).
 *
 * Conventions
 *  - every pointer named d_* is a DEVICE pointer; h_* is a HOST pointer;
 *  - no call allocates, frees, synchronises or throws; `stream` is a
 *    cudaStream_t passed as void* (NULL = legacy default stream);
 *  - return value 0 = success, negative = SCENEEGO_E_* below;
 *    `sceneego_last_error()` returns a thread-local message for the last failure;
 *  - volumes are indexed (x, y, z) with flat voxel index x*V*V + y*V + z
 *    (utils/op.py:212, network/voxel_net_depth.py:121-125).
 */
#ifndef SCENEEGO_B200_H
#define SCENEEGO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCENEEGO_ABI_VERSION 5
/* Most cameras one call of sceneego_unproject_cameras_f32 / sceneego_voxelize_depth_cameras_f64 takes. */
#define SCENEEGO_MAX_CAMERAS 16

enum {
  SCENEEGO_OK = 0,
  SCENEEGO_E_INVALID = -1,   /* bad argument (shape, alignment, null pointer)            */
  SCENEEGO_E_CUDA = -2,      /* a CUDA runtime call or kernel launch failed               */
  SCENEEGO_E_DOMAIN = -3,    /* "norm is zero!" -- a voxel centre on the optical axis
                                (utils/fisheye/FishEyeCalibrated.py:177)                  */
  SCENEEGO_E_UNSUPPORTED = -4
};

int sceneego_abi_version(void);
/* Storage type of the V2V activations and packed weights this library was compiled for: 0 = bf16
 * (libsceneego_b200.so, the default), 1 = IEEE fp16 with saturating stores (libsceneego_b200_f16.so, built from the
 * same sources with -DSCENEEGO_ACT_F16).  The "bf16" in entry-point names means "the 16-bit activation type". */
int sceneego_act_dtype(void);
const char* sceneego_last_error(void);

/* Scaramuzza omnidirectional camera (utils/fisheye/FishEyeCalibrated.py:8-16,
 * utils/fisheye/fisheye.calibration_05_08.json). Polynomials in ascending powers. */
typedef struct sceneego_calib {
  double cx, cy;       /* image centre, pixels                                         */
  double c2w[7];       /* polynomialC2W: pixel radius -> z                             */
  double w2c[11];      /* polynomialW2C: elevation angle -> image radius               */
  int32_t width;       /* image plane of the tables, 1280                              */
  int32_t height;      /* 1024                                                         */
} sceneego_calib_t;

/* ---- tables (built once) ------------------------------------------------- */

/* Unit ray per pixel, fp64, replaces calculated_ray_direction_numpy
 * (network/voxel_net_depth.py:147-155) + camera2world_ray
 * (utils/fisheye/FishEyeCalibrated.py:36-51).  Same arithmetic order as NumPy
 * (Horner without FMA, norm = sqrt((x^2+y^2)+z^2)) so the result is bit-identical.
 * Layout written: d_ray[(y*width + x)*3 + c]  (ROW-major, matching a depth map;
 * the reference's table is the same values in x-major order). */
int sceneego_ray_table_f64(const sceneego_calib_t* calib, double* d_ray, void* stream);

/* Voxel-centre projection, fp32, replaces build_coord_volume
 * (network/voxel_net_depth.py:110-134) + world2camera_pytorch
 * (utils/fisheye/FishEyeCalibrated.py:137-174) + get_grid_coord_proj_batch
 * (utils/op.py:177-184).  Writes pixel coords d_px[N*2] and/or the normalised
 * grid d_grid[N*2] (either may be NULL).  *d_status (int32, device, may be NULL)
 * is set to 1 if any voxel has r == 0 (the reference raises). */
int sceneego_project_voxels_f32(const sceneego_calib_t* calib, int volume_size, float cuboid_side,
                                int heatmap_h, int heatmap_w, float* d_px, float* d_grid,
                                int32_t* d_status, void* stream);

/* Arbitrary points: d_points (N,3) f32 -> d_px (N,2) f32; replaces
 * FishEyeCameraCalibrated.world2camera_pytorch (utils/fisheye/FishEyeCalibrated.py:137-187,
 * normalize=False) as reached through utils/multiview.py:128-130 and utils/op.py:98-116. */
int sceneego_world2camera_f32(const sceneego_calib_t* calib, const float* d_points, int n_points,
                              float* d_px, int32_t* d_status, void* stream);

/* ---- a1: process_features (network/voxel_net_depth.py:58-63) -------------- */

/* 1x1 Conv2d + bias.  d_feat (B,Cin,H,W) f32 NCHW -> d_out (B,H,W,Cout) f32 channel-last.
 * Cout must be 32, Cin a multiple of 32. */
int sceneego_feature_conv1x1_f32(const float* d_feat, const float* d_weight, const float* d_bias,
                                 float* d_out, int batch, int cin, int cout, int h, int w, void* stream);

/* Nearest upsample to (up,up) + zero pad `pad` columns left/right, materialising the
 * tensor the reference returns as output #2: d_in (B,h,w,C) channel-last ->
 * d_out (B,C,up,up+2*pad) f32 NCHW. */
int sceneego_features_upsample_pad_f32(const float* d_in, float* d_out, int batch, int c, int h, int w,
                                       int up, int pad, void* stream);

/* ---- a2/a3/a6: fused unprojection ----------------------------------------- */

/* Activation layout consumed by the V2V kernels ("planar padded", see DESIGN.md):
 * bf16, channel groups of 8, per group a linear array of voxel positions with
 * zero guard columns/lines so that a conv tap is a constant position offset. */
typedef struct sceneego_vol_layout {
  int32_t side;          /* S: voxels per axis                                          */
  int32_t pad;           /* zero positions after each z-line and y-lines after each plane */
  int32_t pitch_y;       /* S + pad      positions per z-line                           */
  int32_t pitch_x;       /* pitch_y^2    positions per x-plane                          */
  int32_t guard;         /* zero positions in front of every frame                      */
  int32_t frame_pitch;   /* guard + S*pitch_x                                           */
  int64_t plane_stride;  /* positions per channel-group plane (all frames + slack)      */
  int32_t s2d;           /* 1: space-to-depth storage of a volume of side 2*S (stem input only):
                            voxel (x,y,z), channel c lives in plane ((x&1)*4+(y&1)*2+(z&1))*(C/8)+c/8 at
                            block position (x>>1,y>>1,z>>1); the occupancy channel (the one after the
                            C feature channels) is ONE extra plane whose cell holds the 8 parity
                            values of the 2x2x2 block as its 8 entries                     */
  int32_t zwin;          /* 1: plane 4 (the one after 32 feature channels) is a Z-WINDOW occupancy plane (input of the
                            marching stem, SCENEEGO_OP_STEM7_MARCH): cell (x,y,z) holds occ[x][y][z-3 .. z+4] as its 8
                            entries (zero outside the volume), so one 16-byte cell serves the seven dz taps of a row */
} sceneego_vol_layout_t;

/* Fill a layout for (side, pad, batch); returns plane_stride (positions). */
int64_t sceneego_vol_layout_make(int side, int pad, int batch, sceneego_vol_layout_t* out);
/* Space-to-depth layout of a volume of side `full_side` (even): S = full_side/2, pad = 2, s2d = 1. */
int64_t sceneego_vol_layout_make_s2d(int full_side, int batch, sceneego_vol_layout_t* out);
/* Input layout of the marching stem: plain planar, pad = 3, zwin = 1 (5 planes: 32 features + z-window occupancy). */
int64_t sceneego_vol_layout_make_zwin(int side, int batch, sceneego_vol_layout_t* out);

/* Bilinear gather of the (virtually) x`scale`-upsampled, zero-padded feature map at the
 * projected voxel centres.  Replaces Upsample+ConstantPad2d (voxel_net_depth.py:60-61)
 * and F.grid_sample(bilinear, zeros, align_corners=True) (utils/op.py:209).
 *   d_feat  (B,h,w,C) f32 channel-last, C == 32
 *   d_grid  (N,2) f32 normalised coords in [-1,1] (table mode), or NULL to project the
 *           voxel centres in-kernel through `calib` (fused Scaramuzza mode)
 *   img_h/img_w : virtual image plane (1024 x 1280); scale = img_h / h; pad = (img_w-img_h)/2
 *   d_out_f32   (B,C,V,V,V) f32 NCDHW or NULL
 *   d_out_bf16  planar padded bf16 (layout `lay`), channels [0,C) or NULL
 *   extra_zero_planes: 8-channel planes after the features cleared at every voxel (the scene
 *           channel of the 33-channel V2V input, torch.cat at voxel_net_depth.py:262) */
int sceneego_unproject_f32(const float* d_feat, const float* d_grid, const sceneego_calib_t* calib,
                           int batch, int h, int w, int c, int volume_size, float cuboid_side,
                           int img_h, int img_w, float* d_out_f32, void* d_out_bf16,
                           const sceneego_vol_layout_t* lay, int extra_zero_planes, void* stream);

/* Same gather with a camera per frame, for batches that mix recordings from several fisheye lenses: frame b is
 * sampled exactly as sceneego_unproject_f32 samples it with camera d_frame_camera[b] (bit for bit).
 *   d_grids  (K,N,2) f32 stacked table-mode grids, row k for camera k; or NULL for fused mode, where
 *   calibs   (host array of K) gives camera k's coefficients
 *   n_cameras K in [1, SCENEEGO_MAX_CAMERAS]
 *   d_frame_camera (B) int32, device: camera of frame b; every entry must lie in [0, K) (the call cannot check this:
 *            the ids live on the device)
 *   d_frame_order  (B) int32, device, or NULL = identity: a permutation of [0, B) in which frames are visited; with
 *            frames that share a camera adjacent (a stable sort by camera), a voxel's geometry is computed once per
 *            run of equal cameras instead of once per frame.  Outputs go to frame b's own slot whatever the order.
 * The other arguments are those of sceneego_unproject_f32. */
int sceneego_unproject_cameras_f32(const float* d_feat, const float* d_grids, const sceneego_calib_t* calibs,
                                   int n_cameras, const int32_t* d_frame_camera, const int32_t* d_frame_order,
                                   int batch, int h, int w, int c, int volume_size, float cuboid_side, int img_h,
                                   int img_w, float* d_out_f32, void* d_out_bf16, const sceneego_vol_layout_t* lay,
                                   int extra_zero_planes, void* stream);

/* Generic bilinear gather with the reference op's own signature: replaces
 * F.grid_sample(heatmaps, grid, align_corners=True) at utils/op.py:209 (and :163) on a
 * materialised image.  d_img (B,C,H,W) f32 NCHW; d_grid (N,2) normalised coords, frame b
 * reads d_grid + b*grid_batch_stride floats (0 = one grid shared by the batch);
 * d_out (B,C,N) f32. */
int sceneego_grid_sample_f32(const float* d_img, const float* d_grid, int64_t grid_batch_stride, int batch,
                             int c, int h, int w, int n_points, float* d_out, void* stream);

/* ---- a4/a5: depth map -> occupancy grid ----------------------------------- */

/* Replaces the per-frame host loop depth_map_to_voxel_numpy + point_cloud_to_voxel_numpy
 * (network/voxel_net_depth.py:194-222, :251-257).  fp64 arithmetic without FMA contraction,
 * round-half-even, bit-exact occupancy.
 *   d_depth (B,h,w) f32; nearest-resized to img_h x img_h, padded to img_w
 *   d_ray   (img_h*img_w*3) fp64 row-major from sceneego_ray_table_f64
 *   d_occ_f32  (B,V,V,V) f32 {0,1}  -- must be zeroed by the caller -- or NULL
 *   d_occ_bf16 planar padded bf16 volume (layout `lay`): channel `channel` set to 1.0
 *              -- that channel must be zeroed by the caller -- or NULL */
int sceneego_voxelize_depth_f64(const float* d_depth, int batch, int h, int w, const double* d_ray,
                                int img_h, int img_w, int volume_size, double cuboid_side,
                                float* d_occ_f32, void* d_occ_bf16, const sceneego_vol_layout_t* lay,
                                int channel, void* stream);

/* Same, with the DATASET's preprocessing of the raw depth map fused into the load (SURVEY section 8f row 2):
 * replaces cv2.resize(depth, (pre_w, pre_h), INTER_NEAREST) when the raw map is not pre_h x pre_w, and
 * depth_map[depth_map > clamp_max] = clamp_max (dataset/demo_dataset.py:86-91, dataset/test_dataset.py:138-143),
 * followed by sceneego_voxelize_depth_f64 on the result (the NETWORK's voxelisation: squash to img_h x img_h, pad).
 * Nearest indices are OpenCV's:
 * min(cvFloor(dst * (1. / ((double)n_dst / n_src))), n_src - 1).  clamp_max = +inf disables the clamp.
 *   d_depth_raw (B,h,w) f32 as decoded from the EXR (first channel) */
int sceneego_voxelize_depth_raw_f64(const float* d_depth_raw, int batch, int h, int w, int pre_h, int pre_w,
                                    float clamp_max, const double* d_ray, int img_h, int img_w, int volume_size,
                                    double cuboid_side, float* d_occ_f32, void* d_occ_bf16,
                                    const sceneego_vol_layout_t* lay, int channel, void* stream);

/* sceneego_voxelize_depth_raw_f64 with a camera per frame: frame b back-projects through ray table d_frame_camera[b]
 * and its occupancy equals, bit for bit, that call's with that camera's table.  pre_h == h, pre_w == w and
 * clamp_max = +inf give sceneego_voxelize_depth_f64.
 *   d_rays   (K, img_h, img_w, 3) fp64, K tables from sceneego_ray_table_f64 stacked;  n_cameras K in [1, SCENEEGO_MAX_CAMERAS]
 *   d_frame_camera (B) int32, device, entries in [0, K) (not checked: they live on the device)
 *   d_frame_order  (B) int32, device, or NULL = identity: a permutation of [0, B); a block's frames are taken in this
 *            order and a pixel's ray is reloaded only when the camera changes (pass a stable sort by camera) */
int sceneego_voxelize_depth_cameras_f64(const float* d_depth, int batch, int h, int w, int pre_h, int pre_w,
                                        float clamp_max, const double* d_rays, int n_cameras,
                                        const int32_t* d_frame_camera, const int32_t* d_frame_order, int img_h,
                                        int img_w, int volume_size, double cuboid_side, float* d_occ_f32,
                                        void* d_occ_bf16, const sceneego_vol_layout_t* lay, int channel, void* stream);

/* The DATASET's voxelisation -- replaces depth_map_to_voxel / point_cloud_to_voxel_pytorch
 * (dataset/real_depth_utils.py:29-60), the voxel_output=True path of dataset/demo_dataset.py:93-94 and
 * dataset/test_dataset.py:145-146.  Unlike the network's, the preprocessed (pre_h, pre_w) map is multiplied by the
 * (pre_h, pre_w) ray table pixel for pixel: no squash to H x H, no zero-padded columns.  The dataset's resize of the
 * raw (h,w) map to (pre_h, pre_w) and its clamp are fused into the load as above.
 *   d_ray (pre_h, pre_w, 3) fp64 row-major;  d_occ_f32 (B,V,V,V) f32, zero-initialised by the caller */
int sceneego_voxelize_depth_dataset_f64(const float* d_depth_raw, int batch, int h, int w, int pre_h, int pre_w,
                                        float clamp_max, const double* d_ray, int volume_size, double cuboid_side,
                                        float* d_occ_f32, void* stream);

/* point_cloud_to_voxel_numpy (network/voxel_net_depth.py:207-222) and point_cloud_to_voxel_pytorch
 * (dataset/real_depth_utils.py:45-60) over a ragged batch of camera-space clouds: the entry for scenes that do not come
 * from a depth map (a reconstructed mesh, SLAM, a LiDAR sweep), whose grids reach the network as `scene_volumes=`.
 * q_xy = ((p + s/2) * V) / s, q_z = (p_z * V) / s, round half-to-even, a point is kept iff 0 <= q <= V-1 on all three
 * axes (-0.0 passes; NaN / inf points and overflowing products are dropped).  The precision follows the cloud's dtype,
 * as in NumPy and torch: fp64 for f64 points, fp32 for f32 points; never contracted to FMA.
 *   d_points    (total, 3) row-major, f64 (points_is_f64 = 1) or f32 (0)
 *   d_offsets   (batch + 1) int64, device: frame b owns points [offsets[b], offsets[b+1]); non-decreasing, and
 *               offsets[batch] <= total (the call cannot check this: the offsets live on the device)
 *   d_occ_f32   (batch, V, V, V) f32, zeroed by the caller; occupied voxels set to 1.0
 * batch == 0 launches nothing. */
int sceneego_voxelize_points(const void* d_points, int points_is_f64, const int64_t* d_offsets, int batch,
                             int volume_size, double cuboid_side, float* d_occ_f32, void* stream);

/* The same occupancy for a static world-space scan seen from `batch` camera poses (a room from a mesh, SLAM or a LiDAR
 * sweep, and the head-mounted camera's trajectory), in one launch and without a transformed copy of the scan.  Frame b's
 * cloud is c_k = ((A[k,0]*x + A[k,1]*y) + A[k,2]*z) + t[k] for the (3,4) block [A|t] of its cam_from_world pose, each
 * operation rounded in the points' precision (NumPy's `A[k,0]*x + A[k,1]*y + A[k,2]*z + t[k]`, no FMA); c is then
 * quantised exactly as sceneego_voxelize_points does it.  The camera frame is the one ray x depth produces, in which the
 * cuboid spans x, y in [-s/2, s/2], z in [0, s].  [A|t] is applied as given (no orthonormality check).
 *   d_points          (n_points, 3) row-major world-space scan, f64 (points_is_f64 = 1) or f32 (0), shared by all frames
 *   d_cam_from_world  (batch, 3, 4) row-major, the points' type: the upper rows of each 4x4 pose
 *   d_occ_f32         (batch, V, V, V) f32, zeroed by the caller; occupied voxels set to 1.0
 * batch == 0 or n_points == 0 launches nothing. */
int sceneego_voxelize_scan(const void* d_points, int points_is_f64, int64_t n_points, const void* d_cam_from_world,
                           int batch, int volume_size, double cuboid_side, float* d_occ_f32, void* stream);

/* with_intersection (network/voxel_net_depth.py:257-260): volumes = cat([volumes, volumes * scene, scene]).
 * In place on a plain planar bf16 volume whose channels [0,c) hold the lifted features and channel 2c the
 * occupancy: writes channels [c,2c) = features * occupancy at every voxel. */
int sceneego_intersect_bf16(void* d_vol, const sceneego_vol_layout_t* lay, int batch, int c, void* stream);

/* Same call site (the scene channel of voxel_net_depth.py:251-262) for the marching stem's z-window layout: build the
 * occupancy plane of `channel` from a plain (B,V,V,V) f32 occupancy grid written by sceneego_voxelize_depth*_f64 with
 * d_occ_f32 -- cell (x,y,z) = occ[x][y][z-3..z+4] -- writing EVERY real cell (no clearing needed beforehand) and
 * leaving the grid all-zero again for the next batch (it must be zero before the first voxelisation). */
int sceneego_occ_expand_zwin_bf16(float* d_occ_f32, void* d_vol, const sceneego_vol_layout_t* lay, int batch, int channel,
                                  void* stream);

/* Conversions between (B,C,S,S,S) f32 NCDHW and planar padded bf16 (for the
 * scene_volumes= input path, voxel_net_depth.py:246-249, and for tests). */
int sceneego_pack_volume_bf16(const float* d_in, int batch, int c, int c_offset, void* d_out,
                              const sceneego_vol_layout_t* lay, void* stream);
int sceneego_unpack_volume_f32(const void* d_in, const sceneego_vol_layout_t* lay, int batch, int c,
                               float* d_out, void* stream);

/* ---- a7: V2V encoder-decoder (network/v2v.py) ------------------------------ */

enum { SCENEEGO_OP_CONV = 0, SCENEEGO_OP_MAXPOOL2 = 1, SCENEEGO_OP_DECONV2 = 2,
       SCENEEGO_OP_STEM7_S2D = 3,  /* Conv3d(33,16,k7)+BN+ReLU from an s2d source, network/v2v.py:147 */
       SCENEEGO_OP_TAIL_MLP = 4    /* back_layers[1], back_layers[2] and output_layer (three 1x1 convs,
                                      network/v2v.py:150-161,168-169) in one pass (three chained tcgen05 GEMMs per
                                      128-voxel tile, hidden activations in shared memory); blob segment at w_offset:
                                      [w1 32x32][w2 32x32][w3 32x16] bf16 (pack_conv layout), then
                                      [b1 32][b2 32][b3 16] f32; dst = (B,cout_real,S,S,S) f32 */,
       SCENEEGO_OP_STEM7_MARCH = 6, /* Conv3d(33,16,k7)+BN+ReLU as an x-marching banded GEMM (csrc/stem_march.cu): input plane x
                                      feeds outputs x-3..x+3 in one N = 128 MMA over a ring of 8 tensor-memory slots with
                                      rotated weight rows; source layout zwin = 1; weights from sceneego_v2v_pack_stem_march */
       SCENEEGO_OP_CONV3_MARCH = 5 /* Conv3d k3 + folded BN (+ residual / ReLU / fused projection shortcut) with
                                      3*cout <= 256 as an x-marching banded GEMM (csrc/march.cu): the three dx taps of
                                      an input plane are one N = 3*cout MMA into a ring of tensor-memory slots, the
                                      weights stay resident in shared memory.  Weights from
                                      sceneego_v2v_pack_conv_march; a fused shortcut's follow in the plain ksize-1
                                      sceneego_v2v_pack_conv layout.  xstack / cta_pair are ignored */ };
enum {
  SCENEEGO_F_RELU = 1,         /* ReLU after bias (+ residual)                              */
  SCENEEGO_F_RESIDUAL = 2,     /* add buffer `res` before the ReLU (Res3DBlock, v2v.py:40-43) */
  SCENEEGO_F_ADD_AFTER = 4,    /* add buffer `res` after the ReLU (decoder skip, v2v.py:125-137) */
  SCENEEGO_F_OUT_F32 = 8       /* write (B,cout_real,S,S,S) f32 NCDHW instead of planar bf16 */
};

/* One step of the V2V program.  Buffers are indices into the `buffers` array given
 * to sceneego_v2v_run; each holds a planar padded bf16 volume with layout lay_*. */
typedef struct sceneego_v2v_op {
  int32_t type;        /* SCENEEGO_OP_*                                                    */
  int32_t flags;       /* SCENEEGO_F_*                                                     */
  int32_t ksize;       /* conv: 1, 3 or 7                                                  */
  int32_t cin;         /* padded to a multiple of 16                                       */
  int32_t cout;        /* padded to a multiple of 16                                       */
  int32_t cout_real;   /* channels actually written (15 for the output layer)             */
  int32_t src, dst, res;  /* buffer indices (res = -1 if unused)                           */
  int32_t impl;        /* 0 = tcgen05 kernels, 1 = CUDA-core checker kernel, 2 = (TAIL_MLP only)
                          the register-resident mma.sync variant; other ops treat 2 like 0  */
  int32_t xstack;      /* conv: GEMM rows produce `xstack` consecutive x-planes (N = xstack*cout),
                          weights packed with the same xstack; 0/1 = off                    */
  int32_t cta_pair;    /* conv: 2 = run on CTA pairs (tcgen05 cta_group::2, M = 256); weights packed
                          with n_split = 2; 0/1 = one CTA per tile                          */
  int64_t w_offset;    /* byte offset of the packed bf16 weights in the blob               */
  int64_t b_offset;    /* byte offset of the fp32 bias (cout entries) in the blob          */
  int32_t src2;        /* conv: second source buffer of a fused 1x1 projection shortcut
                          (Res3DBlock.skip_con, network/v2v.py:32-43), -1 = none; its packed weights
                          (pack_conv with ksize 1, the same xstack / n_split) follow the stencil's
                          inside each (half-)blob, and `bias` is the sum of both folded biases      */
  int32_t cin2;        /* channels of src2, padded: must be cin / 2                        */
  sceneego_vol_layout_t lay_src, lay_dst;
} sceneego_v2v_op_t;

/* Host-side fold + repack (replaces nn.BatchNorm3d eval, v2v.py:13,26,29,37,62, at load time).
 *   h_weight: Conv3d (cout,cin,k,k,k) fp32, or ConvTranspose3d (cin,cout,2,2,2) if transposed
 *   bn_*: NULL for no BatchNorm.  Output: bf16 [tap][cin_pad/8][cout_pad][8] and fp32 bias
 *   (transposed: the 8 output parities in groups of npar = min(8, 256/cout_pad) stacked along N,
 *   [group][cin_pad/8][npar*cout_pad][8], one wide GEMM per group).
 *   xstack > 1: Toeplitz-stacked for x-stacking, [(k+xstack-1)*k*k][cin_pad/8][xstack*cout_pad][8]:
 *   column block s of input-plane offset dxp holds W[dx = dxp - s] (zero where out of range).
 *   n_split = 2 (CTA pairs): the N columns are split in two halves, each a complete blob of its own,
 *   [half][tap][cin_pad/8][N/2][8] -- the B operand of tcgen05.mma.cta_group::2 is N-split over the pair. */
int sceneego_v2v_pack_conv(const float* h_weight, const float* h_bias, const float* h_bn_gamma,
                           const float* h_bn_beta, const float* h_bn_mean, const float* h_bn_var,
                           double eps, int cout, int cin, int ksize, int transposed, int cout_pad,
                           int cin_pad, int xstack, int n_split, uint16_t* h_w_out, float* h_b_out);

/* Fold + repack for SCENEEGO_OP_CONV3_MARCH: h_weight (cout,cin,3,3,3) fp32 -> bf16
 *   [tap (dy,dz)][cin_pad/8][3*cout_pad][8], row block j holding W[dx = 2 - j] (the block that feeds output
 *   plane x - 1 + j from input plane x), 27*cin_pad*cout_pad elements, and cout_pad fp32 biases.  The fold is
 *   the one of sceneego_v2v_pack_conv. */
int sceneego_v2v_pack_conv_march(const float* h_weight, const float* h_bias, const float* h_bn_gamma,
                                 const float* h_bn_beta, const float* h_bn_mean, const float* h_bn_var,
                                 double eps, int cout, int cin, int cout_pad, int cin_pad, uint16_t* h_w_out,
                                 float* h_b_out);

/* Same for the 7^3 stem read from a space-to-depth source (SCENEEGO_OP_STEM7_S2D):
 *   h_weight (16,33,7,7,7) fp32.  Output: sceneego_v2v_stem_s2d_weight_bytes() bytes of bf16 in the
 *   kernel's streaming order (2x2x2 output-stacked Toeplitz blocks per input offset, the occupancy
 *   channel packed along K) and 16 fp32 biases.  n_split = 2 packs the 128 stacked columns as two
 *   half-major blobs for CTA pairs (op.cta_pair = 2). */
size_t sceneego_v2v_stem_s2d_weight_bytes(void);
int sceneego_v2v_pack_stem_s2d(const float* h_weight, const float* h_bias, const float* h_bn_gamma,
                               const float* h_bn_beta, const float* h_bn_mean, const float* h_bn_var,
                               double eps, int n_split, uint16_t* h_w_out, float* h_b_out);

/* Same for SCENEEGO_OP_STEM7_MARCH: sceneego_v2v_stem_march_weight_bytes() bytes of bf16,
 *   [rotation r 8][chunk: (k-step, dy) x 14, then occupancy][tap: dz x 7 | dy pair x 4][k-chunk 2][128 rows][8]:
 *   row block s of rotation r holds W[dx = 6 - j], j = (s - r) mod 8 (zeros for j = 7); the occupancy taps multiply
 *   z-window cells (entry e = dz) of two dy rows per MMA: pairs (0,1) (2,3) (4,5) (5,6), the last one's first half zero. */
size_t sceneego_v2v_stem_march_weight_bytes(void);
int sceneego_v2v_pack_stem_march(const float* h_weight, const float* h_bias, const float* h_bn_gamma,
                                 const float* h_bn_beta, const float* h_bn_mean, const float* h_bn_var,
                                 double eps, uint16_t* h_w_out, float* h_b_out);

/* Execute `n_ops` steps on `batch` frames.  d_blob: packed weights + biases. */
int sceneego_v2v_run(const sceneego_v2v_op_t* ops, int n_ops, void* const* d_buffers, const void* d_blob,
                     int batch, void* stream);

/* Measurement variant of sceneego_v2v_run: brackets every op with CUDA events on `stream`,
 * waits for them (the only entry point that synchronises) and returns per-op milliseconds
 * in h_ms[n_ops].  Used by bench.py for the per-kernel roofline. */
int sceneego_v2v_run_profile(const sceneego_v2v_op_t* ops, int n_ops, void* const* d_buffers,
                             const void* d_blob, int batch, void* stream, float* h_ms);

/* Number of kernels the last sceneego_v2v_run on this thread launched. */
int sceneego_v2v_last_launch_count(void);

/* ---- a8: soft-argmax (utils/op.py:83-96) ----------------------------------- */

/* d_logits (B,J,V,V,V) f32; multiplier applied first (voxel_net_depth.py:271).
 * Coordinates: d_axis (3,V) f32 per-axis voxel-centre table (regular grid), or
 * d_coords (N,3) f32 arbitrary (exactly one non-NULL).  softmax=0 -> ReLU, unnormalised.
 *   d_keypoints (B,J,3) f32;  d_volumes_out (B,J,V,V,V) f32 or NULL
 *   d_workspace: at least sceneego_softargmax_workspace_bytes(B,J,V) bytes */
size_t sceneego_softargmax_workspace_bytes(int batch, int joints, int volume_size);
int sceneego_softargmax3d_f32(const float* d_logits, int batch, int joints, int volume_size,
                              float multiplier, int softmax, const float* d_axis, const float* d_coords,
                              float* d_keypoints, float* d_volumes_out, void* d_workspace, void* stream);

/* ---- backbone hand-off (SURVEY section 8f row 1) ------------------------------ */

/* The LAST stage of pose_resnet's deconvolution head -- ConvTranspose2d(256,256,k4,s2,p1,bias=False) + BatchNorm2d + ReLU
 * (network/pose_resnet.py:203-226,238-240: deconv_layers[6..8]) -- fused with process_features[0] = Conv2d(256,32,1)
 * (network/voxel_net_depth.py:58-63) in one tcgen05 kernel (bf16 operands, fp32 accumulation): the reference's
 * (B,256,64,64) f32 `features` map is never written, the stage receives its channel-last input directly.
 *   sceneego_handoff_pack: host-side fold + repack.  h_deconv_w (256,256,4,4) f32 (ConvTranspose2d layout cin,cout,ky,kx),
 *       BatchNorm gamma/beta/mean/var (256), h_conv_w (32,256) f32, h_conv_b (32) or NULL ->
 *       sceneego_handoff_weight_bytes() bytes: [parity 4][tap 4][K-step 16][k-chunk 2][256 rows][8] bf16 (BN scale folded in),
 *       then the 1x1 weights [K-step 16][k-chunk 2][32 rows][8]; h_b_out = 256 BN shifts + 32 conv biases (f32)
 *   sceneego_backbone_handoff_f32: d_x (B,256,h,w) f32 NCHW = the output of deconv_layers[0..5] -> d_out (B,2h,2w,32) f32
 *       channel-last (what sceneego_feature_conv1x1_f32 produces from the 256-channel map); d_workspace of
 *       sceneego_handoff_workspace_bytes(B,h,w) bytes holds the zero-bordered planar bf16 copy of the input */
size_t sceneego_handoff_weight_bytes(void);
size_t sceneego_handoff_workspace_bytes(int batch, int h, int w);
int sceneego_handoff_pack(const float* h_deconv_w, const float* h_bn_gamma, const float* h_bn_beta, const float* h_bn_mean,
                          const float* h_bn_var, double eps, const float* h_conv_w, const float* h_conv_b,
                          uint16_t* h_w_out, float* h_b_out);
int sceneego_backbone_handoff_f32(const float* d_x, int batch, int cin, int h, int w, const void* d_weights,
                                  const float* d_bias, void* d_workspace, float* d_out, void* stream);

/* ---- evaluation (SURVEY section 8f row 3) ------------------------------------ */

/* The metric loop of test.py (dataset/test_dataset.py:102-112) for a batch of poses: replaces calculate_error
 * (utils/calculate_errors.py:22-28), align_skeleton(estimated, gt, None, scale) (:60-91) and umeyama
 * (utils/rigid_transform_with_scale.py:18-43).  fp64 like the reference's NumPy.
 *   d_pred (B,J,3) network output, f32 (pred_is_f64 == 0) or f64 (the reference keeps the caller's dtype: float32
 *           predictions are promoted element by element, float64 ones used as they are);  d_gt (B,J,3) f64
 *   d_mpjpe[B], d_pampjpe[B]: per-frame mean joint distance before / after the per-frame similarity alignment
 *                             (their means over B are the two numbers test.py prints); either may be NULL
 *   d_aligned (B,J,3) f64 aligned poses, d_gt_out (B,J,3) f64 the ground truth align_skeleton returns
 *                             (centred when scale == 0), d_transform (B,13) f64 = c, R row-major, t; any may be NULL
 *   scale: 1 = pose.dot(R) * c + t;  0 = centre both poses first, pose.dot(R) + t */
int sceneego_pose_errors_f64(const void* d_pred, int pred_is_f64, const double* d_gt, int batch, int joints, int scale,
                             double* d_mpjpe, double* d_pampjpe, double* d_aligned, double* d_gt_out,
                             double* d_transform, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SCENEEGO_B200_H */
