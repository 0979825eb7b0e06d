/*
 * occdepth_b200 -- C ABI of the B200 (sm_100a) kernels behind the OccDepth forward hot path.
 *
 * The reference (megvii-research/OccDepth) has no FFI: its "operator interface" for this path is the
 * sequence of PyTorch library calls inside occdepth/models/*.py.  Each entry point below names the
 * reference call sequence it replaces (file:line relative to the reference tree).
 *
 * Conventions
 *   - plain pointers + sizes only; all pointers are DEVICE pointers unless stated otherwise
 *   - nothing allocates or synchronises; kernels are enqueued on `stream` (a cudaStream_t cast to void*)
 *   - return 0 on success, an OCCD_ERR_* code otherwise; occd_last_error() returns a static message
 *   - activations are "channels-last": [B][D][H][W][C] with C contiguous (D == 1 for 2-D maps)
 */
#ifndef OCCDEPTH_B200_H
#define OCCDEPTH_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define OCCD_ABI_VERSION 2

/* Activation / GEMM-operand element types.  Every kernel that touches channels-last activations takes one of:    */
/*   OCCD_DTYPE_F32  : fp32 storage holding TF32-representable values (each store rounds to the 10-bit TF32        */
/*                     mantissa, round-to-nearest-away); convolutions run as tcgen05 kind::tf32 with fp32          */
/*                     accumulation -- the reference-precision mode (the reference's fp32 nn.Conv*d under PyTorch's */
/*                     CUDA default, TF32 tensor cores)                                                             */
/*   OCCD_DTYPE_BF16 : bf16 storage, tcgen05 kind::f16 -- the throughput mode                                       */
/* One channel "vector" is 8 consecutive channels (32 / 16 bytes): cstride, coff and C are multiples of 8.         */
#define OCCD_DTYPE_F32 0
#define OCCD_DTYPE_BF16 1

/* -------------------------------------------------------------------------------------------- */
/* library                                                                                      */
int occd_abi_version(void);
const char* occd_last_error(void);

/* -------------------------------------------------------------------------------------------- */
/* Stereo-SFA lift (the memory-bound 2D->3D gather)                                              */
/* replaces SFA.forward (occdepth/models/SFA.py:12-106) x len(project_res) as driven by          */
/* OccDepth._forward_2d_to_3d (occdepth/models/OccDepth.py:262-298) and the FlospDepth product   */
/* x3ds * x3ds_depth * 100 (OccDepth.py:339).                                                    */
#define OCCD_SFA_MAX_SCALES 4
#define OCCD_SFA_OUT_F32_PLANAR 0 /* [C][N]   == reference (C,X,Y,Z) fp32                  */
#define OCCD_SFA_OUT_BF16_CL 1    /* [N][cstride] bf16 channels-last (feeds the 3D net)    */
#define OCCD_SFA_OUT_F32_CL 2     /* [N][cstride] fp32 channels-last                       */
#define OCCD_SFA_OUT_TF32_CL 3    /* [N][cstride] fp32 channels-last, values rounded to TF32 (feeds the 3D net) */

typedef struct {
  const void* feat[OCCD_SFA_MAX_SCALES]; /* per scale: [V][h][w][C] channels-last, feat_dtype      */
  int h[OCCD_SFA_MAX_SCALES];
  int w[OCCD_SFA_MAX_SCALES];
  int div[OCCD_SFA_MAX_SCALES]; /* projected_pix // div (floor), OccDepth.py:286-294               */
  long long vstride[OCCD_SFA_MAX_SCALES]; /* elements between consecutive views; 0 = dense (h*w*C)    */
  int n_scales;                 /* 1..4                                                            */
  int n_views;                  /* V, 1..4                                                         */
  int C;                        /* channels, multiple of 4 (f32) / 8 (bf16), <= 256 (f32) / 512 (bf16) */
  int feat_dtype;               /* OCCD_DTYPE_*                                                    */
  const int64_t* pix;           /* [V][N][P][2] (x,y) int64 -- batch["projected_pix_s"][i]         */
                                /* a point with fov set whose flat index (y//div)*w + (x//div) lies */
                                /* outside [0, h*w) gathers zeros but still counts toward the mean  */
                                /* over the pattern and toward the view mask (the reference leaves  */
                                /* this case undefined: its gather raises or wraps)                 */
  const uint8_t* fov;           /* [V][N][P] bool          -- batch["fov_mask_s"][i]               */
  long long N;                  /* voxels                                                          */
  int P;                        /* pattern points per voxel (1 for pattern_id 0)                   */
  void* out;
  int out_mode;    /* OCCD_SFA_OUT_*                                                               */
  int out_cstride; /* channel stride of channels-last outputs (>= C)                               */
  int perm_nyu;    /* 1: voxel n=(i*S2+k)*S1+j is written at (i*S1+j)*S2+k (SFA.py:90-97)          */
  int S1, S2;
  const float* prior; /* optional [N] per-voxel multiplier (FlospDepth occupancy prior), or NULL   */
  float scale_const;  /* out = out * prior * scale_const when prior != NULL                        */
} occd_sfa_params;

int occd_sfa_lift_fwd(const occd_sfa_params* p, void* stream);

/* layout helpers at the module boundary: NCHW/NCDHW fp32 <-> channels-last (f32 or bf16)          */
/* in: [B][C][S] planar fp32, out: [B][S][cstride] channels-last (pad channels zero-filled), every */
/* value rounded to out_dtype: bf16 round-to-nearest-even, or TF32 for OCCD_DTYPE_F32              */
int occd_planar_to_cl(const float* in, void* out, int out_dtype, long long B, int C, long long S,
                      int cstride, void* stream);
/* in: [B][S][cstride] channels-last, out: [B][C][S] planar fp32                                   */
int occd_cl_to_planar(const void* in, int in_dtype, float* out, long long B, int C, long long S,
                      int cstride, void* stream);


/* -------------------------------------------------------------------------------------------- */
/* Generalised N-d convolution as implicit GEMM on tcgen05 (sm_100a)                              */
/* replaces, with BatchNorm folded into weights/bias and the activation / residual adds fused:    */
/*   nn.Conv3d / nn.Conv2d (+BN +ReLU/LeakyReLU/SiLU)  modules.py:6-48,51-235; DDR.py:51-139;      */
/*     unet2d.py:24-46,65-165; CRP3D.py:22-52; flosp_depth.py:201-257; geffnet 1x1 convs           */
/*   nn.ConvTranspose3d k3 s2 (modules.py:278-296) as 8 sub-pixel phase launches                   */
/*   AvgPool3d + 1x1x1 conv (DDR.py:95-109, modules.py:329-339) as strided multi-tap convs          */
/*   torch.bmm of CRP3D.py:81 (as a 1x1x1 conv whose weights are the mega-context)                 */
/* The GEMM:  M = output positions (tile of 128 = TDxTHxTW box), N = output channels,              */
/*            K = sum over "taps" of the source channels.  A tap = (source tensor, integer offset) */
/* so dilation, padding, multi-branch accumulation (ASPP: three sources, three dilations, one      */
/* accumulator) and concat-free skip connections are all tap lists.                                */
#define OCCD_CONV_MAX_TAPS 81
#define OCCD_CONV_MAX_SRC 3
#define OCCD_CONV_MAX_GROUPS 8
#define OCCD_ACT_NONE 0
#define OCCD_ACT_RELU 1
#define OCCD_ACT_LEAKY 2 /* slope 0.01 */
#define OCCD_ACT_SILU 3
#define OCCD_ACT_SIGMOID 4
#define OCCD_CONV_IMPL_TC 0   /* tcgen05 + TMA implicit GEMM                                       */
#define OCCD_CONV_IMPL_SIMT 1 /* CUDA-core direct convolution (cross-check / odd shapes)           */
#define OCCD_CONV_IMPL_HALO 2 /* tcgen05, halo tile loaded once + row-shifted smem views per tap:    */
                              /* stride-1 {-d,0,d}-tap convs, Cin <= 64, resident weights; returns  */
                              /* OCCD_ERR_UNSUPPORTED from plan_create when the shape does not fit   */
#define OCCD_CONV_IMPL_HALOX 3 /* halo tile for grids whose innermost extent W is 8 / 16 / 32 (one warp row): the   */
                              /* three W taps of each (dz,dy) pair packed into ONE MMA (N = 3*Cout_pad <= 256),  */
                              /* epilogue sums the lane-shifted partials (masked lanes == zero padding); taps in  */
                              /* lexicographic (dz,dy,dx) order, one K chunk, stride 1                           */
#define OCCD_CONV_IMPL_TCX 4  /* per-tap kernel, the three W taps of each (src,dz,dy) group packed into    */
                              /* ONE MMA (N = 3*Cout_pad <= 256): taps ordered as groups of dx = -1,0,+1,   */
                              /* W stride 1, tiles 32 wide (30 outputs), epilogue sums lane-shifted partials */
#define OCCD_OUT1_NONE 0
#define OCCD_OUT1_CL 1         /* pre-activation copy, channels-last in the plan's dtype            */
#define OCCD_OUT1_BF16_CL OCCD_OUT1_CL
#define OCCD_OUT1_F32_PLANAR 2 /* pre-activation copy, fp32 [B][C][positions] (reference layout)   */

typedef struct {
  int src;        /* which source tensor                                                          */
  int dz, dy, dx; /* input coordinate = output coordinate * stride + (dz,dy,dx) (padding folded)  */
} occd_conv_tap;

typedef struct {
  int impl; /* OCCD_CONV_IMPL_*                                                                   */
  int dtype; /* OCCD_DTYPE_*: element type of sources, weights, out0, res1, res2 and a channels-last */
             /* out1.  F32 = TF32 operands (K chunk 32/16/8 channels), BF16 (K chunk 64/32/16)       */
  /* sources: channels-last [B][ID][IH][IW][cstride], channels [coff, coff+C) are read             */
  int n_src;
  const void* src[OCCD_CONV_MAX_SRC];
  int src_C[OCCD_CONV_MAX_SRC];
  int src_cstride[OCCD_CONV_MAX_SRC];
  int src_coff[OCCD_CONV_MAX_SRC];
  int B, ID, IH, IW; /* shared by all sources                                                      */
  int src_d0;        /* plane offset added to every source D coordinate: sources that carry halo   */
                     /* margins ([ID] = slab + 2*margin planes, X-slab multi-GPU partition) are     */
                     /* addressed relative to their interior; 0 for ordinary tensors               */
  int stride[3];     /* (sd, sh, sw)                                                               */
  int n_taps;
  occd_conv_tap taps[OCCD_CONV_MAX_TAPS];
  /* weights: dtype [n_taps][Cout_pad][Kpad], K contiguous, zero padded (F32: pre-rounded to TF32);  */
  /* bias fp32 [Cout_pad]                                                                           */
  const void* weight;
  const float* bias;
  int Cout, Cout_pad, Kpad;
  int weight_per_image; /* 1: weight holds B consecutive [n_taps][Cout_pad][Kpad] sets, image b uses set b   */
                        /* (SE gate folded into the projection weights of each image); TC impl only        */
  /* iteration space of the launch and its mapping to output coordinates: o_full = o*omul + oadd    */
  int OD, OH, OW;
  int omul[3], oadd[3];
  int ODf, OHf, OWf; /* full output grid (== OD,OH,OW unless omul != 1)                            */
  /* out0: channels-last.  v = acc + bias + res1 (+ res2 if !res2_post); out1 = v;                  */
  /*       out0 = act(v) (+ res2 if res2_post)                                                      */
  void* out0;
  int out0_cstride, out0_coff;
  int act;
  int out0_exact;   /* 1: F32 plans store out0 without the TF32 rounding (a tensor that is only ever */
                    /* a residual input, never a GEMM operand); no effect for BF16                   */
  const void* res1; /* channels-last on the full output grid, or NULL                              */
  int res1_cstride, res1_coff;
  const void* res2;
  int res2_cstride, res2_coff;
  int res2_post; /* 1: res2 is added AFTER the activation (modules.py Upsample + skip)            */
  /* out1: optional second output holding the PRE-activation value                                  */
  int out1_mode;
  void* out1;
  int out1_cstride, out1_coff; /* channels-last mode                                               */
  int out1_C;                  /* planar mode: channels of the planar tensor, written at coff+n    */
  /* tap groups (OCCD_CONV_IMPL_TC only; 0 or 1 = off): n_groups convolutions over the same sources, iteration    */
  /* space, weights tensor and bias in ONE launch.  Group g uses taps [group_tap0[g], group_tap0[g+1]) and writes   */
  /* o_full = o*omul + group_oadd[g] (`oadd` is ignored): the 8 sub-pixel phases of ConvTranspose3d(k3, s2, p1,     */
  /* op1) (modules.py:278-296).  Order the groups by descending tap count.  Needs out1_mode == NONE and at most     */
  /* one residual (res1, or res2 with res2_post).                                                                  */
  int n_groups;
  int group_tap0[OCCD_CONV_MAX_GROUPS + 1];
  int group_oadd[OCCD_CONV_MAX_GROUPS][3];
} occd_conv_desc;

typedef struct occd_conv_plan occd_conv_plan;

/* Validates the descriptor, encodes the TMA tensor maps (pointers are baked in: buffers must stay  */
/* allocated and in place) and picks the tiling.  Host call; needs a current CUDA context for TC.   */
int occd_conv_plan_create(const occd_conv_desc* desc, occd_conv_plan** plan);
int occd_conv_plan_destroy(occd_conv_plan* plan);
int occd_conv_run(const occd_conv_plan* plan, void* stream);
/* introspection for tests / profiling: tile box (TD,TH,TW), N tile, K chunk, stages, grid          */
int occd_conv_plan_info(const occd_conv_plan* plan, int* info8);
/* debug: plans created while a device buffer ([64][8] int64) is set stamp per-role clock64 values of CTA 0  */
/* into it (tools/conv_trace.py); NULL switches tracing off                                               */
int occd_conv_debug_trace(long long* device_buf);

/* -------------------------------------------------------------------------------------------- */
/* small channels-last helpers                                                                   */
/* nn.Softmax(dim=1) over C<=32 planar fp32 channels, written as a channels-last channel window   */
/* of element type `dtype` (the torch.cat([x_in, softmax(x_occ)]) of modules.py:168-171)           */
int occd_softmax_planar_to_cl(const float* in, void* out, int dtype, long long B, int C, long long S, int cstride,
                              int coff, void* stream);
/* out[b][c][p] = in[b][p][coff+c]: turns a channels-last activation into a K-major GEMM weight  */
/* (the mega-context operand of torch.bmm, CRP3D.py:62-63,81); out rows have leading dim ldo      */
int occd_cl_transpose(const void* in, void* out, int dtype, int B, int P, int C, int cstride, int coff, int ldo,
                      long long out_bstride, void* stream);
/* class map of the callers' post-processing: uint16 out[b][s] = first index of the largest of the   */
/* C planar fp32 logits in[b][c][s] (np.argmax(softmax(ssc_logit), 1).astype(uint16),               */
/* scripts/generate_output.py:94-97; softmax is monotonic, so it is never evaluated).  lut (HOST      */
/* pointer, C ints, C <= 64) or NULL: out = uint16(lut[class]), the inv_map remap of                  */
/* scripts/generate_kitti_submission.py:79 (data/semantic_kitti/io_data.py:99-113)                    */
int occd_argmax_classes(const float* in, void* out, long long B, int C, long long S, const int* lut, void* stream);
/* copy a channel window (C % 8 == 0) between channels-last buffers (torch.cat of CRP3D.py:90)    */
int occd_copy_channels(const void* in, void* out, int dtype, long long positions, int C, int in_cstride,
                       int in_coff, int out_cstride, int out_coff, void* stream);

/* -------------------------------------------------------------------------------------------- */
/* Data pipeline (SURVEY 8f row 2): voxel-centre -> pixel indices on the device, bit for bit what     */
/* occdepth/data/utils/helpers.py:94-169 `vox2pix` returns (vox2world fusion.py:201-217, rigid_transform */
/* :518-522 in float64 with OpenBLAS' sequential-FMA dot order, cam2allpixs :236-343).                 */
/* HOST pointers: cam_E 4x4 row-major (first 3 rows used), float64 or -- pose_is_f32 != 0 -- float32: */
/* the reference multiplies in the pose's own precision; cam_k 3x3 float32 row-major (the reference's   */
/* intr.astype(float32)), vox_origin 3 float32, pattern P x 2 int (dx, dy).                             */
/* DEVICE pointers: pix int64 [N][P][2] (x, y), fov bool [N][P], pix_z [N] in the pose's precision or   */
/* NULL; N = X*Y*Z voxels in C order.                                                                  */
int occd_vox2pix_fwd(const void* cam_E, int pose_is_f32, const float* cam_k, const float* vox_origin,
                     double voxel_size, int X, int Y, int Z, int img_W, int img_H, const int* pattern, int P,
                     long long* pix, unsigned char* fov, void* pix_z, void* stream);

/* uint8 RGB HWC image [H0][W0][3] (device) -> float32 CHW [3][H][W] of the top-left H x W crop:     */
/* ((u8 / 255) - mean[c]) / std[c] in float32 = np.array(img, float32) / 255.0, crop, ToTensor,        */
/* Normalize of the datasets (data/semantic_kitti/kitti_dataset.py:164-171,376-402); mean/std: HOST    */
int occd_normalize_rgb_u8(const void* in, float* out, int H0, int W0, int H, int W, const float* mean,
                          const float* stdv, void* stream);

/* -------------------------------------------------------------------------------------------- */
/* EfficientNet / decoder bandwidth kernels (channels-last 2-D maps of element type `dtype`)       */
/* depthwise KxK (K = 3|5) conv + folded BN + activation; optionally accumulates the per-channel    */
/* spatial SUM of the output into pool[B][C] (squeeze of geffnet SqueezeExcite) as 64-bit FIXED-    */
/* POINT integers in units of 2^-24 (integer atomics: bit-reproducible); explicit top/left padding  */
/* implements TF "SAME" (bottom/right implied by OH/OW). w: fp32 [K*K][C].                          */
int occd_dwconv2d_fwd(const void* in, const float* w, const float* bias, void* out, long long* pool, int dtype,
                      int B, int H, int W, int OH, int OW, int C, int cs_in, int cs_out, int K, int stride,
                      int pad_top, int pad_left, int act, void* stream);
/* same contract, shared-memory-tiled variant: one zero-filled input halo tile per CTA staged with    */
/* cp.async, FMA loop out of shared memory (results equal up to fp32 summation order)                */
int occd_dwconv2d_tiled_fwd(const void* in, const float* w, const float* bias, void* out, long long* pool, int dtype,
                            int B, int H, int W, int OH, int OW, int C, int cs_in, int cs_out, int K, int stride,
                            int pad_top, int pad_left, int act, void* stream);
/* gate[b][c] = sigmoid(W2 silu(W1 (pool[b] 2^-24 / HW) + b1) + b2); zeroes pool. w1 [R][C],       */
/* w2t [R][C]; `gate` must hold B*C + B*R floats (the hidden layer is staged behind the gates)     */
int occd_se_gate_fwd(long long* pool, float inv_hw, const float* w1, const float* b1, const float* w2t,
                     const float* b2, float* gate, int B, int C, int R, void* stream);
/* fused path: squeeze-excite MLP + gate folded into one projection-weight set per image:          */
/* wout[b][row][k] = wdtype(master[row][k] * gate[b][k]) (bf16 / TF32-rounded fp32 GEMM weights);   */
/* hidden: B*R floats of scratch; zeroes pool                                                       */
int occd_se_gate_fold_fwd(long long* pool, float inv_hw, const float* w1, const float* b1, const float* w2t,
                          const float* b2, float* hidden, const float* master, void* wout, int wdtype, int B, int C,
                          int R, int rows, int Kpad, void* stream);
/* out[row][k] = wdtype(master[row][k] * gate[k]): folds x * gate into the next 1x1 conv's weights */
int occd_scale_weights(const float* master, const float* gate, void* out, int wdtype, int rows, int Kpad, int C,
                       void* stream);
/* F.interpolate(mode="bilinear", align_corners=True) of UpSampleBN.forward (unet2d.py:39-44)      */
int occd_upsample_bilinear_ac(const void* in, void* out, int dtype, int B, int h, int w, int OH, int OW, int C,
                              int cs_in, int in_off, int cs_out, int out_off, void* stream);

/* -------------------------------------------------------------------------------------------- */
/* FlospDepth (the "OAD" depth branch, configs with trans_2d_to_3d: "flosp_depth")                */
/* frustum grid generation fused with the trilinear sampling of the depth distribution and of the */
/* all-ones mask volume + per-camera masked mean: FrustumGridGenerator (f2v/frustum_grid_         */
/* generator.py:70-152), bin_depths LID (f2v/utils/depth_utils.py:24-26), normalize_coords        */
/* (f2v/utils/grid_utils.py:4-19), F.grid_sample (f2v/sampler.py:49-65), flosp_depth.py:563-602.   */
/* depth: [V][Dn][h][w] fp32 probabilities; cams: V x 40 floats {T[12], K[12], ida[16]} where T =  */
/* rows 0..2 of lidar_to_cam @ grid_to_lidar; out: [X*Y*Z] fp32 (perm_xzy: written as [X][Z][Y])  */
int occd_frustum_sample_fwd(const float* depth, const float* cams, int V, int Dn, int h, int w, int X, int Y,
                            int Z, float img_w, float img_h, float dmin, float dmax, int mean_mode, float* out,
                            int perm_xzy, void* stream);
/* the infer_mode / ONNX-export route of the same step (OccDepth.py:310-317, flosp_depth.py:564-565, custom  */
/* GridSample symbolic f2v/sampler.py:9-34): the caller supplies the sampling grids, grids: [V][X*Y*Z][3] fp32 */
/* normalised (x, y, z) coordinates of F.grid_sample(bilinear, zeros, align_corners=False)                    */
int occd_grid_sample_prior_fwd(const float* depth, const float* grids, int V, int Dn, int h, int w, int X, int Y,
                               int Z, int mean_mode, float* out, int perm_xzy, void* stream);
/* softmax over the C planar channels of [B][C][S] fp32 (depth_feature.softmax(1), flosp_depth.py:548) */
int occd_softmax_planar(const float* in, float* out, long long B, int C, long long S, void* stream);
/* out[b] = act(W in[b] + bias): the Linear / 1x1-on-a-vector layers of DepthNet.mlp and SELayer    */
int occd_fc_fwd(const float* in, const float* w, const float* bias, float* out, int B, int n_in, int n_out,
                int act, void* stream);
/* x[b][pos][c] *= gate[b][c] in place (SELayer: x * gate(x_se), flosp_depth.py:195-199)            */
int occd_channel_scale(void* x, const float* gate, int dtype, long long B, long long S, int C, int cstride,
                       void* stream);

/* virtual right view for single-view RGB-D inputs: OccDepth.generate_virtual_img (OccDepth.py:233-260). */
/* in/out: channels-last [B][h][w][cs] of `dtype`; depth: fp32 [dh][dw] of batch item 0; bf_scale = bf / scale_2d */
int occd_virtual_view_fwd(const void* in, void* out, const float* depth, int dtype, int B, int h, int w, int C,
                          int cs_in, int cs_out, int dh, int dw, float bf_scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OCCDEPTH_B200_H */
