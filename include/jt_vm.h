/* jt_vm.h -- C ABI of libjt_vm.so, the B200 (sm_100a) implementation of the
 * TensoRF-VM volume-rendering hot path of Nemo1999/Joint-TensoRF.
 *
 * The reference has no FFI: its operator boundary is the Python class
 * `model.tensorf_repr.BAT_VMSplit` (bateRF.py:7, batBase.py:12, tensorBase.py:374,
 * tensoRF.py:145) selected at model/tensorf.py:375. Each entry point below names
 * the reference method / ATen call sequence it replaces; the Python module
 * `joint_tensorf_b200.B200_VMSplit` binds them with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless its name starts with `h_` (host);
 *  - all tensors are fp32 unless stated; `stream` is the CUDA stream to launch on;
 *  - functions never allocate, never synchronise, never touch another stream;
 *  - sample counts that are only known on the device are passed as `n_dev`
 *    (device int*) together with `n_max` (host upper bound used to size grids);
 *    if `n_dev` is NULL, `n_max` is the count;
 *  - return 0 (JT_OK) or a negative error code, see jt_strerror().
 *
 * Layouts
 *  - VM factors are channel-last: plane i is [H_i][W_i][C_i], line i is [L_i][C_i]
 *    (the physical layout of a torch [1,C,H,W] tensor in channels_last format);
 *    h_factors = {plane0, plane1, plane2, line0, line1, line2};
 *    h_dims    = {H0,H1,H2, W0,W1,W2, L0,L1,L2, C0,C1,C2, elem}; C_i % 4 == 0; elem = 0: the factor pointers
 *    address fp32 elements, 1: bf16 elements (the gather-side copy made by jt_cast_bf16_multi; accepted by
 *    jt_vm_gather_fwd, jt_vm_scatter_rays, jt_app_basis_*_fwd_tc; gradients and arithmetic stay fp32).
 *    Plane i is sampled at (x = u[mat0_i] -> W axis, y = u[mat1_i] -> H axis) with
 *    matMode = [[0,1],[0,2],[1,2]], line i at u[vecMode_i], vecMode = [2,1,0]
 *    (tensorBase.py:405-406).
 *  - h_geom    = {aabb0[3], aabb1[3], invaabbSize[3], stepSize, near, far} (12 floats),
 *    computed with torch exactly as tensorBase.py:477-488 does.
 *  - a compacted sample j carries samp[j] = float4 (u_x, u_y, u_z, t): normalised
 *    coordinates (tensorBase.py:502-503) and its depth along the ray.
 */
#ifndef JT_VM_H_
#define JT_VM_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __CUDA_RUNTIME_H__
typedef struct CUstream_st* cudaStream_t;
#endif

/* ---- library ----------------------------------------------------------- */
const char* jt_strerror(int code);
int jt_version(void);            /* ABI version, bumped on any signature or argument-semantics change
                                  * (3: NULL gradients; 4: jt_head_fwd_tc removed) */
/* number of kernel launches issued through this library since load (for bench.py) */
long long jt_launch_count(void);

/* ---- K1: ray marching -------------------------------------------------- */
/* TensorBase.sample_ray (tensorBase.py:572-612) / sample_ray_ndc (554-571) with the
 * alpha-mask cull of batBase.py:76-82 folded in; dense outputs as the reference
 * returns them: pts [N,S,3], z [N,S], valid [N,S] (uint8).
 * aux: metric rays -> per-ray jitter [N] or NULL (is_train False);
 *      NDC rays    -> depth table [S] (torch.linspace (+jitter)), required.
 * mask_bits: bit-packed AlphaGridMask volume or NULL; h_mask_dims = {W,H,D};
 * h_mask_geom = {mask_aabb0[3], invgridSize[3]} (tensorBase.py:85-86). */
int jt_sample_ray_dense(const float* rays_o, const float* rays_d, const float* aux, int ndc, int n_rays,
                        int n_samples, const float* h_geom, const uint32_t* mask_bits, const int* h_mask_dims,
                        const float* h_mask_geom, float* pts, float* z, uint8_t* valid, cudaStream_t stream);

/* Same sampler, compacted: replaces sample_ray + the boolean-mask indexing
 * xyz_sampled[ray_valid] (batBase.py:104-120). Outputs, ray-major and depth-ordered:
 * ray_off [N+1] (exclusive scan of per-ray valid counts; ray_off[N] = V),
 * sidx [V] = ray*S + k, samp [V] float4, dist [V] = z[k+1]-z[k] (0 for k = S-1,
 * batBase.py:69; x |ray_dir| for NDC rays, batBase.py:63-65). ray_cnt [N] is scratch.
 * Capacity of sidx/samp/dist must be N*S. */
int jt_march_compact(const float* rays_o, const float* rays_d, const float* aux, int ndc, int n_rays,
                     int n_samples, const float* h_geom, const uint32_t* mask_bits, const int* h_mask_dims,
                     const float* h_mask_geom, int* ray_cnt, int* ray_off, int* sidx, float* samp, float* dist,
                     cudaStream_t stream);

int jt_exclusive_scan(const int* cnt, int* off, int n, cudaStream_t stream);

/* ---- K2: VM plane x line interpolation --------------------------------- */
/* app = 0: BAT_VMSplit.compute_densityfeature (bateRF.py:41-94, tensoRF.py:230-251):
 *          out[e] = sum_i sum_c plane_i,c(u) * line_i,c(u)                       out [n]
 * app = 1: gather part of compute_appfeature (bateRF.py:97-128, tensoRF.py:254-268):
 *          out[e][off_i + c] = plane_i,c(u) * line_i,c(u)                        out [n][sum C]
 * Element e reads samp[slot ? slot[e] : e]. */
int jt_vm_gather_fwd(int app, const void* const* h_factors, const int* h_dims, const float* samp,
                     const int* slot, const int* n_dev, int n_max, float* out, cudaStream_t stream);

/* Backward of jt_vm_gather_fwd (replaces grid_sampler_2d_backward x12): scatters
 * into the channel-last gradient buffers h_factor_grads (same order/shape as
 * h_factors, pre-zeroed by the caller) and writes dL/du to dsamp (float4 per sample
 * slot, xyz used; accumulate = 0 store, 1 add). gin: app=0 [n], app=1 [n][sum C]. */
int jt_vm_gather_bwd(int app, const void* const* h_factors, void* const* h_factor_grads, const int* h_dims,
                     const float* samp, const int* slot, const int* n_dev, int n_max, const float* gin,
                     float* dsamp, int accumulate, cudaStream_t stream);

/* Ray-walking form of the backward scatter used by the fused render op (vm_scatter.cu).
 * Same factor-gradient semantics as jt_vm_gather_bwd, but (a) consecutive samples of a ray
 * that fall into the same bilinear cell are merged in registers before one RED per corner
 * (the marcher advances half a voxel per sample: tensorBase.py:483-484), and (b) instead of
 * a per-sample dL/du it ACCUMULATES the pose-path gradients directly:
 *   d_o[r] += sum_j dL/du_j * inv,   d_d[r] += sum_j dL/du_j * inv * t_j     (ray r = sidx/S)
 * i.e. the autograd of rays_pts = o + d*t and normalize_coord (tensorBase.py:502-503,597).
 * The element list must be ray-major (as jt_march_compact / jt_alpha_fwd produce it).
 * d_o / d_d [N][3] must be initialised by the caller (zeros, or jt_ray_init for NDC rays).
 * gin_bf16 = 1 (app only): gin rows are bf16 [n][sum C] as jt_head_bwd_tc writes them.
 * max_ctas = 0: persistent grid (one resident wave), segment length derived in the kernel from the device-side
 * count; > 0: the same with at most max_ctas CTAs; < 0: fixed segments of -max_ctas samples on a non-persistent
 * grid (leaves room for a collective running next to the kernel).
 * max_ctas > 0 caps the (persistent) grid, so that the kernel can share the SMs with another
 * kernel running on a second stream; 0 = fill the machine.
 * plane_mask: bit i = walk plane / line pair i in this launch (7 = all three in one launch). The data-parallel
 * backward launches the appearance planes one by one so that each plane's gradients can be all-reduced while the
 * next plane is still being walked.
 * h_factor_grads = NULL (since version 3): coordinate-only walk for a frozen field -- only d_o / d_d are accumulated,
 * no factor gradient is written; every other argument keeps its meaning. */
int jt_vm_scatter_rays(int app, const void* const* h_factors, void* const* h_factor_grads, const int* h_dims,
                       const float* samp, const int* slot, const int* sidx, const int* n_dev, int n_max,
                       const void* gin, int gin_bf16, int n_samples, const float* h_inv, float* d_o, float* d_d,
                       int max_ctas, int plane_mask, cudaStream_t stream);
/* d_o = 0; d_d = dnorm_r / |d|^2 * d  (NDC rays: dists are scaled by |ray_dir|, batBase.py:63-65;
 * dnorm holds dL/d|d| * |d| from jt_render_bwd) or 0 when dnorm is NULL. */
int jt_ray_init(const float* rays_d, const float* dnorm, int n_rays, float* d_o, float* d_d, cudaStream_t stream);

/* ---- K3: basis_mat + shading head (strict fp32 path) -------------------- */
/* Y[m][0..N) = act(sum_k X[m][k] * W(n,k) + bias[n]) (* (mask[m][n] > 0)); W(n,k) =
 * W[n*ldw+k] (torch Linear weight) or W[k*ldw+n] if w_kn. act: 0 none, 1 relu,
 * 2 sigmoid. Replaces basis_mat (tensoRF.py:156,270) and the Linear layers of
 * MLPRender_Fea / _WeakView (tensorBase.py:109-111,189-191) and their input grads. */
int jt_gemm_nt(const float* X, int ldx, const float* W, int ldw, int w_kn, const float* bias, float* Y, int ldy,
               const float* mask, int ldm, const int* m_dev, int m_max, int N, int K, int act,
               cudaStream_t stream);
/* dW[n][k] += sum_m dY[m][n] X[m][k]; db[n] += sum_m dY[m][n] (weight gradients). */
int jt_gemm_tn(const float* dY, int ldy, const float* X, int ldx, const int* m_dev, int m_max, int N, int K,
               float* dW, int ldw, float* db, cudaStream_t stream);
/* positional_encoding (tensorBase.py:43-55) + the input concatenation of
 * MLPRender_Fea.forward (tensorBase.py:116-122; mode 0) or MLPRender_Fea_WeakView
 * (tensorBase.py:198-206; mode 1, view encoding goes to out2). bwd = 1 maps din
 * (gradient of the encoded row) back to dfeat (written to `out`). View directions
 * are rays_d[sidx[aidx[a]] / n_samples], normalised if normalize_dir (NDC). */
int jt_pe_encode(int bwd, int app_dim, int fea_pe, int view_pe, int mode, float fea_progress,
                 float view_progress, int n_samples, int normalize_dir, const float* feat, int ldf,
                 const int* aidx, const int* sidx, const float* rays_d, const int* n_dev, int n_max, float* out,
                 int ldo, float* out2, int ldo2, const float* din, int ldi, cudaStream_t stream);
/* SHRender (tensorBase.py:68-72) with eval_sh_bases(2, .) (sh.py:88-113). */
int jt_sh_shade(int bwd, const float* feat, int ldf, const int* aidx, const int* sidx, const float* rays_d,
                int n_samples, int normalize_dir, const int* n_dev, int n_max, float* rgb, const float* dout,
                float* dfeat, int ldd, cudaStream_t stream);

/* ---- K3, tensor-core path (tcgen05.mma + TMEM) ---------------------------- */
/* Plumbing self test: mode 0  D[128][N] = A[128][K] * B[N][K]^T (K-major smem operands);
 * mode 1  D[m][n] = sum_s X[s][m] * Y[s][n] with X = A [128][Ma], Y = B [128][N]
 * (MN-major operands, the form the weight-gradient GEMMs use). bf16 products, fp32 sums.
 * mode 2 = mode 0 with both operands stored as fp16. */
int jt_tc_selftest(int mode, const float* A, int lda, const float* B, int ldb, float* D, int K, int N, int Ma,
                   cudaStream_t stream);
/* Staging area of the training forward of the tensor-core head: jt_head_tc_stage_bytes(n_max) bytes, 128-byte
 * aligned, one block per tile of 128 appearance samples. The two forward kernels below write the bf16 operand tiles
 * jt_head_bwd_tc reads (exact relu masks and the operands of the weight-gradient GEMMs): jt_app_basis_fwd_tc the
 * component tile, jt_head_mlp_fwd_tc the encoded-input, relu(h1) and relu(h2) tiles. The backward keeps its own
 * gradient tiles in the rest of each block. The SH pair (jt_app_basis_sh_fwd_tc, jt_sh_bwd_tc) uses the same area. */
long long jt_head_tc_stage_bytes(int n_max);
/* basis_mat (tensoRF.py:270) + positional_encoding (tensorBase.py:43-55) + MLPRender_Fea (tensorBase.py:116-126)
 * for app_dim 27 / hidden 64 / fea_pe = view_pe = 2 as two kernels, the form the fused render op uses.
 * split = 1: bf16 operands; split = 2: every operand as hi+lo bf16 terms, 3 MMAs per product (fp32-class accuracy);
 * split = 3 (jt_head_mlp_fwd_tc only, inference: stage NULL): fp16 operands.
 * jt_app_basis_fwd_tc = appearance gather (bateRF.py:97-128) + basis_mat (tensoRF.py:270) per tile
 * of 128 samples: the plane x line products go straight into the bf16 shared-memory operand tile
 * (never to HBM in fp32), one tcgen05 GEMM projects them; out featdir [A][32] = feat 0..26 | 0 |
 * view dir 28..30 | 0. Needs 3 x 48 appearance components and app_dim 27. `stage` (training)
 * receives the bf16 component tile for the basis_mat weight gradient.
 * jt_head_mlp_fwd_tc = positional_encoding + MLPRender_Fea (tensorBase.py:43-55,116-126) on those
 * rows -> rgb [A][4]; `stage` receives the encoded-input / relu(h1) / relu(h2) tiles. */
int jt_app_basis_fwd_tc(int split, const void* const* h_factors, const int* h_dims, const float* samp,
                        const int* aidx, const int* sidx, const float* rays_d, int n_samples, int normalize_dir,
                        const float* Wb, const int* n_dev, int n_max, float* featdir, void* stage,
                        cudaStream_t stream);
int jt_head_mlp_fwd_tc(int split, const float* featdir, const float* W1, const float* b1, const float* W2,
                       const float* b2, const float* W3, const float* b3, const int* n_dev, int n_max,
                       float fea_progress, float view_progress, float* rgb, void* stage, cudaStream_t stream);
/* Backward of the tensor-core head (bf16 tensor-core GEMMs, fp32 accumulation in TMEM): from dout
 * [A][4] (gradient at the head's pre-activation, from jt_render_bwd), feat [A][ldf] and the
 * tiles the forward left in `stage`, computes dcomps [A][144] (for jt_vm_scatter_rays) and ADDS
 * the weight gradients into gWb [27][144], gW1 [64][150], gb1, gW2 [64][64], gb2, gW3 [3][64],
 * gb3. relu masks are the forward's own; nothing is recomputed.
 * All seven weight-gradient pointers NULL (since version 3; frozen head and basis_mat): dcomps alone, bit-identical
 * to the full call; `stage` is still read (relu masks). A mix of NULL and non-NULL pointers returns JT_ERR_ARG. */
int jt_head_bwd_tc(const float* dout, const float* feat, int ldf, const float* Wb, const float* W1, const float* W2,
                   const float* W3, const int* n_dev, int n_max, float fea_progress, void* dcomps, int dcomps_bf16, void* stage,
                   float* gWb, float* gW1, float* gb1, float* gW2, float* gb2, float* gW3, float* gb3,
                   cudaStream_t stream);
/* SH shading on the tensor-core path (SHRender tensorBase.py:68-72 with eval_sh_bases(2, .)
 * sh.py:88-113; BASELINE config "app_dim 27 SH shading").
 * jt_app_basis_sh_fwd_tc = jt_app_basis_fwd_tc whose epilogue shades the sample straight out of
 * TMEM: rgb [A][4] = relu(sum_k Y_k(dir) feat[c*9+k] + 0.5); the 27 features never reach HBM,
 * featdir [A][32] only receives the view direction (floats 28..30) for the backward.
 * jt_sh_bwd_tc = backward of basis_mat + SHRender: dout [A][4] (gradient at the pre-activation,
 * jt_render_bwd with shade_act 2) -> DF = dout (x) Y (bf16) -> dcomps [A][144] = DF * Wb on
 * tcgen05; ADDS d basis_mat into gWb [27][144] from the component tiles the forward staged.
 * gWb = NULL (since version 3; frozen basis_mat): dcomps alone, bit-identical to the full call, and `stage` may be
 * NULL (a forward that staged nothing). */
int jt_app_basis_sh_fwd_tc(int split, const void* const* h_factors, const int* h_dims, const float* samp,
                           const int* aidx, const int* sidx, const float* rays_d, int n_samples, int normalize_dir,
                           const float* Wb, const int* n_dev, int n_max, float* featdir, float* rgb, void* stage,
                           cudaStream_t stream);
int jt_sh_bwd_tc(const float* dout, const float* featdir, int ldf, const float* Wb, const int* n_dev, int n_max,
                 void* dcomps, int dcomps_bf16, void* stage, float* gWb, cudaStream_t stream);

/* ---- K4: alpha compositing --------------------------------------------- */
/* feature2density (tensorBase.py:696-700; act 0 softplus, 1 relu) + raw2alpha
 * (tensorBase.py:57-65) over the compacted samples of each ray, then the app_mask
 * selection weight > thres (batBase.py:127) compacted: app_off [N+1], aidx [A] ->
 * sample slot, app_of [V] -> appearance slot or -1. Also per ray acc = sum w and
 * wz = sum w*t.
 * app_cap bounds the appearance list (capacity of the caller's appearance-stage buffers; N*S = unbounded):
 * entries past it are dropped (app_of = -1), and app_used (device int[2], may be NULL) receives
 * {min(A, app_cap), A > app_cap}; app_off[N] keeps the true A. The appearance-stage kernels take app_used as
 * their device-side count, so an under-estimated capacity degrades that call (flagged) instead of overrunning. */
int jt_alpha_fwd(const int* ray_off, int n_rays, const float* sigfeat, const float* dist, const float* samp,
                 float density_shift, int act, float distance_scale, float thres, float* weight, float* trans,
                 float* acc, float* wz, int* app_cnt, int* app_off, int* aidx, int* app_of, int app_cap,
                 int* app_used, cudaStream_t stream);
/* batBase.py:142-165: rgb_map = clamp(sum w*rgb (+ 1-acc if white_bg), 0, 1);
 * depth = sum w*t + (1-acc)*ray_dir_z + depth_bias (depth_bias = -near + 0.05);
 * opacity = acc. rgb_pre keeps the un-clamped colour for the backward pass.
 * Per-sample colours `rgb` and their gradients `dout` are [A][4] (xyz used). */
int jt_composite_fwd(const int* app_off, int n_rays, const int* aidx, const float* weight, const float* rgb,
                     const float* acc, const float* wz, const float* rays_d, int white_bg, float depth_bias,
                     float* rgb_pre, float* rgb_map, float* depth, float* opacity, int app_cap, cudaStream_t stream);
/* autograd of composite + raw2alpha + feature2density as one reverse scan per ray:
 * (g_rgb [N,3], g_acc [N] or NULL) -> dout [A,3] (gradient at the shading head's
 * pre-activation; shade_act 0 none, 1 sigmoid, 2 relu), dsig [V] (gradient of the
 * density feature), dnorm [N] or NULL (NDC: dL/d|ray_dir| * |ray_dir|). */
int jt_render_bwd(const int* ray_off, int n_rays, const float* sigfeat, const float* dist, const float* weight,
                  const float* trans, const int* app_of, const float* rgb, const float* rgb_pre,
                  const float* g_rgb, const float* g_acc, float density_shift, int act, float distance_scale,
                  int white_bg, int shade_act, float* dout, float* dsig, float* dnorm, cudaStream_t stream);
/* Normal map of the rays jt_alpha_fwd composited: normal_map [N][3] = sum_j weight_j * normals_j over every valid
 * sample j of ray r (ray_off as jt_march_compact writes it; the weights whose sum is the opacity), normals [V][3] the
 * per-sample unit normals of jt_field_density_grad (normals = 1); not renormalised, so |normal_map[r]| <= acc[r].
 * depth and opacity are written exactly as jt_composite_fwd writes them. One warp per ray in a fixed order: a ray's
 * result does not depend on the other rays of the call. */
int jt_normal_composite(const int* ray_off, int n_rays, const float* weight, const float* normals, const float* acc,
                        const float* wz, const float* rays_d, float depth_bias, float* normal_map, float* depth,
                        float* opacity, cudaStream_t stream);
/* ---- K5: separable blur ------------------------------------------------ */
/* BAT_VMSplit.convolute_plane / convolute_line (bateRF.py:8-39) on a channel-last
 * [H][W][C] array: replicate-padded cross-correlation with `h_taps` [ntaps] (HOST
 * array, odd count <= 257; the taps travel in the kernel parameters) along W (axes bit 0)
 * and/or H (bit 1); adjoint = 1 applies the transposed operator (backward pass).
 * tmp [H][W][C] is needed when axes == 3. in / out / tmp 16-byte aligned. */
int jt_blur_cl(const float* in, float* out, float* tmp, int H, int W, int C, const float* h_taps, int ntaps,
               int axes, int adjoint, cudaStream_t stream);
/* The same for up to 12 arrays (all VM factors of a step) in two launches, one per pass: h_in / h_out / h_tmp
 * are HOST arrays of device pointers, h_dims = {H, W, C, axes} per array, array i uses tap set h_tapset[i]
 * (0 .. nsets-1, nsets <= 2: density taps and colour taps, batBase.py:92-101) of h_taps [nsets][ntaps] (host). */
int jt_blur_multi(int n_arrays, const void* const* h_in, void* const* h_out, void* const* h_tmp, const int* h_dims,
                  const int* h_tapset, const float* h_taps, int nsets, int ntaps, int adjoint, cudaStream_t stream);

/* ---- pose -> rays (next row, SURVEY.md section 8f-1) --------------------- */
/* One step's ray set for the sampled pixels only, replacing
 *   model/bat.py:350-353      pose = compose([lie.se3_to_SE3(se3_refine[idx]), pose])   (camera.py:81-99, 43-58)
 *   model/tensorf.py:144-166  camera.get_center_and_ray (camera.py:231-261) for ALL H*W pixels, then [:, ray_idx],
 *                             then camera.convert_NDC (camera.py:303-340) when ndc.
 * se3 [n_rows][6] (w, u) or NULL (no refinement); view b uses row view_idx[b] (or b when view_idx is NULL).
 * base [B][3][4] world-to-camera poses (one shared pose when base_per_view = 0); intr_inv / intr [B][3][3]
 * (shared when *_per_view = 0; intr only read when ndc). Pixel of ray r of view b: pix[r] (pix_per_view = 0),
 * pix[b*R + r] (pix_per_view = 1) or pix_base + r when pix is NULL (a contiguous render slice);
 * pixel p -> (x, y) = (p % width + 0.5, p / width + 0.5). Outputs center, ray [B][R][3] and (optional) the
 * composed poses pose_out [B][3][4]. */
int jt_pose_rays_fwd(const float* se3, const int* view_idx, const float* base, int base_per_view,
                     const float* intr_inv, int kinv_per_view, const float* intr, int k_per_view, const int* pix,
                     int pix_per_view, int pix_base, int n_views, int n_rays_per_view, int width, int ndc,
                     int center_shift, int detach_shift, float near_plane, float* center, float* ray,
                     float* pose_out, cudaStream_t stream);
/* Autograd of the above: (d_center, d_ray [B][R][3]) -> d_se3 [n_rows][6] (ADDED into; may be NULL) and/or
 * d_pose [B][3][4] (gradient w.r.t. the composed pose, stored; may be NULL). scratch12: [B][12] floats. */
int jt_pose_rays_bwd(const float* se3, const int* view_idx, const float* base, int base_per_view,
                     const float* intr_inv, int kinv_per_view, const float* intr, int k_per_view, const int* pix,
                     int pix_per_view, int pix_base, int n_views, int n_rays_per_view, int width, int ndc,
                     int center_shift, int detach_shift, float near_plane, const float* d_center, const float* d_ray,
                     float* scratch12, float* d_se3, float* d_pose, cudaStream_t stream);

/* ---- per-step full-factor sweeps (next row, SURVEY.md section 8f-2) ------ */
/* The regularisers model/tensorf.py:126-130 evaluates every training step:
 *   density_L1 (tensoRF.py:212-216), TV_loss_density / TV_loss_app (tensoRF.py:218-228) with
 *   TVLoss (tensorBase.py:16-41; weight 1, batch 1, the 1e-2 factor of TV_loss_* included).
 * Arrays are channel-last [H][W][C] fp32 buffers (h_x: HOST array of n_arrays <= 12 device pointers,
 * h_dims = {H, W, C} per array; a line factor is H = L, W = 1). h_term[i]: 0 = no TV, 1 = TV summed into
 * TV_density, 2 = into TV_app; h_l1[i] != 0: mean|x| summed into L1.
 * sums_ws: 36 doubles of scratch; out3 = {L1, TV_density, TV_app}. One sweep: every element read once. */
int jt_reg_values(int n_arrays, const void* const* h_x, const int* h_dims, const int* h_term, const int* h_l1,
                  double* sums_ws, float* out3, cudaStream_t stream);
/* Their autograd in one sweep: h_g[i] += d/dx ( c0*L1 + c1*TV_density + c2*TV_app ), c_k = h_coef3[k]
 * (host weights, e.g. opt.loss_weight.*) times up3[k] (optional DEVICE upstream gradients, NULL = 1).
 * Arrays whose host weight is zero are skipped. sign(0) = 0 as in ATen's abs backward. */
int jt_reg_grads(int n_arrays, const void* const* h_x, void* const* h_g, const int* h_dims, const int* h_term,
                 const int* h_l1, const float* h_coef3, const float* up3, cudaStream_t stream);
/* torch.optim.Adam (model/tensorf.py:474-475: betas (0.9, 0.99), eps 1e-8, no weight decay / amsgrad) for all
 * parameter tensors of a step in ONE launch per 32 tensors (the reference's foreach path makes ~6 passes over
 * every tensor). Tensor i: p, g, exp_avg m, exp_avg_sq v (dense fp32 buffers of h_numel[i] elements sharing one
 * physical layout), learning rate h_lr[i] (already decayed by the host, tensorf.py:431-436) and step count
 * h_step[i] >= 1 (the value AFTER this step's increment). g is multiplied by grad_scale first (1/world_size
 * after a summing all-reduce) and is zeroed in the same pass when zero_grad != 0. */
int jt_adam_multi(int n_tensors, void* const* h_p, void* const* h_g, void* const* h_m, void* const* h_v,
                  const long long* h_numel, const double* h_lr, const int* h_step, double beta1, double beta2,
                  double eps, double grad_scale, int zero_grad, cudaStream_t stream);

/* ---- field maintenance between steps (next row, SURVEY.md section 8f-3) -- */
/* BatBase.compute_alpha (batBase.py:27-42) and TensorBase.getDenseAlpha (tensorBase.py:618-633):
 * alpha = 1 - exp(-feature2density(sigma_feature(p)) * length), 0 where the occupancy mask rejects p.
 * xyz != NULL: n_points explicit world-space points [n][3] -> alpha [n].
 * xyz == NULL: the dense grid p = aabb0*(1-s) + aabb1*s with s from the device tables lin_x/y/z
 *   (torch.linspace(0, 1, g), h_grid3 = {gx, gy, gz}); alpha is written in [gz][gy][gx] order (the layout
 *   updateAlphaMask pools, tensorBase.py:639-640). Factors: the (blurred, if a blur is cached) density factors. */
int jt_field_alpha(const void* const* h_factors, const int* h_dims, const float* h_geom, const float* xyz,
                   long long n_points, const float* lin_x, const float* lin_y, const float* lin_z, const int* h_grid3,
                   const uint32_t* mask_bits, const int* h_mask_dims, const float* h_mask_geom, float density_shift,
                   int act, float length, float* alpha, cudaStream_t stream);
/* Density and its spatial gradient at points, forward mode (no atomics, no gradient buffers; deterministic, and each
 * point's result is independent of the others): sigma = feature2density(sigma_feature(p)) with jt_field_alpha's taps
 * and summation order (so 1 - exp(-sigma * length) equals its alpha), and grad = d sigma / d p, the analytic derivative
 * of the piecewise-multilinear field that grid_sample(bilinear, align_corners=True, zeros) evaluates (out-of-range
 * taps count as 0; one-sided at cell boundaries as the tap rounding falls), times feature2density' and the per-axis
 * invaabbSize of normalize_coord: the gradient is in the field's input coordinates (world, or NDC for an NDC field).
 * Points: xyz != NULL: n_max explicit points [n][3] (slot and n_dev NULL), tested against the optional occupancy
 * mask (rejected points give sigma 0, grad 0); samp != NULL: compacted float4 records (normalised coordinates, as
 * jt_march_compact writes them), element e reads samp[slot ? slot[e] : e], count n_dev (device) or n_max; no mask.
 * Exactly one of xyz / samp. normals = 1: grad receives the unit outward normal -grad / |grad| instead ((0,0,0) where
 * grad is zero or not finite). sigma [n] may be NULL; grad [n][3]. Factors: fp32 (elem 0). */
int jt_field_density_grad(const void* const* h_factors, const int* h_dims, const float* h_geom, const float* xyz,
                          const float* samp, const int* slot, const int* n_dev, long long n_max,
                          const uint32_t* mask_bits, const int* h_mask_dims, const float* h_mask_geom,
                          float density_shift, int act, int normals, float* sigma, float* grad, cudaStream_t stream);
/* First hit of each ray on the level set extract_mesh contours. A point p is inside iff point_in_box (the marcher's
 * aabb test) passes and jt_field_alpha's alpha at p, with `length`, the occupancy mask and the same taps, summation
 * order and exp, is >= level (fp32). Candidates are the sample depths t_k of the no-grad forward for the same rays
 * and n_samples: t_min + stepSize * k for metric rays (ztab NULL), ztab[k] for NDC rays; the points are the marcher's
 * separately rounded o + d t. The hit sample k is the first inside one in ray order. For k > 0 the crossing is
 * refined in [t_{k-1}, t_k]: each round evaluates the predicate at P equally spaced interior points lo + w j
 * (w = (hi - lo) / (P + 1), j = 1..P, fp32; P = 15 with 16 channels on every plane, else 7) and keeps the first
 * inside point as hi and the point before it as lo, until hi - lo <= 2^-20 (t_k - t_{k-1}) or no fp32 value lies
 * strictly between them. k == 0 (the ray starts inside): no refinement.
 * Outputs per ray [n_rays]: t = hi (inside; the ray parameter of xyz = o + t d, not the forward's depth_map), +inf on
 * a miss; xyz [n][3] = the fp32 point whose predicate was evaluated at t, 0 on a miss; k = the hit sample, -1 on a
 * miss; rounds (may be NULL) = refinement rounds. Each ray's result depends on nothing but the ray. work: one zeroed
 * device int (rays are handed to warps through it), or NULL (static grid stride; the same results). Factors: fp32
 * only (JT_ERR_UNSUPPORTED for bf16). 0 < level < 1 and n_samples > 0 are checked. */
int jt_raycast(const void* const* h_factors, const int* h_dims, const float* h_geom, const uint32_t* mask_bits,
               const int* h_mask_dims, const float* h_mask_geom, float density_shift, int act, float length,
               float level, const float* rays_o, const float* rays_d, int n_rays, const float* ztab, int n_samples,
               int* work, float* t, float* xyz, int* k, int* rounds, cudaStream_t stream);
/* The rest of updateAlphaMask (tensorBase.py:639-657): clamp(alpha, 0, 1) -> max_pool3d(kernel 5, pad 2, stride 1)
 * -> >= thres, on alpha [D][H][W]. Outputs: vol [D][H][W] floats {0,1} (AlphaGridMask.alpha_volume), bits = the same
 * bit-packed ((W*H*D+31)/32 words, layout of MaskGeom), stats7 = {min_x, max_x, min_y, max_y, min_z, max_z, count}
 * of the kept voxels (the new aabb is the grid position of those indices). tmp: W*H*D floats. */
int jt_alpha_mask_build(const float* alpha, int W, int H, int D, float thres, float* tmp, float* vol, uint32_t* bits,
                        int* stats7, cudaStream_t stream);
/* F.interpolate(mode="bilinear", align_corners=True) of one factor (up_sampling_VM, tensoRF.py:274-287) on the
 * channel-last layout: in [H][W][C] -> out [H2][W2][C]; a line factor is W = W2 = 1. */
int jt_resize_bilinear_cl(const float* in, int H, int W, int C, float* out, int H2, int W2, cudaStream_t stream);

/* ---- mesh export: marching cubes over the dense alpha grid ----------------- */
/* The step TensoRF-family exporters take after getDenseAlpha (tensorBase.py:618-633): marching cubes on a dense fp32
 * volume vol [gz][gy][gx] (jt_field_alpha's dense layout) at `level`; a lattice point is inside when value > level.
 * gx, gy, gz >= 2 and gx*gy*gz < 2^31. Two calls, with one host read of the totals in between to size the outputs:
 *   jt_mc_count  classifies every cell and writes totals[2] (device long long) = {V, F};
 *   jt_mc_emit   writes verts [V][3] fp32 and faces [F][3] int32 from the scratch jt_mc_count left for the same vol,
 *                grid and level; it writes nothing when V or F exceeds INT32_MAX.
 * Vertices: one per lattice edge whose ends straddle the level, ordered by the linear index (z*gy + y)*gx + x of the
 * edge's lower end, then by axis x < y < z; position p_a + t (p_b - p_a), t = (level - a)/(b - a), in fp32, where
 * lattice point (i, j, k) is aabb0*(1-s) + aabb1*s with s from lin_x[i], lin_y[j], lin_z[k] (torch.linspace(0, 1, g),
 * as jt_field_alpha), h_aabb = {aabb0[3], aabb1[3]} (host). Faces: ordered by the linear index of the cell's corner 0,
 * then by the case table (csrc/mc_tables.cuh); normals point toward decreasing value.
 * scratch: jt_mc_scratch_bytes(gx, gy, gz) = ceil(gx*gy*gz / 2048) * 1304 bytes (0.64 bytes per lattice point),
 * 16-byte aligned; returns -1 for a grid outside the limits above. */
long long jt_mc_scratch_bytes(int gx, int gy, int gz);
int jt_mc_count(const float* vol, int gx, int gy, int gz, float level, void* scratch, long long* totals,
                cudaStream_t stream);
int jt_mc_emit(const float* vol, int gx, int gy, int gz, float level, const float* lin_x, const float* lin_y,
               const float* lin_z, const float* h_aabb, const void* scratch, const long long* totals, float* verts,
               int* faces, cudaStream_t stream);
/* Vertex normals of that mesh: normals [V][3] fp32 in jt_mc_emit's vertex order, from the scratch jt_mc_count left
 * for the same vol, grid and level (arguments as jt_mc_emit; it writes nothing when V or F exceeds INT32_MAX).
 * With c_a(i) the lattice coordinate above, the gradient at lattice point i along axis a is
 * (v[i+1] - v[i-1]) / (c_a(i+1) - c_a(i-1)), one-sided at the border ((v[1] - v[0]) / (c(1) - c(0)) and the same at
 * the top end). The normal of the vertex on edge p0 -> p1 is -normalize((1-t) g(p0) + t g(p1)) with jt_mc_emit's
 * fp32 t, (0,0,0) when that vector is zero: it points toward decreasing value, as the face winding does. One warp
 * per 32-point chunk with crossings, no atomics: the output is deterministic. */
int jt_mc_normals(const float* vol, int gx, int gy, int gz, float level, const float* lin_x, const float* lin_y,
                  const float* lin_z, const float* h_aabb, const void* scratch, const long long* totals,
                  float* normals, cudaStream_t stream);

/* ---- 2-D supervision pre-processing and the render loss (next row, SURVEY.md section 8f-4) -- */
/* Model.process_GT_images (model/nerf.py:57-113): separable blur of n_img single-channel images [n_img][H][W]
 * (the reference reshapes [B,3,H,W] to [B*3,H,W]): replicate pad + cross-correlation with h_taps (HOST, ntaps odd,
 * <= 257; 201 in the shipped YAMLs) along W (nerf.py:102-103), then the same along H (105-106). tmp: n_img*H*W floats.
 * `in` may not alias `out` or `tmp`. Taps come from kernels.get_gaussian_kernel / get_average_kernel (kernels.py:16-41). */
int jt_image_blur(const float* in, float* out, float* tmp, int n_img, int H, int W, const float* h_taps, int ntaps,
                  cudaStream_t stream);
/* Model.get_edge_mask (model/nerf.py:116-149) on images [n_img][3][H][W]: replicate pad, the two 3x3 Sobel
 * correlations summed over the colour channels, gg = sqrt(Gx^2 + Gy^2) [n_img][H*W]; then
 *   soft != 0: mask_f = gg / max_b(gg)            (nerf.py:140-143)
 *   soft == 0: mask_u8 = gg > mean_b(gg) * thresh (nerf.py:144-148; hard_edge_mask_mean_thresh, default 1.25).
 * ws: jt_edge_mask_ws_floats(n_img, H, W) floats of scratch; stats: [n_img][2] = {max, mean} per image.
 * The per-image reductions use a fixed order (deterministic). */
long long jt_edge_mask_ws_floats(int n_img, int H, int W);
int jt_edge_mask(const float* images, int n_img, int H, int W, int soft, float thresh, float* gg, float* ws,
                 float* stats, float* mask_f, uint8_t* mask_u8, cudaStream_t stream);
/* The render term of Graph.compute_loss (model/tensorf.py:99-124) with the pixel gathers of :101-102,113 fused:
 * rgb [n_views][n_rays][3]; images [n_cache][3][hw] (the blurred GT cache); mask [n_cache][hw], float
 * (mask_kind 1) or uint8 (mask_kind 2), or NULL (mask_kind 0); ray_idx [n_rays] pixel indices shared by all views
 * (NULL: n_rays == hw, identity); view_idx [n_views] rows of the cache (NULL: identity).
 *   mode 0: MSE(rgb, image)                                                    (tensorf.py:124)
 *   mode 1: MSE(rgb*w, image*w), w = m*edge_factor + non_edge_factor            (soft_edge_loss, :114-116)
 *   mode 2: edge_factor*MSE(rgb*m, image*m) + non_edge_factor*MSE(rgb*(1-m), image*(1-m))   (:118-122)
 * MSE = nanmean of the squared difference (base.py:259-261). ws4: 4 doubles {S_a, S_b, count_a, count_b} kept for
 * the backward; loss: 1 float. One CTA, fixed summation order. */
int jt_render_loss_fwd(const float* rgb, const float* images, const void* mask, int mask_kind, const int* ray_idx,
                       const int* view_idx, int n_views, int n_rays, int hw, int mode, float edge_factor,
                       float non_edge_factor, double* ws4, float* loss, cudaStream_t stream);
/* d loss / d rgb [n_views][n_rays][3], multiplied by the upstream gradient g_loss[0] (device scalar; NULL = 1). */
int jt_render_loss_bwd(const float* rgb, const float* images, const void* mask, int mask_kind, const int* ray_idx,
                       const int* view_idx, int n_views, int n_rays, int hw, int mode, float edge_factor,
                       float non_edge_factor, const double* ws4, const float* g_loss, float* d_rgb,
                       cudaStream_t stream);

/* ---- K3, tensor-core path of the LLFF head ---------------------------------- */
/* basis_mat (bateRF.py:130, Linear 60 -> 20) + positional_encoding (tensorBase.py:43-55) +
 * MLPRender_Fea_WeakView.forward (tensorBase.py:198-214) for 3 x 20 components, app_dim 20, hidden 32, fea_pe =
 * view_pe = 2 (options/bat_llff_VM_MLP.yaml), on tcgen05 with hi + lo bf16 operand terms (fp32-class results).
 * comps [n][60] fp32 = output of jt_vm_gather_fwd(app = 1); aidx / sidx / rays_d / n_samples / normalize_dir locate
 * the view direction of appearance sample e (ray = sidx[aidx[e]] / n_samples; normalised for NDC rays,
 * batBase.py:63-66). Outputs: rgb [n][4] (sigmoid colours, 4th float 0), featdir [n][32] (features 0..19, view
 * direction 28..30: kept for the backward). stage = NULL (inference) or jt_wv_stage_bytes(n_max) bytes, 128-byte
 * aligned: receives the bf16 operand tiles the backward GEMMs need. */
long long jt_wv_stage_bytes(int n_max);
int jt_wv_head_fwd_tc(const float* comps, const int* aidx, const int* sidx, const float* rays_d, int n_samples,
                      int normalize_dir, const float* Wb, const float* W1, const float* b1, const float* W2,
                      const float* b2, const float* W3, const float* b3, const int* n_dev, int n_max,
                      float fea_progress, float view_progress, float* featdir, float* rgb, void* stage,
                      cudaStream_t stream);
/* Autograd of the above (bf16-operand GEMMs, fp32 accumulation in TMEM). dout [n][4] = dL/d(pre-sigmoid) as
 * jt_render_bwd writes it; dcomps [n][60] fp32 = gradient w.r.t. the gathered components (input of
 * jt_vm_scatter_rays); the weight gradients are ACCUMULATED into gWb [20][60], gW1 [32][100], gb1 [32],
 * gW2 [32][32], gb2 [32], gW3 [3][44], gb3 [3] (zero-initialised by the caller).
 * All seven weight-gradient pointers NULL (since version 3): dcomps alone, bit-identical to the full call; a mix of
 * NULL and non-NULL pointers returns JT_ERR_ARG. */
int jt_wv_head_bwd_tc(const float* dout, const float* featdir, const float* Wb, const float* W1, const float* W2,
                      const float* W3, const int* n_dev, int n_max, float fea_progress, float* dcomps, void* stage,
                      float* gWb, float* gW1, float* gb1, float* gW2, float* gb2, float* gW3, float* gb3,
                      cudaStream_t stream);

/* ---- bf16 factor storage -------------------------------------------------- */
/* dst[i][j] = bf16(src[i][j]) (round to nearest even) for n_arrays <= 12 contiguous arrays of h_count[i] elements
 * (multiples of 4; src 16-byte, dst 8-byte aligned), ONE launch. Makes the gather-side bf16 copy of the VM factors
 * (reference: fp32 Parameters tensoRF.py:159-169 sampled by F.grid_sample; north star: "bf16/fp32 gathers"). */
int jt_cast_bf16_multi(int n_arrays, const void* const* h_src, void* const* h_dst, const long long* h_count,
                       cudaStream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* JT_VM_H_ */
