/* kpf_b200.h -- C ABI of libkpf_b200.so: the B200 (sm_100a) kernels of the KeypointFusion fusion hot path.
 *
 * The reference (ru1ven/KeypointFusion) has no FFI: its boundary is Python object identity (SURVEY.md 8b).
 * Each entry point below is what a ctypes binding in the reference would call instead of the cited
 * Python/PyTorch function; the host-side drop-in classes in keypointfusion_b200/ do exactly that.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch storage); nothing is allocated here;
 *   - tensors are dense row-major in the layout stated per function; "strided depth" arguments let the
 *     caller pass either the down-sampled map [B,1,fs,fs] or the full crop with row/col strides (the fused
 *     nearest down-sample of model.py:409);
 *   - launches are asynchronous on `stream`; no host synchronisation, no global state, re-entrant;
 *   - return value: 0 on success, a positive cudaError_t, or a negative KPF_ERR_* code.  No C++ exceptions.
 */
#ifndef KPF_B200_H
#define KPF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __CUDA_RUNTIME_H__
typedef struct CUstream_st* cudaStream_t;
#endif

enum { KPF_F32 = 0, KPF_BF16 = 1 };
enum { KPF_ERR_BAD_ARGUMENT = -1, KPF_ERR_UNSUPPORTED = -2 };
#define KPF_POINT_EMBED_STAGE_BYTES_PER_TILE 79200   /* kpf_point_embed stage_out / stage_in: bytes per 64-point tile */

/* Library ABI version (bumped on any signature change). */
int kpf_abi_version(void);

/* ---- a1-a3  util/img2pcl.py:11-40 Pcl_utils.getpcl  ==  dataloader/loader.py:843-893 + :1173-1186 ------------
 * img [B,1,S,S] f32 (background == 1.0), com3D [B,3], cube [B,3], M [B,3,3], cam [B,4] (fx,fy,fu,fv), S <= 256.
 * pcl_out [B,sample_num,3] f32, count_out [B] i32 (number of valid pixels P; may be NULL).
 * ranks: NULL -> built-in counter-based permutation keyed by (seed, b); else [B,sample_num] i32 ranks into the
 * row-major ordered list of valid pixels (clamped to P-1).  P == 0 -> zeros.  clamp != 0 -> clip to [-1,1]. */
int kpf_getpcl(const float* img, const float* com3D, const float* cube, const float* M, const float* cam, int B, int S,
               int sample_num, const int32_t* ranks, uint32_t seed, int clamp, float flip, float* pcl_out, int32_t* count_out,
               cudaStream_t stream);

/* Every valid point in row-major pixel order (loader.py:843-893 without the resample):
 * xyz_out [B,S*S,3] (rows >= P zero), pix_out [B,S*S] i32 flat pixel index (-1 padding; may be NULL), count_out [B]. */
int kpf_backproject_all(const float* img, const float* com3D, const float* cube, const float* M, const float* cam, int B, int S,
                        float flip, float* xyz_out, int32_t* pix_out, int32_t* count_out, cudaStream_t stream);

/* ---- a5  dataloader/loader.py:775-789 uvd_nl2xyznl_tensor, :821-834 xyz_nl2uvdnl_tensor ----------------------
 * [B,P,3] f32 -> [B,P,3] f32.  M^-1 is a closed-form fp64 adjugate (no torch.linalg.inv host sync). */
int kpf_uvd2xyz(const float* uvd, const float* center, const float* M, const float* cube, const float* cam, int B, int P,
                float img_size, float flip, float* out, cudaStream_t stream);
int kpf_xyz2uvd(const float* xyz, const float* center, const float* M, const float* cube, const float* cam, int B, int P,
                float img_size, float flip, float* out, cudaStream_t stream);

/* ---- a6  dataloader/loader.py:936-967 img2pcl_index ---------------------------------------------------------------
 * pcl [B,N,3]; depth element (b,r,c) at depth[b*depth_bs + r*depth_rs + c*depth_cs], r,c < fs.
 * closeness [B,N,K] f32; index64 [B,N,K] i64 and/or index32 [B,N,K] i32 (either may be NULL): flat cell index
 * row*fs+col of the K nearest cells in normalised 3-D space, ascending distance, ties -> lower index. K in 1..9 or 16.
 * order: NULL, or [B,N] i32 from kpf_spatial_order -- the order in which threads take the points (results identical). */
int kpf_img2pcl_index(const float* pcl, const float* depth, long long depth_bs, int depth_rs, int depth_cs, const float* center,
                      const float* M, const float* cube, const float* cam, int B, int N, int fs, float img_size, float flip, int K,
                      const int32_t* order, float* closeness, long long* index64, int32_t* index32, cudaStream_t stream);

/* ---- scheduling helper (no reference counterpart): order [B,N] i32 = the permutation that sorts each sample's points by the
 * fs x fs feature-map cell they project to (row-major cell, point id as tie break).  kpf_img2pcl_index and kpf_point_embed
 * accept it so that neighbouring threads / 128-point tiles touch neighbouring cells; outputs do not depend on it except
 * for the partition of kpf_point_embed's per-tile partial sums.  N <= 8192. */
int kpf_spatial_order(const float* pcl, const float* center, const float* M, const float* cube, const float* cam, int B, int N, int fs,
                      float img_size, float flip, int32_t* order, cudaStream_t stream);

/* ---- a4  model/model.py:466-500 offset2joint_weight (== util/generateFeature.py:166-195) ------------------------
 * offset [B,5J,fs,fs] (dtype), depth [B,1,S,S] f32 (nearest down-sampled to fs inside), kernel_vec [J] f32.
 * joint_out [B,J,3] f32 (uvd). */
int kpf_offset2joint_weight(const void* offset, int dtype, const float* depth, int B, int J, int fs, int S,
                            const float* kernel_vec, float* joint_out, cudaStream_t stream);

/* ---- a7  model/model.py:503-525 pcl_joint2offset -> out [B,N,4J] f32 (3J joint-major unit vectors, then J closeness) */
int kpf_pcl_joint2offset(const float* joint, const float* pcl, const float* kernel_vec, int B, int J, int N, float* out,
                         cudaStream_t stream);

/* ---- a8  model/model.py:297-306 K-tap weighted gathers ------------------------------------------------------------
 * feat: [B,C,HW] (dtype) with batch stride feat_batch_stride elements (lets a channel slice of a wider map be
 * passed); index [B,N,K] i64 (index_is_i64 != 0) or i32; closeness [B,N,K] f32.
 * out (dtype): element (b,n,c) at out[(b*N+n)*out_stride + out_c0 + c]  (out_stride >= out_c0 + C).
 * One launch when HW * 16 bytes <= 96 KB (the [channels x HW] slab of a channel block is transposed into shared memory and the taps
 * are read there; workspace may be NULL); larger maps take two launches through `workspace`, a caller buffer of B*HW*ceil8(C) elements
 * of dtype, 16-byte aligned (the map as channels-last rows; contents undefined). */
int kpf_gather_taps(const void* feat, int dtype, long long feat_batch_stride, int B, int C, int HW, const void* index,
                    int index_is_i64, const float* closeness, int N, int K, void* out, int out_stride, int out_c0, void* workspace,
                    cudaStream_t stream);

/* ---- a10  util/generateFeature.py:584-600 GFM.joint2heatmap: joint [B,J,joint_stride>=2] -> out [B,J,S,S] -------- */
int kpf_joint2heatmap(const float* joint, int joint_stride, int B, int J, int S, float stdv, float sigma, float* out,
                      cudaStream_t stream);

/* ---- a11  dataloader/loader.py:791-819 img2anchor_dis: joint_uvd [B,J,3] -> out [B,J,fs,fs] ---------------------- */
int kpf_img2anchor_dis(const float* joint_uvd, const float* depth, long long depth_bs, int depth_rs, int depth_cs,
                       const float* center, const float* M, const float* cube, const float* cam, int B, int J, int fs,
                       float img_size, float flip, float gamma, float* out, cudaStream_t stream);

/* ---- a16  util/generateFeature.py:59-84 GFM.joint2offset (eps 1e-8) / model/model.py:440-463 (eps 0) --------------
 * joint [B,J,3], depth [B,1,S,S] -> out [B,4J,fs,fs] f32. */
int kpf_joint2offset(const float* joint, const float* depth, int B, int J, int S, int fs, const float* kernel_vec, float eps,
                     float* out, cudaStream_t stream);

/* ---- a12 (+a10,a11 fused)  model/model.py:334-344 ---------------------------------------------------------------
 * feat_rgb [B,C,fs,fs] (dtype); joints [B,J,3] = refined_3d_joints (treated as uvd, like the reference);
 * Wa [J,C+J] = atten_spatial.weight, ba [J]; weight_dis [1]; fc_w [fs*fs], fc_b [1]; prev [B,J,C] or NULL.
 * sw_out [B,J,fs,fs] f32 (spatial_weight_loss), feat_j_out [B,J,C] f32; hm_out / gam_out [B,J,fs,fs] optional. */
int kpf_spatial_aggregate(const void* feat_rgb, int dtype, const float* joints, const float* depth, long long depth_bs,
                          int depth_rs, int depth_cs, const float* center, const float* M, const float* cube, const float* cam,
                          const float* Wa, const float* ba, const float* weight_dis, const float* fc_w, const float* fc_b,
                          const float* prev, int B, int C, int J, int fs, float img_size, float flip, float hm_std, float hm_sigma,
                          float gamma, float* sw_out, float* feat_j_out, float* hm_out, float* gam_out, cudaStream_t stream);

/* ---- a13  model/transfusion_head.py:684-708 updatedDecoder.forward (its one live TransformerDecoderLayer) ------
 * anchor [B,J,C] (queries), tokens [B,J,C] (keys = values), out_cj [B,C,J] and/or out_jc (element (b,t,c) at
 * out_jc[(b*J+t)*out_jc_stride + out_jc_c0 + c]); either may be NULL.
 * wpack (f32, contiguous): self_posembed[J*C] cross_posembed[J*C] WqT[C*C] bq[C] WkvT[C*2C] bkv[2C] WoT[C*C] bo[C]
 *   norm2.w[C] norm2.b[C] W1T[C*F] b1[F] W2T[F*C] b2[C] norm3.w[C] norm3.b[C];  "T" = transposed ([in][out]). */
int kpf_cross_decoder_layer(const float* anchor, const float* tokens, const float* wpack, int B, int J, int C, int F, int heads,
                            float* out_cj, float* out_jc, int out_jc_stride, int out_jc_c0, cudaStream_t stream);

/* ---- 8b exports off the live path: general-shape attention  model/transfusion_head.py:16-91, :94-173, :176-300, :303-556,
 * :560-632 (detrDecoder), :711-783 (spatial_aggregate_TR).  All fp32; strides are in ELEMENTS.
 * kpf_linear_rows: Y[(b,p)][o] = act(((X[(b,p)][:] + pos_row[:]) . W[o][:] + bias[o]) * scale)  = F.linear (:403-468) with the
 *   with_pos_embed addition (:141-142) and the q scaling (:468) folded in.  X element (b,p,k) at X[b*x_bs + p*x_ps + k*x_ks];
 *   pos (optional) likewise, or -- when pos_idx [B*P] i64 is given -- row pos_idx[b*P+p] of an nn.Embedding table
 *   (pos_ps = its row stride); W [O][K] row-major; bias [O] or NULL; Y element (b,p,o) at Y[b*y_bs + p*y_ps + o*y_os]. */
int kpf_linear_rows(const float* X, long long x_bs, long long x_ps, long long x_ks, const float* pos, long long pos_bs, long long pos_ps,
                    long long pos_ks, const long long* pos_idx, const float* W, const float* bias, int B, int P, int K, int O, float scale,
                    int relu, float* Y, long long y_bs, long long y_ps, long long y_os, cudaStream_t stream);

/* softmax(Q K^T + attn_mask, key_padding_mask -> -inf) V per head (:519-546).  Q (already scaled) / K / V / O element (b,p,c) at
 * base[b*bs + p*ps + c], C = H * head_dim, head_dim <= 64; attn_mask additive [Pq][Pk] f32 or NULL; key_padding_mask [B][Pk] u8
 * (non-zero = masked) or NULL; stats [B][Pq][H][2] (row max, row sum) optional, required when weights_out [B][Pq][Pk] (the
 * head-averaged attention weights, :551-554) is requested. */
int kpf_mha_core(const float* Q, long long q_bs, long long q_ps, const float* K, long long k_bs, long long k_ps, const float* V,
                 long long v_bs, long long v_ps, const float* attn_mask, const unsigned char* key_padding_mask, int B, int Pq, int Pk, int C,
                 int H, float* O, long long o_bs, long long o_ps, float* stats, float* weights_out, cudaStream_t stream);

/* y = LayerNorm(x + r) * gamma + beta over C (:150-151, :164-169): x element (b,p,c) at x[b*x_bs + p*x_ps + c*x_cs]; r [B*P][C] or
 * NULL; y element (b,p,c) at y[b*y_bs + p*y_ps + c*y_cs] (y_cs = P, y_ps = 1 writes the reference's [B,C,P] result, :172). */
int kpf_add_layernorm_rows(const float* x, long long x_bs, long long x_ps, long long x_cs, const float* r, const float* gamma,
                           const float* beta, int B, int P, int C, float eps, float* y, long long y_bs, long long y_ps, long long y_cs,
                           cudaStream_t stream);

/* DetrSinePositionEmbedding.forward (:75-91): mask [B][H][W] f32 (NULL = all ones), dim_t [D] = temperature ** (2 * (i // 2) / D)
 * -> out [B][2D][H][W] f32 (pos_y channels, then pos_x; even channels sin, odd cos). */
int kpf_sine_posembed(const float* mask, const float* dim_t, int B, int H, int W, int D, int normalize, float scale, float* out,
                      cudaStream_t stream);

/* ---- a14  model/fusion_layer.py:56-83 RGBDFusion.forward ------------------------------------------------------------
 * rgb, depth [B,C,HW] (dtype); gate_w [2][2C] = (gate_rgb.weight, gate_depth.weight), gate_b [2];
 * outputs (dtype) [B,C,HW]; attn_sum [2] f32 (pre-zeroed) accumulates the two attention maps (train_writer path) or NULL. */
int kpf_rgbd_fusion(const void* rgb, const void* depth, int dtype, const float* gate_w, const float* gate_b, int B, int C, int HW,
                    void* rgb_out, void* depth_out, void* merge_out, float* attn_sum, cudaStream_t stream);

/* AdaptiveAvgPool2d(1): x [rows,HW] (dtype) -> out [rows] f32. */
int kpf_channel_mean(const void* x, int dtype, int rows, int HW, float* out, cudaStream_t stream);

/* ---- a15  model/fusion_layer.py:101-116 ACFusion.forward (means from kpf_channel_mean) ---------------------------- */
int kpf_ac_fusion(const void* rgb, const void* depth, int dtype, const float* mean_rgb, const float* mean_depth,
                  const float* w_rgb, const float* b_rgb, const float* w_depth, const float* b_depth, int B, int C, int HW,
                  void* rgb_out, void* depth_out, void* merge_out, cudaStream_t stream);

/* ---- a15  model/fusion_layer.py:28-37 FSP.forward (FilterLayer :6-22): out = main + sigmoid(fc2(relu(fc0(mean(cat))))) * guide */
int kpf_fsp(const void* guide, const void* mainp, int dtype, const float* mean_guide, const float* mean_main, const float* w0,
            const float* b0, const float* w2, const float* b2, int B, int C, int Hd, int HW, void* out, cudaStream_t stream);

/* ---- 8f-1  model/model.py:158,:174 pointnet2_ops QueryAndGroup's ball query (pointnet2_ops 3.0.0, not vendored) ----
 * xyz [B,Np,3], centers [B,J,3] -> idx_out [B,J,nsample] i32: first nsample indices (ascending) with d2 < r^2,
 * remaining slots = first hit (0 if none). */
int kpf_ball_query(const float* xyz, const float* centers, int B, int Np, int J, float radius, int nsample, int32_t* idx_out,
                   cudaStream_t stream);

/* ---- a13 / 8f-2 on tensor cores: keypoint-token transformer stacks (csrc/token_stack.cu) ------------------------
 * One launch runs, in this order and each optional:  cross != 0: updatedDecoder's live layer (transfusion_head.py:684-708)
 * on x = anchor [B,J,128], y = tokens [B,J,128];  pre != 0: DESA's fusion conv on desa [B,3,J,128] | jf [B,J,128]
 * (model.py:160-164);  L > 0: KP_Interaction_TR.forward (model.py:45-126) with L BertLayers on
 *   - x [B,J,D] (D = 128, or 128 < D <= 144 with the D-128 extra inputs LEADING like cat([joints, feats])), or
 *   - the fusion-conv output (pre), or
 *   - cat([r3d [B,J,D-128], cross output]) (cross != 0: crossTR + final_TR fused, model.py:347-349).
 * Outputs: L > 0 -> tokens_out [B,J,128] (may be NULL), pred_out [B,J,3];  cross only -> out_cj [B,128,J] and/or out_jc.
 * wmat (16-bit canonical half-K weight tiles, hi and lo planes), wseq ((offset, count, vector layer, 0) int32 quadruples, n_weights
 * of them), wvec (f32): ops.pack_token_program.  F, Fc (FFN widths) in {16, 128}.
 * Split-precision tensor-core operands (fmt: 0 = fp16 planes, 1 = bf16 planes; csrc/tcgen05.cuh): fp32-class results;
 * fp32 accumulation, residual stream, LayerNorm, softmax and regression heads.  J <= 32. */
int kpf_token_stack(const float* x, const float* y, const float* r3d, const float* desa, const float* jf, const void* wmat,
                    const void* wseq, const float* wvec, int n_weights, int cross, int pre, int B, int J, int D, int L, int F, int Fc,
                    int fmt, float* tokens_out, float* pred_out, float* out_cj, float* out_jc, int out_jc_stride, int out_jc_c0,
                    const void* peer_bases, const int* xstep, int world, int row0, int rows_total /* fused exchange step, see below */,
                    cudaStream_t stream);

/* ---- the path's one exchange step, fused into the kernel that produces the joints (SURVEY.md 2b row C1; the reference gathers through
 * DataParallel, train.py:81).  Every rank owns an exchange buffer at the SAME offsets in peer-accessible (symmetric) memory:
 *   bytes [0,64): header, u32 `arrived` at 0 (zero initially);  then two halves of [rows_total, J, 3] f32 (double buffered by step parity).
 * kpf_token_stack with peer_bases != NULL (device array of `world` u64 base addresses of those buffers, xstep = device int step counter,
 * row0 = this rank's first row) stores pred ALSO into half (*xstep & 1), rows [row0, row0+B), of EVERY rank's buffer with peer stores
 * over NVLink and then counts the sample as arrived on every rank (system-scope release add).
 * kpf_exchange_wait is the receiving side; `inflight` is a device int flag (zero initially) saying a step's joints are on their way:
 *   mode 0, launched at the START of a step: completes the previous step if one is in flight (waits until `samples_per_step`
 *           (= rows_total) samples have arrived here, increments *xstep) -- by then the other ranks have long finished it, so no
 *           per-step rank skew sits on the critical path -- and marks the new step in flight;
 *   mode 1: completes the step in flight (end of a run / before a consumer reads the gathered tensor).
 * The gathered joints of the step whose index was *xstep when it ran are in half (index & 1).
 * No NCCL call, no host involvement; every rank must run the same number of steps. */
int kpf_exchange_wait(const void* exchange_buffer, int* xstep, int samples_per_step, int* inflight, int mode, cudaStream_t stream);

/* ---- a7-a9 fused point stage (csrc/point_embed.cu), model/model.py:295-320 ------------------------------------------
 * kpf_repack_features: f_d, f_rgb [B,128,HW], f_w [B,J,HW] (batch stride w_batch_stride elements; = img_offset[:,4J:])
 *   -> out [B,HW,288] bf16 channels-last rows (128 | 128 | J zero-padded to 32).  bf16 maps are exact in that one plane
 *   (out_lo = NULL); fp32 maps (dtype KPF_F32) are carried as two bf16 planes, out = rn(x) and out_lo = rn(x - out).
 * kpf_point_embed: feat_hi / feat_lo (NULL for bf16 maps) from above; idx [B,N,4] i32 / clos [B,N,4] f32 from kpf_img2pcl_index
 *   (K = 4); pcl [B,N,3]; joint [B,J,3] (J <= 21); order NULL or [B,N] i32 (kpf_spatial_order: tile t = points
 *   order[64t .. 64t+64)); wmat/wvec from ops.pack_point_embed -> e_out [B,N,256] 16-bit: per point the features after the four
 *   folded Conv1d+BN embeddings and both relus as a row [hi 128 | lo 128] of two planes in format fmt (0 = fp16, 1 = bf16);
 *   part_acc [B,N/64,128,32] f32 and part_ms [B,N/64,2,32] f32: per 64-point tile the softmax-aggregation numerators
 *   sum_n e[n][c]*exp(w[n][j]-max_tile) and (max_tile, sum_tile).  N % 64 == 0.  Split-precision tensor-core GEMMs
 *   (csrc/tcgen05.cuh), weights resident in tensor memory: fp32-class results.
 *   stage_out / stage_in (either or both NULL, never both set): the gathered inputs do not depend on the joints, and the two
 *   blocks of KPFusion gather the same taps (model.py:297-306 per block).  With stage_out the launch also stores every tile's
 *   gathered operand image ([B*N/64] x KPF_POINT_EMBED_STAGE_BYTES_PER_TILE bytes, 16-byte aligned); a later launch on the
 *   same maps / idx / clos / order passes it as stage_in and loads the images with the TMA engine instead of gathering
 *   (feat_hi / feat_lo / idx / clos are then not read).  Results are bit-identical to the unstaged launch. */
int kpf_repack_features(const void* f_d, const void* f_rgb, const void* f_w, long long w_batch_stride, int dtype, int B, int C, int J,
                        int HW, void* out, void* out_lo, cudaStream_t stream);
int kpf_point_embed(const void* feat_hi, const void* feat_lo, const int32_t* idx, const float* clos, const float* pcl, const float* joint,
                    const int32_t* order, const void* wmat, const float* wvec, int B, int N, int J, int HW, float kernel_size, int fmt,
                    void* e_out,
                    long long e_batch_stride /* 16-bit elements between samples of e_out, >= N*256; (N+J)*256 or more when kpf_desa_fused follows */,
                    float* part_acc, float* part_ms, void* stage_out, const void* stage_in, int num_sms, cudaStream_t stream);

/* ---- 8f-1 DESA on tensor cores (csrc/desa_fused.cu), model/model.py:129-204 + joint embeddings :323-325 ---------------
 * e / part_acc / part_ms: outputs of kpf_point_embed; pcl [B,N,3]; joint [B,J,3]; S scales with radii r0..r3 and
 * `nsample` grouped points each; wmat/wvec from ops.pack_desa.  -> desa_part [B,S,J,128] f32 (per-scale max-pooled MLP
 * outputs) and jf_out [B,J,128] f32 (embedded joint features); the 512->128 fusion conv consumes [desa_part | jf].
 * e is [B][>= N+J][256] 16-bit rows [hi | lo] (format fmt) with batch stride e_batch_stride: rows < N from kpf_point_embed; the prep
 * launch WRITES the J joint feature rows behind them (the joints are members N..N+J-1 of the grouped point set, model.py:168-169).
 * Two launches (prep: joint embedding, its W1 products, ball query; persistent tile kernel on `num_sms` CTAs, W1 / W2 planes in
 * tensor memory) that hand over through `scratch`: caller workspace of B*S*J*128*4 + B*(N+32)*16 + B*S*J*nsample*2 + B*S*4 bytes,
 * 16-byte aligned, contents undefined.  A scale whose widest ball of the launch holds <= 16 / 32 points is grouped 16 / 32 rows per
 * joint instead of nsample (the ball query pads with copies of the first hit; the max-pool does not see copies): same bits, fewer
 * tiles.  Split-precision GEMMs: fp32-class results. */
int kpf_desa_fused(void* e, long long e_batch_stride, const float* part_acc, const float* part_ms, const float* pcl, const float* joint,
                   const void* wmat, const float* wvec, int B, int N, int J, int S, int nsample, float r0, float r1, float r2, float r3,
                   int fmt, const float* jf_in /* NULL, or [B,J,128]: joint features given (stand-alone DESA.forward, model.py:166); the
                   joint embedding is skipped and part_acc / part_ms may be NULL */,
                   float* desa_part, float* jf_out, void* scratch, int num_sms, cudaStream_t stream);

/* ---- a12 on tensor cores (csrc/spatial_agg_tc.cu): same contract as kpf_spatial_aggregate for feat_rgb [B,128,fs,fs] with
 * fs*fs % 128 == 0, given as bf16 (feat_rgb_lo = NULL: exact in one plane) or as the two bf16 planes of an fp32 map
 * (kpf_split_planes); wa_packed from ops.pack_spatial_wa (atten_spatial.weight as canonical 16-bit planes, format fmt).
 * Split-precision GEMMs (csrc/tcgen05.cuh; fmt 0 = fp16 planes, 1 = bf16 planes for the computed operands): fp32-class results.
 * split > 1: each sample's cell tiles are spread over `split` CTAs; caller workspace scratch [B,split,128,32] f32 and
 * counters [B] i32 (ZERO on entry; the kernel leaves them zero again), reduction order fixed (deterministic). */
int kpf_spatial_aggregate_tc(const void* feat_rgb, const void* feat_rgb_lo, const float* joints, const float* depth, long long depth_bs,
                             int depth_rs, int depth_cs, const float* center, const float* M, const float* cube, const float* cam,
                             const void* wa_packed, const float* ba, const float* weight_dis, const float* fc_w, const float* fc_b,
                             const float* prev, int B, int C, int J, int fs, float img_size, float flip, float hm_std, float hm_sigma,
                             float gamma, int fmt, float* sw_out, float* feat_j_out, float* scratch, int* counters, int split,
                             cudaStream_t stream);

/* x [n] f32 -> hi [n] bf16 = rn(x), lo [n] bf16 = rn(x - hi): how an fp32 feature map enters the split-precision kernels. n % 4 == 0. */
int kpf_split_planes(const float* x, long long n, void* hi, void* lo, cudaStream_t stream);

/* ---- 8f-3 crop + normalise front end for in-the-wild frames (demo_RGBD.py:253-276, :378-385, :410-569) ------------------
 * depth_u16 [F,Hf,Wf] uint16 (mm), rgb_u8 [F,Hf,Wf,3] uint8 (BGR as cv2 reads it); bbox [B,4] f64 (x,y,w,h), one box per hand;
 * center [B,3] f64 (u,v,d_mm); cube [B,3] f32 (mm); cam [B,4] f64 (fx,fy,fu,fv) -- f64 because the reference computes its
 * integer crop bounds from Python floats.  Integer work is bit-exact vs the reference (cv2 INTER_NEAREST rule included).
 * frame_index [B] i32: box b reads frame frame_index[b], so a frame with several hands is uploaded and stored once;
 *   NULL: box b reads frame b (requires F == B).  An index outside [0,F) is never dereferenced: every output of that box
 *   (center_out, img_out, M_out, com3d_out, the rgb crop) is NaN; the other boxes are unaffected.
 * kpf_center_from_bbox -> center_out [B,3] f64;  kpf_crop_depth -> img_out [B,1,dsize,dsize] f32 (normalised, background 1),
 * M_out [B,3,3] f32 (frame px -> crop px), com3d_out [B,3] f32;  kpf_crop_rgb -> out [B,3,dsize,dsize] f32 in [0,1]. */
int kpf_center_from_bbox(const void* depth_u16, const double* bbox, const int32_t* frame_index, int F, int B, int Hf, int Wf, int upper,
                         int lower, double* center_out, cudaStream_t stream);
int kpf_crop_depth(const void* depth_u16, const double* center, const float* cube, const double* cam, const int32_t* frame_index, int F,
                   int B, int Hf, int Wf, int dsize, float* img_out, float* M_out, float* com3d_out, cudaStream_t stream);
int kpf_crop_rgb(const void* rgb_u8, const double* center, const float* cube, const double* cam, const int32_t* frame_index, int F, int B,
                 int Hf, int Wf, int dsize, float* out, cudaStream_t stream);

/* ---- a5 (frame half)  dataloader/loader.py:821-834 xyz_nl2uvdnl_tensor up to points3DToImg (:277-288) -----------------------
 * joints [B,P,3] f32 normalised xyz, center [B,3] f32 (mm, the com3d of the crop), cube [B,3] f32, cam [B,4] f32 ->
 * xyz_cam_out [B,P,3] f32 = joints * cube / 2 + center (camera space, mm);
 * uvd_frame_out [B,P,3] f32 = (X*fx/(Z+1e-8) + fu, flip*Y*fy/Z + fv, Z): frame pixels and depth in mm.
 * Same fp32 operations in the same order as kpf_xyz2uvd (one shared device function), which goes on through M into the crop. */
int kpf_joints_to_frame(const float* joints, const float* center, const float* cube, const float* cam, int B, int P, float flip,
                        float* uvd_frame_out, float* xyz_cam_out, cudaStream_t stream);

/* ---- 8f-4 evaluation tail (train.py:330-386, :470-488; util/generateFeature.py:681-703) -----------------------------------
 * pred, gt [B,J,3] f32 normalised xyz, cube [B,3] -> err [B,J] f32 (mm) and, if pa_err != NULL, pa_err [B,J] f32: the error
 * after GFM.rigid_align (similarity Procrustes, 3x3 SVD per sample in fp64 on the device). */
int kpf_eval_errors(const float* pred, const float* gt, const float* cube, int B, int J, float* err, float* pa_err, cudaStream_t stream);

/* ---- bring-up self-test of the tcgen05 primitives (csrc/tcgen05.cuh): D[128,N] f32 = A * B^T with bf16 operands.
 * a_mn == 0: A is [128,K] row-major (K-major operand), else A is given transposed [K,128] (MN-major operand);
 * b_mn == 0: B is [N,K] row-major, else B is given as [K,N]. */
int kpf_umma_selftest(const void* A, const void* B, float* D, int N, int K, int a_mn, int b_mn, cudaStream_t stream);

/* split-precision forms (csrc/tcgen05.cuh): D[128,N] f32 = A[128,K] * B[N,K]^T with fp32 A, B carried as (hi, lo) 16-bit planes
 * (fmt 0 = fp16, 1 = bf16), K in {16, 32, 64, 128, 256} (anything else is KPF_ERR_BAD_ARGUMENT), A read from shared memory
 * (a_tmem = 0) or from tensor memory (1); a_exact = 1 drops A's lo plane.
 * cycles (2 x int64 device, may be NULL): one GEMM issue -> completion, eight GEMMs back to back. */
int kpf_umma_split_selftest(const float* A, const float* B, float* D, int N, int K, int fmt, int a_tmem, int a_exact, long long* cycles,
                            cudaStream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* KPF_B200_H */
