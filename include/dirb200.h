/* dirb200 - C ABI of the B200-native descriptor-extraction + retrieval hot path.
 *
 * The reference (naver/deep-image-retrieval, "dirtorch") has no FFI: its boundary is a Python
 * duck-type (SURVEY.md 8b).  This header is the boundary a binding for that path would target:
 * plain C types, raw device/host pointers + sizes, a CUDA stream as void*, no torch types.
 * Each entry point names the reference call it replaces (file:line relative to the reference).
 *
 * Conventions
 *   - every function returns 0 on success, a negative DIRB200_E* code for library errors, or a
 *     positive cudaError_t; dirb200_last_error() returns a thread-local message;
 *   - "dev" pointers are device memory owned by the caller; the library allocates only inside
 *     opaque handles (packed weights, workspaces) freed by the matching *_destroy;
 *   - all launches are asynchronous on the given stream unless the name ends in _host;
 *   - a handle is bound to one device and is not re-entrant (one handle per GPU / stream);
 *   - there is NO CPU fallback: on a machine without an sm_100 device every compute entry
 *     point fails with DIRB200_ENODEVICE.
 */
#ifndef DIRB200_H_
#define DIRB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DIRB200_OK 0
#define DIRB200_EINVAL (-1)    /* bad argument                                            */
#define DIRB200_ENOTSUP (-2)   /* shape / option outside what the kernels support          */
#define DIRB200_EDRIVER (-3)   /* driver entry point (cuTensorMapEncodeTiled) unavailable  */
#define DIRB200_EOVERFLOW (-4) /* candidate buffer overflow that could not be resolved     */
#define DIRB200_ESTATE (-5)    /* handle used in the wrong state                           */
#define DIRB200_ENODEVICE (-6) /* no sm_100 CUDA device                                    */
#define DIRB200_EKEY (-7)      /* unknown tensor / option name                             */

typedef struct dirb200_net dirb200_net;     /* one ResNet-GeM network on one GPU            */
typedef struct dirb200_index dirb200_index; /* one row-shard of a descriptor database       */
typedef struct dirb200_exchange dirb200_exchange; /* this rank's window of the peer-memory exchange of a sharded search */

int dirb200_version(void);
const char* dirb200_last_error(void);
/* 0 if `device` exists and is compute capability 10.x. */
int dirb200_device_check(int device);

/* ------------------------------------------------------------------ network (extraction)
 * Replaces nets.create_model(arch, **model_options) + net.load_state_dict(sd) + net(imgs):
 * dirtorch/nets/__init__.py:24-64, dirtorch/nets/rmac_resnet.py:12-69,
 * dirtorch/nets/backbones/resnet.py:46-87,102-174, dirtorch/nets/layers/pooling.py:38-54.   */

/* Process-wide kernel selectors (they pick which kernel a launcher uses; no reference counterpart - the reference
 * delegates kernel choice to torch.backends.cudnn, utils/common.py:74-75 cudnn.benchmark / cudnn.fastest).  Set them once,
 * not concurrently with a running call: "halo" 1 (default) / 0 = 3x3 stride-1 convolutions load their input patch
 * once per tile (conv_halo.cuh) or tap by tap; "pdl" 1 (default) = programmatic dependent launch between consecutive
 * kernels; "res_variant" tile-variant selector of the residual 1x1 convolutions; "l2_prefetch" 1 = the 1x1
 * convolutions request the next tile's activation / residual boxes into L2 ahead of time; "head_fused" 1 (default) =
 * pooling + FC + L2 of the plain head as ONE persistent kernel, 0 = one kernel per phase (bit-identical results);
 * "epi_mode" epilogue organisation of the convolution kernels (bit 0: two warp groups, bit 1: early buffer release);
 * "epi_warps" 16 (default) / 8 epilogue warps in the 1x1 convolutions whose tile time is the epilogue (residual, short K).
 * dirb200_net_set_option forwards these keys here. */
int dirb200_set_global_option(const char* key, double value);
int dirb200_get_global_option(const char* key, double* value);
/* arch: "resnet18_rmac" (BasicBlock trunk) | "resnet50_rmac" | "resnet101_rmac" | "resnet152_rmac" (Bottleneck trunks,
 * rmac_resnet.py:74-88), or the FPN heads "resnet{18,50,101,152}_fpn_rmac" (mode 1) and "resnet101_fpn0_rmac" (mode 0,
 * rmac_resnet_fpn.py:92-110). */
int dirb200_net_create(const char* arch, int device, dirb200_net** out);
/* Options.
 * Model options of rmac_resnet.py:15-37 (the three marked * must be set BEFORE dirb200_net_finalize, later
 * changes return DIRB200_ESTATE): "pooling"* 0=gem 1=max 2=avg; "without_fc"* 0/1; "out_dim"*; "norm_features" 0/1;
 * "center_bias" b >= 0 (rmac_resnet.py:52-56); "gem_eps" (pooling.py:39, default 1e-6);
 * "mean0".."mean2", "std0".."std2": Normalize constants of the uint8 entry points (default resnet.py:110-111).
 * Scheduling: "chunk" images per pass of the network (0 = auto); "host_chunk" images per pipeline stage of
 * dirb200_net_forward_host (default 16); "stage_sched" 1 = run each stage in L2-sized sub-chunks ("sub0".."sub4"
 * images per sub-chunk of stem / layer1..4), 0 (default, faster as measured) = whole chunk per stage.
 * Implementation A/B switches: "conv_impl" 0 = persistent tcgen05 implicit GEMM (default), 1 = mma.sync implicit
 * GEMM (validation path), 2 = one-tile-per-CTA tcgen05 kernel (baseline); "fuse_ds" 1 (default) = projection
 * shortcut fused into conv3 as a K-concatenated GEMM; "fuse_c23" 0 (default, the fused kernel measured slower,
 * DESIGN.md section 7) / 1 where every SM gets several tiles / 2 wherever the kernel supports the shape = conv2 + conv3
 * (+ residual) of the identity blocks with 64 / 128 / 256 mid channels as one kernel (dirb200_conv_c23), "c23_variant"
 * 1 (default) = CTA pairs, 0 = one CTA per tile.  PROCESS-WIDE (they select kernels, not handle state; set
 * them once, not concurrently with a running forward): "halo" 1 (default) / 0 = 3x3 stride-1 convolutions load
 * their input patch once per tile (conv_halo.cuh) or tap by tap; "pdl" 1 (default) = programmatic dependent
 * launch between consecutive kernels; "res_variant" tile-variant selector of the residual 1x1 convolutions.
 * Diagnostics: "debug_taps" 1 = keep copies of the stage outputs for dirb200_net_debug_stage; "profile" 1 = time
 * every launch with CUDA events (dirb200_net_profile). */
int dirb200_net_set_option(dirb200_net* net, const char* key, double value);
/* One state_dict tensor by its reference key ("layer3.5.bn2.running_var", "adpool.p", "fc.weight" ...),
 * fp32 host memory, reference shape (conv OIHW).  "num_batches_tracked" keys are ignored. */
int dirb200_net_set_tensor(dirb200_net* net, const char* name, const float* host_data, const int64_t* shape,
                           int ndim);
/* Fold BN into per-channel scale/shift, repack conv weights to [Cout][KH][KW][Cin] fp16, upload. */
int dirb200_net_finalize(dirb200_net* net);
/* net(imgs): imgs_dev = NCHW fp32 normalised images (B,3,H,W); desc_dev = (B,out_dim) fp32 L2-normalised
 * descriptors; desc16_dev (optional, may be NULL) = the same in fp16.  test_dir.py:74. */
int dirb200_net_forward(dirb200_net* net, const float* imgs_dev, int B, int H, int W, float* desc_dev,
                        void* desc16_dev, void* stream);
/* Same through HOST buffers: H2D copy of the images, forward, D2H copy of the descriptors, stream sync
 * (the common.variables() -> net() -> tonumpy() sequence, common.py:205-218,23-27).  The batch is processed in
 * chunks of "host_chunk" images (option, default 16) with the H2D copy of the next chunk overlapping the compute
 * of the current one; pass pinned memory for the overlap to take effect. */
int dirb200_net_forward_host(dirb200_net* net, const float* imgs_host, int B, int H, int W, float* desc_host);
/* uint8 input (what an image decoder yields): imgs = HWC uint8 pixels (B,H,W,3); ToTensor + Normalize(mean,std)
 * (dirtorch/utils/transforms.py:27; options "mean0".."mean2", "std0".."std2", default = ImageNet values of
 * resnet.py:110-111) are applied on the fly in the stem's input stage, bit-identically to the fp32 entry points.
 * 4x fewer host->device bytes than the fp32 path (SURVEY.md 8f rank 1, first step). */
int dirb200_net_forward_u8(dirb200_net* net, const uint8_t* imgs_dev, int B, int H, int W, float* desc_dev,
                           void* desc16_dev, void* stream);
int dirb200_net_forward_host_u8(dirb200_net* net, const uint8_t* imgs_host, int B, int H, int W, float* desc_host);
/* Bilinear resize of uint8 HWC RGB images (B,H,W,3) -> (B,Ho,Wo,3), byte-identical to PIL's
 * Image.resize((Wo,Ho), Image.BILINEAR) - the `Scale` transform of dirtorch/utils/transforms.py:133-185 - so that
 * multi-scale extraction (Scale(0.7), Scale(1.4)) can stay on the GPU in front of dirb200_net_forward_u8.
 * dirb200_resize_coeffs is the host-only coefficient table of one axis (bounds_out [2*out], kk_out [out*ksize];
 * call with kk_out == NULL to query ksize). */
int dirb200_resize_bilinear_u8(const uint8_t* in_dev, int B, int H, int W, int Ho, int Wo, uint8_t* out_dev, void* stream);
int dirb200_resize_coeffs(int in_size, int out_size, int* bounds_out, int* kk_out, int* ksize_out);
/* Debug tap (needs option "debug_taps"): copy the NHWC fp16 activation after stage `what` ("stem","layer1".."layer4",
 * "fpn_c4" for FPN heads of mode 1) of the LAST chunk of the last forward into dst_dev (capacity in bytes); returns
 * its dims as {n,h,w,c}.  "layer4" and "fpn_c4" hold the last sub-chunk of that chunk (option "stage_sched").
 * Two-call protocol: dst_dev = NULL only fills dims; dims are filled as well when capacity is too small
 * (DIRB200_EINVAL), so the caller can size its buffer as n*h*w*c*2 bytes. */
int dirb200_net_debug_stage(dirb200_net* net, const char* what, void* dst_dev, size_t capacity, int dims[4],
                            void* stream);
/* Per-class CUDA-event timing of the last forward run with option "profile" = 1: out16 = 4 rows of
 * {launches, milliseconds, algorithmic FLOPs, algorithmic bytes} for 0 tcgen05 convolutions, 1 stem convolution,
 * 2 layout + maxpool, 3 head.  Synchronises the device. */
int dirb200_net_profile(dirb200_net* net, double* out16);
/* Option "profile" = 1 (next forward) or 2 (accumulate over forwards until the option is set again): per launch TYPE
 * (e.g. "1x1 256->1024 +res @64x64") the launches, CUDA-event milliseconds, algorithmic FLOPs and bytes, as JSON text.
 * Two-call protocol: buf = NULL returns the size through *needed. */
int dirb200_net_profile_table(dirb200_net* net, char* buf, size_t cap, size_t* needed);
/* Number of kernels the last forward launched / algorithmic conv+fc FLOPs of the last forward. */
int dirb200_net_last_launches(dirb200_net* net, int64_t* launches, double* flops);
int dirb200_net_destroy(dirb200_net* net);

/* ------------------------------------------------------------------ single operators
 * (the building blocks of the network, exported for parity tests and reuse)                 */

/* NCHW fp32 (B,3,H,W) -> NHWC fp16 (B,H,W,8), channels 3..7 zero.  Input staging of resnet.py:158. */
int dirb200_nchw_to_nhwc8(const float* in_dev, int B, int H, int W, void* out_dev, void* stream);
/* Conv2d(bias=False) + folded BatchNorm (+ residual add) (+ ReLU), NHWC fp16 in/out.
 * w_dev: [Cout][KH][KW][Cin] fp16; scale/shift: [Cout] fp32; res_dev may be NULL.
 * impl: 0 persistent tcgen05 (needs Cin%64==0, Cout%64==0), 1 mma.sync (needs Cin%8==0, Cout%64==0), 2 one-tile-per-CTA tcgen05.
 * resnet.py:56-63,70-85,115-118. */
int dirb200_conv_bn_act(const void* in_dev, int B, int H, int W, int Cin, const void* w_dev, int Cout, int KH,
                        int KW, int stride, int pad, const float* scale_dev, const float* shift_dev,
                        const void* res_dev, int relu, int impl, void* out_dev, void* stream);
/* conv2 + conv3 of a Bottleneck in one kernel (resnet.py:75-85): out = relu(bn3(conv1x1(relu(bn2(conv3x3(t1))))) + res).
 * t1 NHWC fp16 (B,H,W,Cm), w2 [Cm][3][3][Cm] fp16, w3 [4*Cm][Cm] fp16 (the layouts of dirb200_conv_bn_act), res / out
 * NHWC fp16 (B,H,W,4*Cm).  Cm in {64, 128, 256}, H >= 16, W >= 8, stride 1.  The conv2 output stays in shared memory as the
 * A operand of conv3 (fp16, the same rounding as the two-kernel path).  variant 1: CTA pairs - every MMA spans two SMs
 * (tcgen05 cta_group::2), each CTA loads half of every weight tile; variant 0: one CTA per tile. */
int dirb200_conv_c23(const void* t1_dev, int B, int H, int W, int Cm, const void* w2_dev, const float* scale2_dev,
                     const float* shift2_dev, const void* w3_dev, const float* scale3_dev, const float* shift3_dev,
                     const void* res_dev, void* out_dev, int variant, void* stream);
/* The stem on tensor cores: Conv2d(3, 64, 7, stride 2, pad 3, bias=False) + folded BN + ReLU, resnet.py:115-118.
 * imgs_dev NCHW fp32 (B,3,H,W); w2_dev = the [64][256] fp16 weight layout produced (on the host) by
 * dirb200_stem_pack_weight from the OIHW fp32 [64][3][7][7] tensor; ws_dev scratch of
 * dirb200_stem_workspace_bytes(B,H,W) bytes; out_dev NHWC fp16 (B,Ho,Wo,64). */
size_t dirb200_stem_workspace_bytes(int B, int H, int W);
int dirb200_stem_pack_weight(const float* w_oihw_host, void* w2_host);
int dirb200_stem_conv(const float* imgs_dev, int B, int H, int W, const void* w2_dev, const float* scale_dev,
                      const float* shift_dev, void* ws_dev, void* out_dev, void* stream);
/* MaxPool2d(3, stride 2, pad 1) on NHWC fp16.  resnet.py:119,161. */
int dirb200_maxpool_3x3s2(const void* in_dev, int B, int H, int W, int C, void* out_dev, void* stream);
/* Global pooling + (L2 over C) + FC + L2: rmac_resnet.py:59-68, pooling.py:38-40.
 * feat_dev NHWC fp16 (B,h,w,C); pooling 0 gem(p, eps) / 1 max / 2 avg; fc_w_dev [out_dim][C] fp32 (NULL = without_fc);
 * ws_dev: fp32 scratch of dirb200_head_workspace_floats(B,h*w,C,out_dim) floats. */
size_t dirb200_head_workspace_floats(int B, int HW, int C, int out_dim);
int dirb200_head_pool_fc_l2(const void* feat_dev, int B, int HW, int C, int pooling, float p, float eps,
                            int norm_features, const float* fc_w_dev, const float* fc_b_dev, int out_dim,
                            float* ws_dev, float* desc_dev, void* desc16_dev, void* stream);

/* center_bias option, rmac_resnet.py:52-56: feat[n][h][w][:] *= 1 + bilinear(align_corners) resize to (H,W) of the
 * 4x4 map holding b on its central 2x2; in place on the NHWC fp16 map that feeds the global pooling. */
int dirb200_center_bias(void* feat_dev, int B, int H, int W, int C, float b, void* stream);

/* ------------------------------------------------------------------ descriptor post-processing */

/* common.pool + F.normalize: common.py:41-55, test_dir.py:121-122.  xs_dev: (S,N,D) fp32 stacked;
 * mode 0 mean, 1 gem (signed power gemp); l2 != 0 appends the row L2 normalisation. */
int dirb200_pool_scales(const float* xs_dev, int S, int64_t N, int D, int mode, float gemp, int l2, float* out_dev,
                        void* stream);
/* Row L2 normalisation, eps as F.normalize (1e-12). */
int dirb200_l2_normalize(const float* x_dev, int64_t N, int D, float eps, float* out_dev, void* out16_dev,
                         void* stream);
/* common.whiten_features: common.py:221-239.  Y = ((X - mean) . comp^T) * colscale, optional row L2.
 * comp_dev [Dout][D] fp32 (pca.components_[:whitenv]); mean_dev [D] or NULL; colscale_dev [Dout] =
 * 1 / (whitenm * explained_variance_^whitenp) or NULL; y16_dev optional fp16 copy. */
int dirb200_whiten(const float* x_dev, int64_t N, int D, const float* comp_dev, const float* mean_dev,
                   const float* colscale_dev, int Dout, int l2norm, float* y_dev, void* y16_dev, void* stream);
int dirb200_f32_to_f16(const float* x_dev, int64_t n, void* out16_dev, void* stream);

/* ------------------------------------------------------------------ similarity + top-k
 * Replaces scores = common.matmul(q, db) (common.py:30-38, test_dir.py:145) followed by the per-query
 * ranking (generic.py:207,221; dataset.py:100; test_dir.py:36) for the first k ranks.  Ordering: exact
 * (fp64-accumulated) dot product of the fp32 rows, descending; ties -> lower index first.               */

int dirb200_index_create(int device, int dim, dirb200_index** out);
/* Attach one row shard: db32_dev [N][dim] fp32 (exact re-scoring), db16_dev [N][dim] fp16 (tensor-core pass);
 * both caller-owned and must outlive the index.  index_offset is added to every returned index
 * (row-wise sharding across GPUs, SURVEY.md 8e). */
int dirb200_index_set_db(dirb200_index* idx, const float* db32_dev, const void* db16_dev, int64_t N,
                         int64_t index_offset);
/* "eps16": bound on |fp16-path score - exact score| used for the candidate band (default 1.2e-3, valid for
 * unit-norm rows); "sample_rows": rows scored densely to seed the threshold (0 = auto); "cand_cap": per-query
 * candidate-list capacity (0 = auto; a small value forces the overflow -> tightened re-run path); "retries": gated
 * retry passes enqueued after the filter pass (default 1; they return at once unless a list overflowed);
 * "deferred_check" = 1: search calls never synchronise the host, the caller collects the status with
 * dirb200_index_check (it is also collected at the start of the next search); "profile". */
int dirb200_index_set_option(dirb200_index* idx, const char* key, double value);
/* q32_dev [Q][dim] fp32.  Outputs (device): scores_dev [Q][k] fp64 exact scores, idx_dev [Q][k] int64.
 * If N < k the tail is filled with score -inf / index -1.  Everything is enqueued on `stream`; the call then waits
 * once for the status block (overflow that the device-side retries could not resolve -> DIRB200_EOVERFLOW) unless
 * option "deferred_check" is set. */
int dirb200_index_search(dirb200_index* idx, const float* q32_dev, int Q, int k, double* scores_dev,
                         int64_t* idx_dev, void* stream);
/* The same search in two phases, for a database sharded over several GPUs.  Phase 1 runs the tensor-core passes and
 * writes to sel_dev[Q] (caller-owned) the local min(k_shard, N_local)-th best fp16-path score per query (+inf for an
 * empty shard).  The caller MIN-reduces sel_dev over the shards (ncclAllReduce, 4*Q bytes): shard g holds
 * min(k_shard, N_g) rows at or above its own value, so the minimum is a valid lower bound on the global k-th best
 * PROVIDED  sum_g min(k_shard, N_g) >= min(k, sum_g N_g)  - the caller's obligation.  k_shard = ceil(k / shards)
 * satisfies it when every shard holds at least that many rows; with small shards use a larger value (k always
 * works; deep-image-retrieval_b200/dist.py: shard_quota picks the smallest valid one from the shard sizes).  The
 * tight bound lets each shard re-score only ~1.4 * k / shards rows instead of ~1.4 * k.  Phase 2 re-scores the rows
 * within the band of max(sel_dev[q], local k-th) exactly and returns the shard's ordered list. */
int dirb200_index_search_begin(dirb200_index* idx, const float* q32_dev, int Q, int k, int k_shard, float* sel_dev,
                               void* stream);
int dirb200_index_search_finish(dirb200_index* idx, const float* q32_dev, const float* sel_dev, double* scores_dev,
                                int64_t* idx_dev, void* stream);
/* Status of the last search, for option "deferred_check": waits for it to finish; DIRB200_EOVERFLOW if a candidate
 * list still overflowed after the retry passes or more than cap2 rows sat within the band of the k-th score. */
int dirb200_index_check(dirb200_index* idx);
/* Statistics of the last search: {dense_rows, candidates_total, survivors_total, retry passes run, launches}
 * (waits for a deferred search to finish). */
int dirb200_index_last_stats(dirb200_index* idx, int64_t stats[5]);
/* With option "profile" = 1: CUDA-event milliseconds of the phases of the last search (valid after its status was
 * collected), out9[0..6] = {query fp16 conversion + clears, seed GEMM, seed k-th select, filter GEMM, candidate k-th
 * select, gated retry passes (+ any cross-shard exchange between the phases), survivors + exact re-scoring + sort}. */
int dirb200_index_last_profile(dirb200_index* idx, double out9[9]);
int dirb200_index_destroy(dirb200_index* idx);

/* Rank statistics for AP without the Q x N score matrix (replaces the per-query np.argsort of generic.py:207,221 +
 * junk removal :204-206,216-221 as far as the positions of the labelled rows are concerned).  Targets = the labelled
 * rows of each query, grouped by query: t_off[Q+1] (CSR), t_q[T] (query of target t), t_rows[T] GLOBAL database
 * indices, t_flags[T] (1 = count the rows ranking before this target - the positives; 0 = score only - junk rows).
 *   dirb200_index_target_scores: t_score_dev[t] = exact score <q, db[row]> for rows this shard owns, 0 otherwise
 *                                (several shards: SUM all-reduce of t_score_dev, 8*T bytes).
 *   dirb200_index_rank_count:    above_dev[t] = number of rows OF THIS SHARD that rank before target t under the
 *                                order of dirb200_index_search (exact score desc, ties -> lower global index), for
 *                                flagged targets (several shards: SUM all-reduce of above_dev).  t_score_dev must hold
 *                                the complete scores.  One tensor-core pass; queries whose candidate list overflows
 *                                ("count_cap", default 32768 rows scoring above their lowest positive) are counted
 *                                exactly from the fp32 rows instead (last_stats[3] = number of such queries).
 *                                Synchronises the stream.  Rows are assumed unit-norm (option "eps16"). */
int dirb200_index_target_scores(dirb200_index* idx, const float* q32_dev, int Q, const int* t_q_dev,
                                const int64_t* t_rows_dev, int T, double* t_score_dev, void* stream);
int dirb200_index_rank_count(dirb200_index* idx, const float* q32_dev, int Q, const int* t_off_host, const int* t_off_dev,
                             const int64_t* t_rows_dev, const unsigned char* t_flags_dev, const double* t_score_dev,
                             int T, int64_t* above_dev, void* stream);

/* Merge G per-shard top-k lists (scores fp64 + global indices int64, as produced by an all-gather of
 * dirb200_index_search outputs: each list ordered best first, empty slots = index -1 at the tail, no row in two
 * lists) into the global top-k with the same ordering rule.  Shard g's [Q][k] block starts
 * shard_stride elements after shard g-1's (0 = dense [G][Q][k]); a packed all-gather buffer [G][2][Q][k] uses
 * shard_stride = 2*Q*k with idx_dev = scores_dev + Q*k. */
int dirb200_topk_merge(const double* scores_dev, const int64_t* idx_dev, int G, int Q, int k, int64_t shard_stride,
                       double* out_scores_dev, int64_t* out_idx_dev, void* stream);
/* Sharded search over PEER MEMORY (one process per GPU of one NVLink / NVSwitch box; the reference's analogue of a
 * multi-GPU database is nn.DataParallel, utils/common.py:155, and scores = matmul(q, db) over the whole database,
 * common.py:30-38 + datasets/generic.py:207).  Every rank creates an exchange window (device buffer for up to max_q
 * queries x max_k results from `world` <= 8 ranks), hands its 64-byte CUDA IPC handle to the others (any transport:
 * torch.distributed, MPI, a file), and opens theirs.  dirb200_index_search_sharded then runs the whole two-phase
 * protocol on the caller's stream without any library collective: seed bounds, selection thresholds and the per-shard
 * lists are written by the producing kernels straight into every peer's window (stores over NVLink), the consuming
 * kernels wait on flags in their own window - two MIN all-reduces and the all-gather fused into the search kernels.  The
 * first MIN (every shard's k_shard-th seed bound) tightens the filter threshold of all shards before their filter pass:
 * ~k_shard / k of the candidates a stand-alone shard search captures.  It is a collective
 * call: every rank calls it the same number of times with the same Q, k, k_shard (k_shard: see _search_begin).
 * Results: global exact top-k on every rank.  Never synchronises; collect the status with dirb200_index_check
 * (DIRB200_EOVERFLOW also when a peer did not arrive within ~10 s).
 *   _open        handles = world x 64 bytes in rank order (entry `rank` is ignored)
 *   _open_local  same-process variant: all = the `world` exchange objects of this process (several shards driven by
 *                one process, tests); the four phases of the search (1 seed pass + seed bounds, 2 filter pass + selection
 *                thresholds, 3 exact re-scoring + lists, 4 merge) can then be issued shard by shard on one stream with
 *                dirb200_index_search_sharded_phase: phase p for every shard before phase p + 1 of any. */
int dirb200_exchange_create(int device, int world, int rank, int max_q, int max_k, dirb200_exchange** out);
int dirb200_exchange_ipc_handle(dirb200_exchange* x, void* handle64_out);
int dirb200_exchange_open(dirb200_exchange* x, const void* handles);
int dirb200_exchange_open_local(dirb200_exchange* x, dirb200_exchange* const* all);
int dirb200_exchange_close_peers(dirb200_exchange* x);   /* unmap the peers' windows; barrier among the ranks; then _destroy */
int dirb200_exchange_destroy(dirb200_exchange* x);
int dirb200_index_search_sharded(dirb200_index* idx, dirb200_exchange* x, const float* q32_dev, int Q, int k, int k_shard,
                                 double* scores_dev, int64_t* idx_dev, void* stream);
int dirb200_index_search_sharded_phase(dirb200_index* idx, dirb200_exchange* x, int phase, const float* q32_dev, int Q, int k,
                                       int k_shard, double* scores_dev, int64_t* idx_dev, void* stream);
/* Full exact score matrix (fp64 accumulate, fp32 out): the literal common.matmul for small evaluation sets. */
int dirb200_scores_exact(const float* q_dev, int Q, const float* db_dev, int64_t N, int D, float* out_dev,
                         void* stream);
/* Alpha query expansion, test_dir.py:24-44:  out_i = normalize(mean([q_i] + [db_j * s_ij^alpha, j in topk(i)])).
 * nn_idx_dev/nn_scores_dev: [Q][k] neighbour indices (-1 = none) and their scores.  Sharded mode (partial != 0, or
 * n_rows > 0): the indices are GLOBAL and db32_dev holds the rows [row_offset, row_offset+n_rows) of a sharded
 * database; neighbours owned by other shards are skipped (an EMPTY shard, n_rows == 0 with partial != 0, owns none and
 * may pass db32_dev = NULL).  Otherwise (partial == 0 and n_rows <= 0) the indices are plain rows of db32_dev.
 * partial != 0 writes the un-normalised SUM over the owned neighbours only, for a cross-GPU all-reduce. */
int dirb200_aqe_expand(const float* q_dev, int Q, int D, const float* db32_dev, const int64_t* nn_idx_dev,
                       const double* nn_scores_dev, int k, double alpha, int partial, int64_t row_offset, int64_t n_rows,
                       float* out_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DIRB200_H_ */
