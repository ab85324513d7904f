/* pips_b200 -- C ABI of the B200-native PIPs refinement hot path.
 *
 * The reference (aharley/pips) has no FFI / plugin registry: its boundary is the Python class
 * nets.pips.Pips (nets/pips.py:400-611).  This header is what a reference-side binding (ctypes,
 * see INTEGRATION.md) calls instead of the torch ops inside Pips.forward's refinement loop
 * (nets/pips.py:459-559).  Every entry point:
 *   - takes plain device pointers, sizes and a CUDA stream handle (cudaStream_t as void*),
 *   - launches asynchronously on that stream, never allocates device memory, never synchronises,
 *   - returns 0 on success, non-zero on error with the message available from pips_last_error().
 * All tensors are contiguous unless a leading dimension is given.  S (frames per window) must be 8
 * and the feature dimension 128, as in every caller of the reference (nets/pips.py:401,:408).
 *
 * Layouts
 *   fmaps        (B*S, 128, H8, W8) fp32 NCHW              output of fnet           nets/pips.py:444-445
 *   pyramid      4 levels, (B*S, H_l, W_l, 128) NHWC       avg-pool chain           nets/pips.py:346-352
 *   coords       (B, S, N, 2) fp32, feature-map pixels     loop state               nets/pips.py:453
 *   ffeats       (B*N, S, 128) fp32                        loop state               nets/pips.py:466,:522
 *   mixer rows   r = (b*N + n)*S + s                       the "(B*N, S, C)" order  nets/pips.py:516-522
 */
#ifndef PIPS_B200_H
#define PIPS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PIPS_B200_ABI_VERSION 3

enum { PIPS_S = 8, PIPS_C = 128, PIPS_LEVELS = 4, PIPS_RADIUS = 3 };
enum { PIPS_KITCHEN = 519, PIPS_KITCHEN_PAD = 576, PIPS_DIM = 512, PIPS_HIDDEN = 2048, PIPS_DEPTH = 12, PIPS_HEAD = 1040 };

/* storage type of the correlation pyramid */
enum { PIPS_FEAT_F32 = 0, PIPS_FEAT_BF16 = 1 };
/* arithmetic of the mixer's dense layers */
enum { PIPS_PREC_F32 = 0,      /* fp32 CUDA-core GEMMs (exact; validation / small problems)            */
       PIPS_PREC_BF16X3 = 1,   /* tcgen05, operands split hi+lo bf16, 3 MMAs per product (~fp32)       */
       PIPS_PREC_BF16 = 2 };   /* tcgen05, plain bf16 operands (fast mode, does not meet 1e-3 px)      */
/* GEMM epilogues */
enum { PIPS_EPI_BIAS = 0,        /* out_f32 = acc + bias                                              */
       PIPS_EPI_BIAS_GELU = 1,   /* out    = gelu_erf(acc + bias)  (bf16 hi[/lo] or fp32)             */
       PIPS_EPI_BIAS_RESID = 2 };/* out_f32 += acc + bias                                             */

int pips_abi_version(void);
const char* pips_last_error(void);

/* nets/pips.py:346-352 (CorrBlock.__init__): NCHW fp32 fmaps -> 4-level channels-last pyramid.
 * lvl_f32[l] are always written (level 0 is the transposed input); lvl_bf16[l], when the array is
 * non-NULL, receive the same values rounded to bf16. */
int pips_pyramid_build(const float* fmaps_nchw, int frames, int H, int W,
                       float* const* lvl_f32, void* const* lvl_bf16, void* stream);
/* same, for feature maps that are already channels-last (B*S, H, W, 128) -- what the fused encoder path emits */
int pips_pyramid_build_nhwc(const float* fmaps_nhwc, int frames, int H, int W,
                            float* const* lvl_f32, void* const* lvl_bf16, void* stream);

/* utils/samp.py:5-78 via nets/pips.py:463-466: bilinear gather of frame 0 at the query (indices
 * clamped, weights not), broadcast over S.  coords is the full (B,S,N,2) state (frame 0 is read). */
int pips_init_gather(const float* lvl0_f32, int B, int S, int N, int H, int W, const float* coords,
                     const int* frame_base /* NULL or [B*N] */, int frames_per_batch,
                     float* ffeat /* (B*N,128) */, float* ffeats /* (B*N,S,128) */, void* stream);

/* nets/pips.py:502,:513 (CorrBlock.corr + .sample) fused with the layout glue :517-522 and
 * utils/misc.py:44-69 (get_3d_embedding): writes the 519-wide mixer input row
 *   [ ffeat 128 | corr 4x49 | sin/cos(flow_x) 64 | (flow_y) 64 | (t) 64 | flow_x flow_y t | 0-pad to 576 ]
 * for every (b,n,s) without materialising the all-pairs volume.  Any of x_hi/x_lo/x_f32 may be NULL.
 * Chained long-video tracking (chain_demo.py:40-83): when frame_base is non-NULL the pyramid holds
 * frames_per_batch (T) frames per batch element and track (b,n) reads frames min(frame_base[b*N+n] + s, T-1). */
int pips_corr_gather(const void* const* lvl, int feat_dtype, int B, int S, int N, int H, int W,
                     const float* coords, const float* ffeats, const float* times /* [S] */,
                     const int* frame_base /* NULL or [B*N] */, int frames_per_batch,
                     void* x_hi, void* x_lo, float* x_f32, int ldx, void* stream);

/* nn.Linear on tensor cores: out = epi(A[M,K] . W[N,K]^T + bias).  a_lo/w_lo NULL => plain bf16. */
int pips_gemm_tc(const void* a_hi, const void* a_lo, int lda, int a_rows,
                 const void* w_hi, const void* w_lo, int ldw, int w_rows,
                 int M, int N, int K, const float* bias, int epilogue,
                 float* out_f32, int ldo, void* out_hi, void* out_lo, int ldh, void* stream);

/* the same contract in fp32 on CUDA cores (PIPS_PREC_F32) */
int pips_gemm_f32(const float* a, int lda, const float* w, int ldw, int M, int N, int K,
                  const float* bias, int epilogue, float* out, int ldo, void* stream);

/* nets/pips.py:117 (token-mixing PreNormResidual: LN -> Conv1d(8,32,1) -> GELU -> Conv1d(32,8,1) -> +x)
 * followed by the LayerNorm of the channel-mixing block (:118, :100), in place on x (seqs*8, 512).
 * y_* receive LN2(x_new) as the A operand of FC1. */
int pips_tokenmix(float* x, int seqs, const float* ln1_w, const float* ln1_b,
                  const float* w1 /* (32,8) */, const float* b1, const float* w2 /* (8,32) */, const float* b2,
                  const float* ln2_w, const float* ln2_b, void* y_hi, void* y_lo, float* y_f32, void* stream);

/* the same with the two contractions as tcgen05 MMAs (channels as the M dimension, bf16x3 folded into K); bf16
 * outputs only.  Selected inside pips_tokenmix by PIPS_B200_TOKENMIX=tc; see csrc/tokenmix_tc.cu for its status. */
int pips_tokenmix_tc(float* x, int seqs, const float* ln1_w, const float* ln1_b, const float* w1, const float* b1,
                     const float* w2, const float* b2, const float* ln2_w, const float* ln2_b, void* y_hi, void* y_lo,
                     void* stream);

/* nets/pips.py:120-121: final LayerNorm(512) then mean over the S rows of each sequence. */
int pips_ln_pool(const float* x, int seqs, const float* ln_w, const float* ln_b,
                 void* p_hi, void* p_lo, float* p_f32, void* stream);

/* ---- results written straight into every rank's memory over NVLink (SURVEY.md section 8e: "fusing the coord
 * all-gather into the update epilogue") ----
 * Particle-sharded runs: rank g owns particles [n_offset, n_offset + N) of n_total.  out[r] is rank r's copy of the
 * FULL (B,S,n_total,2) result of the current iteration, mapped into this process (pips_peer_open; out[own rank] is
 * the local allocation).  The update kernel stores its slice into all of them, so after pips_peer_barrier every
 * rank holds the whole result and no collective library call sits on the data path.  n_peers == 0: off. */
#define PIPS_MAX_PEERS 16
typedef struct pips_peer_out {
    float* out[PIPS_MAX_PEERS];
    int n_peers, n_offset, n_total;
} pips_peer_out;

/* cudaMalloc + cudaIpcGetMemHandle: *ptr is the local allocation, handle (64 bytes) goes to the other ranks. */
int pips_peer_alloc(size_t bytes, void** ptr, unsigned char* handle64);
/* cudaIpcOpenMemHandle (peer access enabled lazily) / cudaIpcCloseMemHandle / cudaFree */
int pips_peer_open(const unsigned char* handle64, void** ptr);
int pips_peer_close(void* ptr);
int pips_peer_free(void* ptr);
/* copy src (rows, cols) fp32, contiguous, into dst[r] (rows, cols_total) at column col_offset, for r < n_peers */
int pips_peer_scatter(const float* src, int rows, int cols, float* const* dst, int n_peers, int cols_total, int col_offset,
                      void* stream);
/* flag barrier across the ranks of one node: store `epoch` into flags[r][rank] of every rank r (system-scope release
 * after a system fence), then wait until flags[rank][r] >= epoch for all r.  flags[r] is rank r's int[PIPS_MAX_PEERS]
 * array as mapped here.  Traps after timeout_ms (a lost rank must not hang the device). */
int pips_peer_barrier(int* const* flags, int rank, int n_peers, int epoch, int timeout_ms, void* stream);

/* nets/pips.py:525-539: split delta, ffeats += GELU(Linear(GroupNorm(1,128)(dfeat))), coords += dcoord,
 * re-lock frame 0, emit coords*stride.  delta is (B*N, S*130). */
int pips_update(const float* delta, float* coords, const float* coords0, float* ffeats,
                const float* gn_w, const float* gn_b, const float* wu /* (128,128) */, const float* bu,
                float* out_px /* (B,S,N,2) */, float stride, int B, int S, int N, void* stream);
/* pips_update that also stores coords*stride into every rank's full-size result (peer may be NULL) */
int pips_update_peer(const float* delta, float* coords, const float* coords0, float* ffeats,
                     const float* gn_w, const float* gn_b, const float* wu, const float* bu,
                     float* out_px, float stride, int B, int S, int N, const pips_peer_out* peer, void* stream);

/* nets/pips.py:559: vis_e = Linear(128,1)(ffeats) -> (B,S,N) logits */
int pips_vis_head(const float* ffeats, const float* w, const float* b, float* vis, int B, int S, int N, void* stream);

/* nets/pips.py:504-511 for chosen particles only (SURVEY.md 8f-3): the dense score map
 *   fcp[b,s,j,:,:] = sum_l interpolate(<ffeats[b,s,sel[j]], fmaps_l[b,s]> / sqrt(C), (H8,W8), bilinear, align_corners=True)
 * read from the pyramid levels (channels-last, feat_dtype); ffeats is the loop state ((b*N+n), s, c).
 * sel[n_sel]: particle indices in [0,N); slot[n_sel] (or NULL = identity): position of query j in the output;
 * out element (b*S+s, slot, y, x) lives at out[(b*S+s)*out_frame_stride + (slot*H8 + y)*W8 + x].
 * scratch: pips_heatmap_scratch_floats(B*S, n_sel, H8, W8) floats. */
size_t pips_heatmap_scratch_floats(int frames, int n_sel, int H8, int W8);
int pips_heatmap(const void* const* lvl, int feat_dtype, int B, int S, int N, int H8, int W8, const float* ffeats,
                 const int* sel, const int* slot, int n_sel, float* scratch, float* out, size_t out_frame_stride, void* stream);

/* ---- score-map loss of a supervised evaluation call (nets/pips.py:58-90 score_map_loss with :14-37 balanced_ce_loss,
 * on the score maps of :502-511), without the dense (B,S,I,N,H8,W8) score maps.  Always bf16x3 on tcgen05, whatever
 * the mixer precision.  Order per forward: pips_score_grid once after the pyramid, pips_score_loss once per iteration
 * before pips_refine_iter (it reads the ffeats the iteration starts from), pips_score_loss_finalize once at the end.
 *
 * Replaces nets/pips.py:504-511 for the loss: bilinear interpolation is linear, so every score map is <f, Gr> with
 *   Gr = sum_l interpolate(lvl_f32[l] -> H8 x W8, bilinear, align_corners=True) / sqrt(128)
 * grid: (2, frames, Ppad, 128) bf16 -- the hi plane, then the lo plane (Gr ~= hi + lo); Ppad = H8*W8 rounded up to
 * PIPS_SCORE_TILE, padding rows zero. */
enum { PIPS_SCORE_TILE = 256 };
int pips_score_grid(const float* const* lvl_f32, int frames, int H8, int W8, void* grid, void* stream);
/* floats of the `partial` buffer for rows = B*S*n_total tracks and `iters` iterations (0 for an empty problem) */
size_t pips_score_loss_scratch_floats(int rows, int iters, int H8, int W8);
/* nets/pips.py:58-90 per iteration, for particles [n_offset, n_offset + N) of n_total: the GEMM of the score maps with
 * an epilogue that writes, per (track, 128-pixel block), the sum of softplus(fcp) over the block's pixels other than the
 * target, and fcp at the target.  ffeats (B*N, S, 128) fp32 is the loop state of this call's particles; target
 * (B, S, n_total) int32 holds y*W8 + x of the rounded ground truth (stride-scaled), or -1 for a track the loss excludes
 * (outside the map, valids == 0 or vis_g == 0).  Every partial depends only on its (track, pixel block): chunking the
 * particles over several calls gives identical bits. */
int pips_score_loss(const void* grid, int B, int S, int N, int H8, int W8, const float* ffeats, const int* target,
                    int n_offset, int n_total, int iter, int iters, float* partial, void* stream);
/* nets/pips.py:14-37 + :58-90 (masked means): reduces the partials of all iterations in fp64 in a fixed order, counts
 * the kept tracks K from target, and writes ce = sum_pos / (1e-6 + K*I) + sum_neg / (1e-6 + K*I*(H8*W8 - 1)) (fp32,
 * 0 when K = 0) to *ce. */
int pips_score_loss_finalize(const int* target, int rows, int iters, int H8, int W8, float* partial, float* ce, void* stream);

/* v -> (hi, lo) bf16 with hi = rn(v), lo = rn(v - hi); lo may be NULL.  Used to pack weights. */
int pips_split_bf16(const float* src, void* hi, void* lo, size_t n, void* stream);

/* ---- channels-last element-wise stages of fnet (BasicEncoder, nets/pips.py:131-281; upstream of the loop) ----
 * InstanceNorm2d statistics of y (N, HW, C) NHWC: stats = [N][2][C] (mean, rstd); partial is [N][chunks][2][C] scratch. */
int pips_inorm_stats(const float* y, int N, int HW, int C, float* partial, int chunks, float* stats, void* stream);
/* out = relu_out?( relu_main?( norm(y) ) + norm?(r) ); written as plain fp32 and/or as the [hi|lo|hi] TF32 split
 * (3*C channels at row stride split_ld) that conv2d_3xtf32 consumes.  stats_y / r / stats_r may be NULL. */
int pips_inorm_apply(const float* y, const float* stats_y, const float* r, const float* stats_r, int relu_main, int relu_out,
                     float* out_plain, float* out_split, int split_ld, int N, int HW, int C, void* stream);
/* F.interpolate(bilinear, align_corners=True) (nets/pips.py:269-272) of src (N,Hs,Ws,C) into channels
 * [c_off, c_off+C) of the split concat dst (N,Ho,Wo,3*Ctot). */
int pips_resize_split3(const float* src, int N, int Hs, int Ws, int C, float* dst, int Ho, int Wo, int Ctot, int c_off,
                       void* stream);

/* bf16 (hi, lo) flavours of the two functions above: the operand layout of pips_conv_tc (row stride pair_ld /
 * Ctot channels).  The K-padding channels are written as zero by these calls themselves: pips_inorm_apply_pair
 * zeroes [C, pair_ld); pips_resize_pair zeroes [c_off+C, Ctot) when fewer than 64 channels remain after its slice
 * (i.e. the slice is the last one before the padding of a row padded to a multiple of 64). */
int pips_inorm_apply_pair(const float* y, const float* stats_y, const float* r, const float* stats_r, int relu_main, int relu_out,
                          float* out_plain, void* out_hi, void* out_lo, int pair_ld, int N, int HW, int C, void* stream);
int pips_resize_pair(const float* src, int N, int Hs, int Ws, int C, void* dst_hi, void* dst_lo, int Ho, int Wo, int Ctot, int c_off,
                     void* stream);
/* nn.Conv2d (3x3 / 1x1, stride 1 / 2; nets/pips.py:135-136,:170,:221-223) as an implicit GEMM on the tensor cores
 * (tcgen05, CTA pairs, bf16x3).  x_hi/x_lo (N,H,W,Cp) bf16 with Cp % 64 == 0; w_hi/w_lo (BN, R*S*Cp) bf16,
 * k = (r*S + s)*Cp + ci, BN = Cout rounded up to 64/128/256 with zero rows; out (N,Ho,Wo,Cout) fp32; bias may be NULL. */
int pips_conv_tc(const void* x_hi, const void* x_lo, int N, int H, int W, int Cp, const void* w_hi, const void* w_lo,
                 int Cout, int R, int S, int stride, int pad, const float* bias, float* out, void* stream);

/* 3x3 / stride 1 / pad 1 convolution with 64 input and 64 output channels (BasicEncoder layer1, nets/pips.py:135-136):
 * every input row is loaded once into a ring of row buffers and serves all 9 filter taps (csrc/conv_rows.cu).
 * x_hi/x_lo (N,H,W,64) bf16, w_hi/w_lo (64, 9*64) bf16 [k = (r*3+s)*64 + ci], out (N,H,W,64) fp32.  partial (optional):
 * (N, pips_conv_rows_chunks(H,W), 2, 64) per-chunk (sum, sum of squares) of `out` per channel -- the InstanceNorm
 * statistics (nets/pips.py:154-157), reduced by pips_inorm_finalize. */
int pips_conv_rows_chunks(int H, int W);
int pips_conv_rows(const void* x_hi, const void* x_lo, int N, int H, int W, const void* w_hi, const void* w_lo, float* out,
                   float* partial, void* stream);
/* (mean, 1/sqrt(var + 1e-5)) per (image, channel) from `chunks` partial (sum, sum of squares) rows per image. */
int pips_inorm_finalize(const float* partial, int N, int chunks, int HW, int C, float* stats, void* stream);

int pips_conv_tc_aniso(const void* x_hi, const void* x_lo, int N, int H, int W, int Cp, const void* w_hi, const void* w_lo,
                       int Cout, int R, int S, int stride_y, int stride_x, int pad_y, int pad_x, const float* bias, float* out,
                       void* stream);
/* pips_conv_tc_aniso that also accumulates, in its epilogue, the InstanceNorm partial statistics of its output
 * (nets/pips.py:154-157): partial (N, pips_conv_tc_chunks(geometry), 2, Cout) fp32 per-chunk (sum, sum of squares) per
 * channel; the chunking depends on the image geometry only.  Reduce with pips_inorm_finalize. */
int pips_conv_tc_chunks(int H, int W, int R, int S, int stride_y, int stride_x, int pad_y, int pad_x);
int pips_conv_tc_stats(const void* x_hi, const void* x_lo, int N, int H, int W, int Cp, const void* w_hi, const void* w_lo,
                       int Cout, int R, int S, int stride_y, int stride_x, int pad_y, int pad_x, const float* bias, float* out,
                       float* partial, void* stream);
/* nets/pips.py:436 + the unfolding of the 7x7/2 stem (:206) into a 4x1 stride-1 convolution: rgb (N,3,H,W) fp32
 * (dtype 0) or bf16 (dtype 1), 0..255 -> (N, Ho+3, Wo, 64) bf16 (hi, lo), Ho = (H-1)/2+1, Wo = (W-1)/2+1; pixel (j, ox)
 * holds input rows y = 2j-3 (channels 0..31) and y = 2j-2 (channels 32..63), channel k = s*3 + colour of a row =
 * 2*(rgb/255)-1 at x = 2*ox + s - 3, zero outside the image / for k >= 21.  (ABI 3; ABI 2 unfolded the columns only.) */
int pips_stem_pack(const void* rgb, int dtype, int N, int H, int W, void* out_hi, void* out_lo, void* stream);

/* Whole-iteration operator: everything between `for itr in range(iters)` and the append of
 * coords*stride (nets/pips.py:499-539, minus the dead fcp heat-map :504-511). */
typedef struct pips_layer_weights {
    const float *ln1_w, *ln1_b, *tok_w1, *tok_b1, *tok_w2, *tok_b2, *ln2_w, *ln2_b;
    const float *fc1_b, *fc2_b;
    const void *fc1_w_hi, *fc1_w_lo, *fc2_w_hi, *fc2_w_lo;   /* bf16 (2048,512) / (512,2048)            */
    const float *fc1_w_f32, *fc2_w_f32;                      /* used by PIPS_PREC_F32 only             */
} pips_layer_weights;

typedef struct pips_weights {
    const void *in_w_hi, *in_w_lo;        /* (512, 576) bf16, K zero-padded from 519                   */
    const float* in_w_f32;                /* (512, 576) fp32                                           */
    const float* in_b;
    pips_layer_weights layer[PIPS_DEPTH];
    const float *out_ln_w, *out_ln_b;
    const void *head_w_hi, *head_w_lo;    /* (1280, 512) bf16, rows zero-padded from 1040              */
    const float* head_w_f32;              /* (1040, 512)                                               */
    const float* head_b;
    const float *gn_w, *gn_b, *upd_w, *upd_b, *vis_w, *vis_b;
} pips_weights;

typedef struct pips_workspace {
    int rows_alloc;                       /* allocated mixer rows (>= B*N*S, multiple of 128)          */
    int seqs_alloc;                       /* allocated pooled rows (>= B*N, multiple of 128)           */
    void *x0_hi, *x0_lo;  float* x0_f32;  /* (rows_alloc, 576)                                         */
    float* x;                             /* (rows_alloc, 512) residual stream                         */
    void *y_hi, *y_lo;    float* y_f32;   /* (rows_alloc, 512)                                         */
    void *h_hi, *h_lo;    float* h_f32;   /* (rows_alloc, 2048)                                        */
    void *p_hi, *p_lo;    float* p_f32;   /* (seqs_alloc, 512)                                         */
    float* delta;                         /* (seqs_alloc, 1040)                                        */
} pips_workspace;

typedef struct pips_problem {
    int B, S, N, H, W;                    /* H, W of pyramid level 0                                   */
    int feat_dtype, precision;
    const void* lvl[PIPS_LEVELS];
    const float* times;                   /* [S] = linspace(0,S,S)  nets/pips.py:519                   */
    float* coords;                        /* (B,S,N,2) in/out                                          */
    const float* coords0;                 /* (B,S,N,2) initial coords (frame 0 is re-locked)           */
    float* ffeats;                        /* (B*N,S,128) in/out                                        */
    float stride;
    const int* frame_base;                /* NULL, or [B*N] window starts for chained tracking         */
    int frames_per_batch;                 /* frames per batch element in the pyramid when frame_base   */
    pips_peer_out peer;                   /* n_peers > 0: also scatter coords*stride to every rank     */
} pips_problem;

/* DeltaBlock.forward on prepared input rows (nets/pips.py:304-311, mixer :111-123): x0 -> ws->delta */
int pips_mixer_forward(const pips_weights* w, const pips_workspace* ws, int seqs, int precision, void* stream);

/* one refinement iteration; out_px receives coords*stride (B,S,N,2) */
int pips_refine_iter(const pips_problem* p, const pips_weights* w, const pips_workspace* ws,
                     float* out_px, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PIPS_B200_H */
