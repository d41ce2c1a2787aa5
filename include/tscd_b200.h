/*
 * tscd_b200.h -- C-ABI of the B200-native TSCD aggregation stage (libtscd_b200.so).
 *
 * The reference (Video-Object-Detection/TSCD) has no FFI: its seam is the nn.Module head chosen in
 * Exp.get_model() (exps/TSCD_OVIS/ovis_tscd_large.py:106-151).  Each entry point below replaces a
 * group of eager PyTorch / torchvision / scipy calls inside TSCDHead.forward (yolox/models/tscd_head.py:
 * 374-733); the reference interface it stands in for is cited next to it.  Python binds these with ctypes
 * (tscd_b200/_lib.py); INTEGRATION.md shows the reference-side binding.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless named host_*;
 *   - no allocation inside: the caller provides outputs and workspaces sized for the worst case;
 *   - row counts that depend on the data live in device memory (counts / prefix offsets); kernels are
 *     launched over the worst case and exit early, so the whole stage runs without a host sync and can be
 *     captured in a CUDA graph;
 *   - `stream` is a cudaStream_t passed as void*;
 *   - return value: 0 on success, a negative TSCD_ERR_* otherwise (never throws).
 */
#ifndef TSCD_B200_H_
#define TSCD_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TSCD_OK 0
#define TSCD_ERR_INVALID_ARG (-1)
#define TSCD_ERR_UNSUPPORTED (-2)
#define TSCD_ERR_CAPACITY (-3)
#define TSCD_ERR_CUDA (-4)
#define TSCD_ERR_FRAME_SLOT (-5)   /* device flag of tscd_clip_assemble / tscd_frame_scatter: a frame-store slot out of range or never written */

/* element types of boundary / operand tensors */
#define TSCD_F32 0
#define TSCD_F16 1
#define TSCD_BF16 2

#define TSCD_MAX_LEVELS 3

/* Per-frame proposal capacity of the aggregation kernels.  Up to 512 proposals per frame (the default tier) every kernel
 * runs the paths it always has; the wide tier (513 .. TSCD_MAX_PROPOSALS) takes the CTA-cooperative LSAP solver of
 * tscd_cafm_lap and the global-memory merge of tscd_nms (cand_cap > 16384).  Mirrored by tscd_b200.selection.MAX_PROPOSALS. */
#define TSCD_MAX_PROPOSALS 2048

/* Strided view of one per-anchor quantity with `channels` channels over up to 3 FPN levels.
 * element(frame f, level l, local anchor a, channel c) = ptr[l] + f*frame_stride[l] + a*anchor_stride[l]
 *                                                        + c*chan_stride[l]            (strides in elements)
 * Row-major [F,A,ch] tensors use one level; NCHW conv outputs use anchor_stride=1, chan_stride=H*W;
 * channels_last conv outputs use chan_stride=1, anchor_stride=ch. */
typedef struct {
    const void* ptr[TSCD_MAX_LEVELS];
    int64_t frame_stride[TSCD_MAX_LEVELS];
    int64_t anchor_stride[TSCD_MAX_LEVELS];
    int64_t chan_stride[TSCD_MAX_LEVELS];
} tscd_view;

/* Anchor geometry: level-major, row-major within a level (tscd_head.py:374-376, 755-766). */
typedef struct {
    int32_t num_levels;
    int32_t level_h[TSCD_MAX_LEVELS];
    int32_t level_w[TSCD_MAX_LEVELS];
    int32_t level_stride[TSCD_MAX_LEVELS]; /* 8,16,32 */
    int32_t level_start[TSCD_MAX_LEVELS + 1]; /* anchor offset of each level; [num_levels] = A */
} tscd_anchors;

/* ---- K1: decode + score + select -------------------------------------------------------------------
 * Replaces: sigmoid/concat (tscd_head.py:357-359), decode_outputs (:755-770), the cxcywh->xyxy step,
 * class max, thresholding and torch.topk of TSCDHead.postprocess_widx (:1561-1624, mode B) and of
 * postpro_woclass (post_process.py:476-508, mode A).
 * Emits, per frame, a candidate list (anchor id, xyxy box, score = obj*class_conf, class id):
 *   mode A: the top-`pre_k` anchors by objectness, descending (ties: lower anchor id first);
 *   mode B: anchors with score >= conf_thresh subject to minimal/maximal limits, ascending anchor id.
 * Mode A needs the class max of the survivors only: with class-contiguous logits (cls.chan_stride == 1, channels_last
 * conv outputs) only the survivors' class rows are read; with anchor-contiguous planes (NCHW) and a workspace the class
 * max of every anchor is streamed by a separate kernel (classmax_kernel); otherwise one fused kernel streams the planes. */
typedef struct {
    int32_t mode;          /* 0 = A (postpro_woclass), 1 = B (postprocess_widx) */
    int32_t num_frames;    /* total frames in the batch (clips * frames per clip) */
    int32_t num_classes;
    int32_t head_dtype;    /* TSCD_F32 / TSCD_F16 */
    int32_t apply_sigmoid; /* 1: obj/cls are raw logits (seam S1); 0: already sigmoid-ed (S2/S3) */
    int32_t apply_decode;  /* 1: reg is (dx,dy,dw,dh) (S1/S2); 0: already decoded cxcywh (S3) */
    int32_t pre_k;         /* mode A: P */
    float conf_thresh;     /* mode B: 0.001 */
    int32_t minimal_limit; /* mode B */
    int32_t maximal_limit; /* mode B */
    int32_t cand_cap;      /* capacity (per frame) of the candidate arrays */
    tscd_anchors anchors;
    tscd_view reg, obj, cls; /* 4, 1 and C channels */
    /* outputs [num_frames, cand_cap] (SoA) + [num_frames] */
    int32_t* cand_idx;
    float* cand_box; /* [.,.,4] */
    float* cand_score;
    int32_t* cand_cls;
    int32_t* cand_count;
    /* optional workspace (mode A): with both set and anchor-contiguous class planes, the class max / arg-max of every
     * anchor is computed by a separate streaming kernel and read back for the survivors only */
    void* ws_conf;           /* [num_frames, ws_pitch] head_dtype */
    unsigned char* ws_cls;   /* [num_frames, ws_pitch] */
    int32_t ws_pitch;        /* >= A, multiple of 16 */
    /* optional [1] device flag: set to TSCD_ERR_CAPACITY when a frame selects more anchors than cand_cap (mode B without
     * a maximal_limit: the reference's list is unbounded, postprocess_widx tscd_head.py:1591-1607; the candidate arrays
     * are not).  The frame is truncated to its first cand_cap anchors and the caller must treat the batch as failed. */
    int32_t* status;
    /* optional (mode A, fused-row layout): when set, the objectness sort is SKIPPED -- candidates are emitted in ascending
     * anchor order and cand_rank[f, i] = (16-bit objectness key << 16) | (0xffff - i) carries the order instead; pass it to
     * tscd_nms as `rank` so that equal product scores keep the reference's tie order (topk order, post_process.py:506-517).
     * The selected SET, the NMS keep list and everything downstream are identical; only the order of cand_* differs. */
    uint32_t* cand_rank;
} tscd_select_args;
int tscd_select(const tscd_select_args* args, void* stream);

/* ---- head pack: the FUSED head layout (SURVEY 8(f)-2, conv-tower seam) ---------------------------------------
 * Replaces the flatten / cat / permute copies of tscd_head.py:374-376 (outputs -> [F, A, 5+C]) with ONE pass that
 * writes, per anchor, a single aligned row  [reg 4 | obj 1 | cls C | zero pad]  of `row_pitch` fp16 elements (32 = 64
 * bytes for C <= 27, 64 = 128 bytes for C <= 59) plus the objectness logits once more as a dense [F, obj_pitch] plane.
 * tscd_select / tscd_gather recognise this layout from the views (reg.ptr + 5 == cls.ptr, anchor stride == row_pitch,
 * chan stride 1) and take the row kernels of csrc/select_rows.cu: the selection streams only the 2-byte objectness plane
 * and fetches the survivors' rows as whole 64-byte sectors (from device memory or, for forward_host, in place from
 * pinned host memory). Values are copied bit-for-bit (logits stay logits; sigmoid / decode remain fused in K1 / K3). */
typedef struct {
    int32_t num_frames;
    int32_t num_classes;
    int32_t head_dtype;       /* TSCD_F16 */
    int32_t row_pitch;        /* 32 or 64 elements */
    int64_t obj_pitch;        /* elements per frame of obj_plane, >= A */
    tscd_anchors anchors;
    tscd_view reg, obj, cls;  /* inputs: 4, 1 and C channels, any strided layout */
    void* rows;               /* out [num_frames, A, row_pitch] fp16, 16-byte aligned */
    void* obj_plane;          /* out [num_frames, obj_pitch] fp16 */
} tscd_pack_head_args;
int tscd_pack_head(const tscd_pack_head_args* args, void* stream);

/* Test hook: canonical 16-bit selection key (csrc/select_rows.cu canon_key16) and fp32 score of n fp16 bit patterns.
 * tests/test_gpu_selection.py runs it over all 65536 patterns to prove that ordering by key == ordering by score. */
int tscd_debug_select_keys(const unsigned short* half_bits, int n, int apply_sigmoid, unsigned short* key, float* score,
                           void* stream);

/* ---- K2: class-aware batched NMS ---------------------------------------------------------------------
 * Replaces torchvision.ops.batched_nms (coordinate trick + nms) at tscd_head.py:1630,
 * post_process.py:58,73,510.  Keep lists are positions into the candidate arrays in descending-score order
 * (stable: ties keep the lower position first), truncated to max_keep.
 *   cand_cap <= 4096: one CTA per frame, everything in shared memory;
 *   4096 < cand_cap <= 16384 (the final per-class NMS of post_process.py:36-65 sees up to proposals x classes rows,
 *   500 x 25 = 12 500 for the shipped OVIS-L limits): three kernels over a caller-provided workspace -- per-frame class
 *   partition, one CTA per (frame, class) greedy NMS (exact whenever no cross-class pair of offset boxes exceeds the
 *   threshold, which is tested explicitly), per-frame score-ordered merge; frames that fail the test take an exact general
 *   path.  `ws` must then hold tscd_nms_workspace_bytes(num_frames, cand_cap) bytes.
 *   16384 < cand_cap <= 65536 (wide tier: 2048 proposals x 30 classes = 61 440 rows): the same partition and per-class kernels,
 *   then the merge goes through the workspace -- runs of 16384 positions sorted in shared memory, each entry ranked against the
 *   other runs by binary search; frames that fail the cross-class test run the general path over the merged order in global
 *   memory.  Same keep lists, same workspace contract (tscd_nms_workspace_bytes grows by 20 bytes per candidate row).
 * cand_cap > 65536 returns TSCD_ERR_CAPACITY from the call itself. */
typedef struct {
    int32_t num_frames;
    int32_t cand_cap;     /* row pitch of the candidate arrays */
    int32_t max_keep;     /* pitch of keep[]; mode A passes K (first K survivors) */
    float iou_thresh;
    const float* box;     /* [F,cap,4] */
    const float* score;   /* [F,cap] */
    const int32_t* cls;   /* [F,cap] */
    const int32_t* count; /* [F] */
    int32_t* keep;        /* [F,max_keep] */
    int32_t* keep_count;  /* [F] */
    int32_t* status;      /* [1] device flag: set to TSCD_ERR_CAPACITY if any frame exceeded the cap */
    void* ws;             /* workspace for cand_cap > 4096 (NULL otherwise) */
    int64_t ws_bytes;
    int32_t strict_keep;  /* 1: a frame that keeps MORE than max_keep boxes is an error (status = TSCD_ERR_CAPACITY) instead
                           * of a truncation -- mode B with pre-NMS, where max_keep is a buffer capacity and not the
                           * reference's top-K (tscd_head.py:1629-1635 keeps everything) */
    const uint32_t* rank; /* optional [F,cap] tie-break keys written by tscd_select (cand_rank): candidates are then in ascending
                           * anchor order and equal scores are ordered by DESCENDING rank (= the objectness order the reference's
                           * topk would have put them in); the low 16 bits of a rank are 0xffff - position.  Top-K use only
                           * (4 * max_keep < cand_cap <= 4096). */
} tscd_nms_args;
int tscd_nms(const tscd_nms_args* args, void* stream);
int64_t tscd_nms_workspace_bytes(int32_t num_frames, int32_t cand_cap);

/* ---- K3: rows + feature gather into the clip bank -------------------------------------------------------
 * Replaces the row build (tscd_head.py:1581-1582, 1670-1684) and find_feature_score (:976-1006).
 * For every kept proposal writes the reference row [x1,y1,x2,y2,obj,class_conf,class_pred,cls*C] (fp32),
 * its anchor id, and gathers the three 256-channel feature rows into the packed bank (row order: frames in
 * input order, proposals in selection order; offsets = exclusive prefix sum of the per-frame counts). */
typedef struct {
    int32_t num_frames;
    int32_t num_classes;
    int32_t head_dtype, apply_sigmoid, apply_decode;
    int32_t cand_cap;
    int32_t max_keep;       /* pitch of keep / rows / idx */
    int32_t use_keep;       /* 0: kept = candidates[0:count] (no pre-NMS) */
    int32_t feat_dim;       /* D (256) */
    int32_t feat_dtype;     /* dtype of the feature planes */
    int32_t bank_dtype;     /* TSCD_F16 / TSCD_BF16 / TSCD_F32 */
    tscd_anchors anchors;
    tscd_view reg, obj, cls;
    tscd_view feat_cls, feat_reg, feat_edge; /* D channels each; feat_edge.ptr[0] == NULL: no edge plane (bank_edge untouched,
                                              * filled by tscd_edge_patches / tscd_edge_combine instead) */
    const int32_t* cand_idx;
    const int32_t* cand_count;
    const int32_t* keep;
    const int32_t* keep_count;
    /* outputs */
    int32_t* sel_count;     /* [F] */
    int32_t* row_off;       /* [F+1] exclusive prefix of sel_count */
    int32_t* sel_idx;       /* [F,max_keep] anchor ids */
    float* sel_rows;        /* [F,max_keep,7+C] */
    void* bank_cls;         /* [cap_rows, D] */
    void* bank_reg;
    void* bank_edge;
    float* bank_score;      /* [cap_rows] class_conf (cls_scores) */
    float* bank_fg;         /* [cap_rows] objectness (fg_scores) */
    float* bank_box;        /* [cap_rows,4] */
} tscd_gather_args;
int tscd_gather(const tscd_gather_args* args, void* stream);

/* Offsets of the local rows (the first L frames of each clip; tscd_head.py:986-1005 concatenates them first):
 * lrow_off[b*L + f] = sum of sel_count over the local frames before (b, f); lrow_off[B*L] = total. */
typedef struct {
    int32_t B, F, L;
    const int32_t* sel_count;   /* [B*F] */
    int32_t* lrow_off;          /* [B*L+1] */
} tscd_local_offsets_args;
int tscd_local_offsets(const tscd_local_offsets_args* args, void* stream);

/* ---- Linear layer (tcgen05 GEMM) --------------------------------------------------------------------------
 * y[M,N] = x[M,K] * w[N,K]^T + bias.  Replaces every F.linear on the path (post_trans.py:613-618,687-689,
 * 1159-1161; tscd_matching.py:37-39,165-167,756; tscd_head.py:507,515-520).  x / w are fp16 or bf16 with K
 * contiguous (row pitches ldx / ldw in elements, multiples of 8; pointers 16-byte aligned); accumulation is
 * fp32 in tensor memory.  M is the row CAPACITY; if m_dev is non-null only the first min(M, *m_dev) rows are
 * computed (data-dependent row counts stay on the device).  Either or both outputs may be given. */
typedef struct {
    int32_t M, N, K;
    int32_t dtype;        /* TSCD_F16 / TSCD_BF16 operand type (also the type of out16) */
    const void* x;
    int64_t ldx;
    const void* w;
    int64_t ldw;
    const float* bias;    /* [N] or NULL */
    const int32_t* m_dev; /* device row count or NULL */
    void* out16;          /* [M, ld16] or NULL */
    int32_t ld16;
    float* out32;         /* [M, ld32] or NULL */
    int32_t ld32;
} tscd_linear_args;
int tscd_linear(const tscd_linear_args* args, void* stream);

/* ---- K4: cross-frame attention aggregation (tcgen05) -----------------------------------------------------
 * Replaces Attention_mca_g2l.forward (post_trans.py:601-714, called once per local frame by
 * MCA_tscd_g2l_reg.forward :1127-1162) and Attention_msa.forward (:734-826).
 *
 * The bank of a clip is [local rows | global rows]; a query (local row of frame f) attends to the rows of its
 * own frame and to all global rows ("no inter-frame mixing"); with self_attn=1 every row attends to every row
 * of its clip (gen-1 MSA).  Three entry points:
 *   tscd_attn_prep    per-head L2 normalisation of q,k,v (no epsilon, post_trans.py:623-628), folding of
 *                     25 * cls_score[key] into k_cls and 25 into k_reg (:658-660), the transposed value
 *                     matrices V^T per clip, and the copy of the query rows' raw v (x_ori, :680,684);
 *   tscd_attn_pv      softmax(QK^T) of both branches, attn = (attn_cls + attn_reg)/2, attn @ v_cls and
 *                     attn @ v_reg (:672-685), plus the per-row softmax statistics;
 *   tscd_attn_round2  the `ave` round (:692-712): head-mean raw-v cosine masks (> sim_thresh, > conf_sim_thresh),
 *                     softmax of the head-mean attention restricted to the mask and renormalised, times V.
 * Rows: `row_off` [B*F+1] bank offsets per frame; queries of clip b are bank rows
 * [row_off[b*F], row_off[b*F+L]); their packed output index is lrow_off[b*L] + (row - row_off[b*F]). */
typedef struct {
    int32_t B, F, L;          /* clips, frames per clip, local frames per clip */
    int32_t self_attn;        /* 1: every row is a query and every key of the clip is visible (MSA) */
    int32_t dtype;            /* TSCD_F16 / TSCD_BF16 */
    int32_t row_cap;          /* rows of the [.,256] operand arrays */
    int32_t nk_pitch;         /* columns (keys) of each V^T row; multiple of 128 */
    const int32_t* row_off;   /* [B*F+1] */
    const int32_t* lrow_off;  /* [B*L+1] (== row_off when self_attn) */
} tscd_attn_layout;

typedef struct {
    tscd_attn_layout lay;
    float scale;              /* 25 */
    const void* qkv_cls;      /* [row_cap, ld_qkv]: q | k | v (256 columns each) of the cls branch */
    const void* qkv_reg;
    int32_t ld_qkv;
    const float* key_score;   /* [row_cap] cls_score of every bank row (bank_score) */
    void *qn_cls, *kn_cls, *vn_cls, *qn_reg, *kn_reg, *vn_reg; /* [row_cap,256] outputs */
    void *vt_cls, *vt_reg;    /* [B*256, nk_pitch] outputs: V^T per clip (un-normalised v) */
    void* xori_cls;           /* [loc_cap, ld_xori] raw v of the query rows (x_ori), or NULL */
    void* xori_reg;
    int32_t ld_xori;
    int32_t* row_frame;       /* [row_cap] frame index (within its clip) of every bank row */
} tscd_attn_prep_args;
int tscd_attn_prep(const tscd_attn_prep_args* args, void* stream);

/* Fused q|k|v projection of one branch (replaces tscd_linear + tscd_attn_prep for that branch): the tcgen05 GEMM
 * x[rows,256] @ w[768,256]^T whose epilogue applies what tscd_attn_prep would do to its output -- per-head L2
 * normalisation of q (query rows only), k (x scale [x key_score]) and v, the raw-v rows of the queries (x_ori) and the
 * transposed raw v (V^T) -- straight from the fp32 accumulators; the [rows,768] q|k|v intermediate never exists.
 * row_meta / row_frame come from tscd_attn_rowmeta, which also zero-fills the padding columns of V^T. */
typedef struct {
    tscd_attn_layout lay;
    int32_t rows;             /* capacity rows of x (row_cap) */
    const int32_t* m_dev;     /* device count of valid bank rows */
    const void* x;            /* [rows, ldx] bank features (lay.dtype) */
    int64_t ldx;
    const void* w;            /* [768,256]: Wq | Wk | Wv */
    const int32_t* row_meta;  /* [rows] (clip << 16) | key index */
    const float* key_score;   /* [rows] or NULL (reg branch) */
    float scale;              /* 25 */
    void *qn, *kn, *vn;       /* [rows,256] */
    void* vt;                 /* [B*256, nk_pitch], or NULL: not computed (the reg branch of a module run with need_reg = 0) */
    void* xori;               /* [loc_cap, ld_xori] or NULL */
    int32_t ld_xori;
} tscd_qkv_project_args;
int tscd_qkv_project(const tscd_qkv_project_args* args, void* stream);

typedef struct {
    tscd_attn_layout lay;
    int32_t* row_frame;       /* [row_cap] frame index (within its clip) of every bank row */
    int32_t* row_meta;        /* [row_cap] (clip << 16) | key index within the clip */
    void* vt_cls;             /* [B*256, nk_pitch]: columns [n_clip, round-up-128) of every clip are zero-filled */
    void* vt_reg;             /* same, may be NULL */
} tscd_attn_rowmeta_args;
int tscd_attn_rowmeta(const tscd_attn_rowmeta_args* args, void* stream);

typedef struct {
    tscd_attn_layout lay;
    const void *qn_cls, *kn_cls, *qn_reg, *kn_reg;
    const void *vt_cls, *vt_reg;   /* vt_reg may be NULL when need_reg = 0 */
    const int32_t* row_frame;
    int32_t need_reg;         /* 0: skip attn @ v_reg (TSCD `agg` discards it, tscd_head.py:480) */
    void* x_cls;              /* [loc_cap, ld_x] attn @ v_cls, heads concatenated */
    void* x_reg;
    int32_t ld_x;
    float* stats;             /* [loc_cap,16]: row max (cls h0-3, reg h0-3), row sum (cls h0-3, reg h0-3) */
    float max_logit;          /* > 0 with BF16 operands: single-pass mode -- an upper bound of every logit (the key scale, 25:
                               * |q^ . k^| <= 1 and the class scores are <= 1) replaces the row maxima of pass A (BF16 probabilities keep
                               * their exponent range) and stats[0..7] = max_logit.  0, or fp16 operands: exact two-pass statistics */
} tscd_attn_pv_args;
int tscd_attn_pv(const tscd_attn_pv_args* args, void* stream);

typedef struct {
    tscd_attn_layout lay;
    const void *qn_cls, *kn_cls, *qn_reg, *kn_reg, *vn_cls, *vn_reg;
    const void* vt;           /* [B*256, nk_pitch] value matrix (transposed) to aggregate */
    const int32_t* row_frame;
    const float* stats;
    int32_t use_obj_mask;     /* 0: weights = sim_mask (cls output); 1: sim_mask * obj_mask (reg output) */
    float sim_thresh;         /* 0.75 */
    float conf_sim_thresh;    /* 0.99 */
    void* out;                /* [loc_cap, ld_out] 256 columns */
    int32_t ld_out;
    /* weight hand-over between the two launches of one module (both optional, [loc_cap, nk_pitch], lay.dtype):
     * w_out (use_obj_mask = 0): store  sim_mask * exp(mean attention);  w_in (use_obj_mask = 1): reuse it -- the launch
     * then only evaluates the reg-branch raw-v similarity (no score recomputation, no exponentials) */
    void* w_out;
    const void* w_in;
} tscd_attn_round2_args;
int tscd_attn_round2(const tscd_attn_round2_args* args, void* stream);

/* Per-clip transpose of a 16-bit row-major matrix x[row_cap, width] (width multiple of 256) into
 * xt[(b*width + c), key] (pitch nk_pitch), key = row - row_off[b*F]; pad keys are zero-filled up to the next
 * multiple of 128.  Used by the gen-1 MSA, whose round 2 aggregates linear1's OUTPUT (MSA_yolov.find_similar_round2,
 * post_trans.py:1238-1254) rather than the raw values. */
typedef struct {
    tscd_attn_layout lay;
    int32_t width;
    const void* x;
    int32_t ld_x;
    void* xt;
} tscd_transpose_args;
int tscd_transpose_clip(const tscd_transpose_args* args, void* stream);

/* ---- K5: CAFM (AwarePositionRegMatcher) -------------------------------------------------------------------
 * Replaces AwarePositionRegMatcher.forward (tscd_matching.py:722-888) with its ReferringCrossAttentionLayer
 * (:566-589), SEModule (:278-283), PositionMHAttention (:31-60), double_match_embds (:912-937) and the scipy
 * Hungarian solve (:935) -- here a device-side shortest-augmenting-path LSAP in fp64 with SciPy's tie rules.
 * The key / value projections (k_reg, v_reg) and the time-embedding Linear run as tscd_linear GEMMs before.
 *   tscd_cafm_prep   gathers the local rows' raw reg / edge features, builds the key-side input
 *                    SE(feat, edge) + time_embedding[frame], and the (|x| + 1e-6) norms used by the matching cost;
 *   tscd_cafm_chain  one CTA per clip walks its local frames in order: cost -> LSAP -> permutation ->
 *                    query = W_q (SE(prev_out, prev_edge) + prev_time) -> 8-head cosine attention over the
 *                    CURRENT frame only (no inter-frame mixing) -> LayerNorm(identity + attn) -> decoder_norm.
 * State (last frame's outputs / embeddings, tscd_matching.py:708-715) lives in caller-owned buffers so that
 * consecutive clips of one video can be chained with resume=1. */
typedef struct {
    int32_t B, F, L, D;          /* D = 256; embed dim of the matching features = 4*D */
    int32_t bank_dtype;          /* dtype of bank_reg / bank_edge and of the 16-bit outputs */
    const int32_t* row_off;      /* [B*F+1] */
    const int32_t* lrow_off;     /* [B*L+1] */
    const void* bank_reg;        /* [row_cap, D] */
    const void* bank_edge;
    const float* time_emb;       /* [B*L, D] output of absolute_position_embedding */
    const float* se_w1;          /* [32,2]  CA.fc.0.weight */
    const float* se_w2;          /* [2,32]  CA.fc.2.weight */
    const float* emb_reg;        /* [loc_cap, 4D] agg_iou reg output (matching only) */
    const float* emb_cls;        /* [loc_cap, 4D] agg_iou cls output (matching only) */
    float* feat;                 /* out [loc_cap, D] raw reg features of the local rows */
    float* edge;                 /* out [loc_cap, D] */
    void* feat16;                /* out [loc_cap, D] 16-bit copy (value projection input) */
    void* kin16;                 /* out [loc_cap, D] 16-bit key-side input SE(feat,edge)+time */
    float* kin;                  /* out [loc_cap, D] fp32 copy (first-frame query input) */
    float* norm_reg;             /* out [loc_cap] |emb_reg| + 1e-6 */
    float* norm_cls;             /* out [loc_cap] */
    int32_t emb_dtype;           /* TSCD_F32 (0): emb_* are fp32 and the norms are computed here; TSCD_F16 / TSCD_BF16: emb_* are not
                                  * read, tscd_cafm_cost computes the norms from the 16-bit embeddings */
} tscd_cafm_prep_args;
int tscd_cafm_prep(const tscd_cafm_prep_args* args, void* stream);

/* Matching costs of every local frame against its reference frame (the previous non-empty local frame in its
 * ORIGINAL row order, the carried-over state when the clip resumes, or itself for a first frame), for all clips
 * at once: cost[lf][r][c] = 1 - (cos_reg + cos_cls)/2 (tscd_matching.py:912-929), pitch kmax.  The chain kernel
 * only re-indexes rows by the previous frame's assignment. */
typedef struct {
    int32_t B, L, D, kmax;
    const int32_t* lrow_off;
    const int32_t* resume;
    const int32_t* st_n;
    const float* emb_reg; const float* emb_cls; const float* norm_reg; const float* norm_cls;
    const float* st_reg; const float* st_cls; const float* st_nreg; const float* st_ncls;
    float* cost;                 /* [B*L, kmax, kmax] */
    int32_t* ref_n;              /* [B*L] rows on the reference side of every frame's matching (0 for empty frames) */
    /* kmax <= TSCD_MAX_PROPOSALS; above 512 only the 16-bit-copy kernel below (emb_dtype TSCD_F32 with emb_reg16 / emb_cls16 set),
     * anything else returns TSCD_ERR_UNSUPPORTED.
     * TSCD_F32 (0): emb_* / norm_* as declared above (fp32 FMA kernel, any kmax <= 512).  TSCD_F16 / TSCD_BF16 (kmax <= 32): emb_reg /
     * emb_cls point to 16-bit [loc_cap, 4D] embeddings (the GEMM outputs as the tensor cores produced them), the costs run on
     * mma.sync with fp32 accumulation and norm_reg / norm_cls are OUTPUTS (written for the rows of every frame) */
    int32_t emb_dtype;
    /* optional, with emb_dtype == TSCD_F32 and kmax > 32: 16-bit copies of emb_reg / emb_cls ([loc_cap, 4D], the same GEMM's
     * 16-bit output).  When both are set the costs of the wide frames run on mma.sync tensor cores (128 x 64 tiles, fp32
     * accumulation, fp32 norms from tscd_cafm_prep; a carried fp32 state is converted while it is staged) instead of the
     * fp32 FMA kernel. */
    const void* emb_reg16;
    const void* emb_cls16;
    int32_t emb16_dtype;         /* TSCD_F16 / TSCD_BF16 */
    /* optional state slot map: clip b reads the carried state (st_*) of slot slot[b] instead of slot b.  resume, lrow_off and
     * the outputs stay indexed by the batch position b.  NULL = slot b (the state then holds exactly B slots). */
    const int32_t* slot;         /* [B] */
} tscd_cafm_cost_args;
int tscd_cafm_cost(const tscd_cafm_cost_args* args, void* stream);

/* Rectangular LSAP of every frame's cost table in parallel (one warp per frame; scipy.optimize.
 * linear_sum_assignment semantics, fp64).  The assignment of a frame does not depend on the order in which the
 * previous frame remembers its rows, so all frames are solved before the sequential chain, which only re-indexes:
 * lap_col[lf][r] = matched column of reference row r (-1: none), lap_row[lf][c] = matched reference row of column c.
 * kmax <= TSCD_MAX_PROPOSALS.  Problems with max(ref_n, n) <= 512 are solved by one warp each exactly as before; larger ones (wide
 * tier) by one 512-thread CTA each (CTA-cooperative column scan and arg-min, fp64 potentials, state in ~42 x kmax bytes of shared
 * memory), with the same scan order and tie rules, i.e. SciPy's assignment.  The solver is chosen per problem on the device. */
typedef struct {
    int32_t num_frames, kmax;
    const int32_t* lrow_off;
    const int32_t* ref_n;
    const float* cost;
    int32_t* lap_col;            /* [B*L, kmax] */
    int32_t* lap_row;            /* [B*L, kmax] */
} tscd_cafm_lap_args;
int tscd_cafm_lap(const tscd_cafm_lap_args* args, void* stream);

typedef struct {
    int32_t B, F, L, D, kmax;    /* kmax: capacity (rows per frame) of the state / scratch buffers, <= 512 */
    int32_t out_dtype;
    const int32_t* row_off;
    const int32_t* lrow_off;
    const int32_t* resume;       /* [B] 1: continue from the state buffers (tscd_matching.py:779) */
    const float* feat;           /* [loc_cap, D] */
    const float* edge;
    const float* kin;            /* [loc_cap, D] */
    const float* kproj;          /* [loc_cap, D] k_reg(kin)  (generic path) */
    const float* vproj;          /* [loc_cap, D] v_reg(feat) (generic path) */
    /* fast path (kmax <= 32): set all five and the chain runs entirely out of shared memory on mma.sync tensor-core
     * tiles; feat / edge / kin / kproj / vproj / wq_t / sc_* are then unused and may be NULL */
    const void* kproj16;         /* [loc_cap, D] k_reg(kin), 16-bit (out_dtype) */
    const void* vproj16;         /* [loc_cap, D] v_reg(feat), 16-bit */
    const void* wq16;            /* [D(out), D(in)] q_reg.weight, 16-bit */
    const void* bank_reg;        /* [row_cap, D] packed clip bank (16-bit, out_dtype): identity / unmatched-row features */
    const void* bank_edge;       /* [row_cap, D] */
    const float* time_emb;       /* [B*L, D] */
    const float* emb_reg;        /* [loc_cap, 4D] */
    const float* emb_cls;
    const float* norm_reg;
    const float* norm_cls;
    const float* wq_t;           /* [D(in), D(out)] q_reg.weight transposed, fp32 */
    const float* se_w1;
    const float* se_w2;
    const float* ln_w;           /* layer norm of the cross-attention layer */
    const float* ln_b;
    const float* dec_w;          /* decoder_norm */
    const float* dec_b;
    /* state, caller-owned, persists across calls; [B, ...] below reads [slots, ...] when `slot` is set */
    int32_t* st_n;               /* [B] rows held (0 = no memory) */
    float* st_out;               /* [B,kmax,D] */
    float* st_edge;              /* [B,kmax,D] */
    float* st_reg;               /* [B,kmax,4D] */
    float* st_cls;               /* [B,kmax,4D] */
    float* st_nreg;              /* [B,kmax] */
    float* st_ncls;              /* [B,kmax] */
    float* st_time;              /* [B,D] */
    /* scratch */
    float* sc_qin;               /* [B,kmax,D] */
    float* sc_q;                 /* [B,kmax,D] */
    float* sc_k;                 /* [B,kmax,D] */
    const int32_t* ref_n;        /* [B*L] from tscd_cafm_cost */
    const int32_t* lap_col;      /* [B*L,kmax] from tscd_cafm_lap */
    const int32_t* lap_row;      /* [B*L,kmax] */
    /* outputs */
    void* out16;                 /* [loc_cap, D] CAFM output after decoder_norm, original row order */
    float* out32;                /* [loc_cap, D] same in fp32 (may be NULL) */
    int32_t* perm;               /* [loc_cap] matched column of every output row (debug / tests; may be NULL) */
    int32_t* status;
    int32_t emb_dtype;           /* element type of emb_reg / emb_cls: TSCD_F32 (0), or 16-bit with the fast path (widened into the state) */
    /* optional state slot map: clip b reads and writes the state (st_*) of slot slot[b] instead of slot b, so a caller-owned
     * state may hold more slots than the batch (one per concurrent video stream) and a call runs any B distinct slots of it
     * without copies.  resume, the bank, the layout, the scratch and the outputs stay indexed by the batch position b.  The
     * slots of one call must be distinct.  NULL = slot b.  tscd_cafm_wide reads it through `base`. */
    const int32_t* slot;         /* [B] */
} tscd_cafm_chain_args;
int tscd_cafm_chain(const tscd_cafm_chain_args* args, void* stream);

/* Wide CAFM chain for frames of MORE than 32 proposals (mode B: 50..500 per frame, the shipped TSCD-L configurations).  The
 * recurrence over the local frames stays sequential, but every frame's step runs as batch-wide launches over all clips instead
 * of inside one CTA per clip (see csrc/cafm.cu):  phase 0 once;  per frame f: phase 1 (permutation + 16-bit query input
 * rows into qin16), then the CALLER runs tscd_linear (q = W_q qin16, rows [B*kmax]) and tscd_frame_flash (8 heads x 32, row
 * ranges q_beg/q_end/kv_beg/kv_end, keys / values = the k_reg / v_reg projections) into `attn`, then phase 2 (identity +
 * LayerNorms, outputs, state);  phase 3 once (matching embeddings into the carried state).  `base` is the argument block of
 * tscd_cafm_chain: feat / edge / kin (fp32), lap_*, state and output fields are used; kproj*, vproj*, wq*, sc_* are not. */
/* tscd_cafm_wide accepts kmax <= TSCD_MAX_PROPOSALS (tscd_cafm_chain itself stays at kmax <= 512); the permutation kernel walks
 * the frame's rows in chunks of 512, so frames of up to 2048 proposals keep the same row order and state layout. */
typedef struct {
    tscd_cafm_chain_args base;
    void* qin16;             /* out (phase 1) [B*kmax, D] 16-bit (out_dtype) */
    const float* attn;       /* in  (phase 2) [B*kmax, D] attention output of the caller's tscd_frame_flash */
    int32_t* q_beg;          /* out (phase 1) [B] row ranges for tscd_frame_flash */
    int32_t* q_end;
    int32_t* kv_beg;
    int32_t* kv_end;
    int32_t* ctl;            /* scratch [B,8] */
    int32_t* perm_s;         /* scratch [B,kmax] */
    int32_t* prow_s;         /* scratch [B,kmax] */
    int32_t* ord_prev;       /* scratch [B,kmax] */
    int32_t* n_prev;         /* scratch [B] */
    int32_t* last_l0;        /* scratch [B] */
} tscd_cafm_wide_args;
int tscd_cafm_wide(const tscd_cafm_wide_args* args, int phase, int frame, void* stream);

/* Cosine multi-head attention over ragged row sets (csrc/frame_flash.cu): for item i and every head,
 * softmax(q^ k^T) v with q = rows [q_beg[i], q_end[i]) of `q`, k / v = rows [kv_beg[i], kv_end[i]) of `k` / `v`, q and k
 * L2-normalised per head, no scale -- PositionMHAttention.forward (tscd_matching.py:31-60) and MHAttention.forward (:159-181)
 * for frames of any size (mma.sync flash kernel; head_dim 32 or 128; 16-bit q / k / v, fp32 output written at the query rows). */
typedef struct {
    int32_t num_items;
    int32_t heads, head_dim;
    int32_t dtype;               /* TSCD_F16 / TSCD_BF16 */
    int32_t max_q;               /* upper bound of q_end[i] - q_beg[i] (grid size) */
    const int32_t* q_beg; const int32_t* q_end;      /* [num_items] device */
    const int32_t* kv_beg; const int32_t* kv_end;
    const void* q; int32_t ldq;  /* row pitches in elements, multiples of 8 */
    const void* k; int32_t ldk;
    const void* v; int32_t ldv;
    float* out; int32_t ldo;
} tscd_frame_flash_args;
int tscd_frame_flash(const tscd_frame_flash_args* args, void* stream);

/* ---- WaveletsHFBlock at the selected anchors only (SURVEY 8f-2) ------------------------------------------------
 * Replaces the dense edge_enhance_reg[k](vid_feat_reg) of the head (tscd_head.py:367; surrounding_extraction.py:215-267)
 * followed by the row lookup of find_feature_score (tscd_head.py:991): the block's output is evaluated only at the kept
 * proposals.  tscd_gather is called with a null feat_edge view (it then leaves bank_edge alone) and
 *   tscd_edge_patches   writes, per kept proposal, the zero-padded 3x3 patch [9*256] (tap-major: (ky,kx), channel) and the Haar
 *                       high-pass sub-bands [LH|HL|HH] (3*256) of its 2x2 block as 16-bit rows.  Every pyramid level has its
 *                       own conv weights, so rows are grouped by level: level l owns slots [seg_base[l], seg_base[l]+seg_cap[l])
 *                       and level_count[l] (device) says how many are filled; slot[bank row] = 4*slot + 2*(y&1) + (x&1);
 *   tscd_linear         per level: content = patches x W3^T + b3 (filter2, weight [256, 9*256] tap-major) and
 *                       hf_out = hf x W1^T + b1 (filter1, weight [768,768]), m_dev = &level_count[l];
 *   tscd_edge_combine   bank_edge[row] = ReLU(content) * 1/2 (s_lh ReLU(LH') + s_hl ReLU(HL') + s_hh ReLU(HH')) (inverse Haar with
 *                       LL = 0; s_lh = -1 on odd rows, s_hl = -1 on odd columns, s_hh = s_lh * s_hl).
 * Feature maps need even height and width (the reference's stride-2 transform has no same-size inverse otherwise). */
typedef struct {
    int32_t num_frames, max_keep;
    int32_t feat_dtype;                   /* TSCD_F32 / TSCD_F16 / TSCD_BF16: type of feat_reg */
    int32_t op_dtype;                     /* TSCD_F16 / TSCD_BF16: type of patches / hf */
    tscd_anchors anchors;
    tscd_view feat_reg;                   /* 256 channels per anchor */
    const int32_t* sel_idx;               /* [num_frames, max_keep] anchor ids (tscd_gather) */
    const int32_t* sel_count;             /* [num_frames] */
    const int32_t* row_off;               /* [num_frames+1] */
    int32_t seg_base[TSCD_MAX_LEVELS];
    int32_t seg_cap[TSCD_MAX_LEVELS];
    int32_t* level_count;                 /* [TSCD_MAX_LEVELS] out (zeroed by the call) */
    int32_t* slot;                        /* [bank rows] out */
    void* patches;                        /* [slots, 2304] out */
    void* hf;                             /* [slots, 768] out */
    int32_t* status;                      /* TSCD_ERR_CAPACITY if a level's segment overflowed, or NULL */
} tscd_edge_patches_args;
int tscd_edge_patches(const tscd_edge_patches_args* args, void* stream);

typedef struct {
    int32_t rows_cap;                     /* bank row capacity (grid size) */
    int32_t op_dtype;                     /* TSCD_F16 / TSCD_BF16: type of content / hf_out / bank_edge */
    const int32_t* total_rows;            /* device: number of bank rows (= row_off[num_frames]) */
    const int32_t* slot;                  /* [bank rows] from tscd_edge_patches */
    const void* content;                  /* [slots, 256] pre-ReLU filter2 output */
    const void* hf_out;                   /* [slots, 768] pre-ReLU filter1 output */
    void* bank_edge;                      /* [bank rows, 256] out */
} tscd_edge_combine_args;
int tscd_edge_combine(const tscd_edge_combine_args* args, void* stream);

/* ---- TaskAligned attention + LayerNorms ---------------------------------------------------------------------
 * tscd_frame_attention: MHAttention.forward (tscd_matching.py:159-181) for every local frame at once:
 * per frame and head, softmax(q^ k^T) v with L2-normalised q,k (no scale), queries/keys/values all from the
 * SAME frame.  q/k/v are the GEMM outputs of the projections (tscd_linear): fp32 for the generic kernel, 16-bit for the
 * mma.sync tensor-core kernel used when every frame holds <= 32 proposals.
 * tscd_residual_ln2: y = LN_b(LN_a(x + r))  -- CrossAttentionLayer.forward_post's norm followed by the
 * decoder_norm of TaskAligned (tscd_matching.py:421-433, 1133-1137); optionally also the 1-output objectness head. */
typedef struct {
    int32_t num_frames;          /* B*L local frames */
    int32_t heads, head_dim;
    int32_t in_dtype;            /* TSCD_F32: generic kernel; TSCD_F16 / TSCD_BF16: tensor-core kernel (frames <= 32 rows, head_dim 128) */
    const int32_t* lrow_off;     /* [num_frames+1] */
    const void* q; int32_t ldq;  /* row pitches in elements */
    const void* k; int32_t ldk;
    const void* v; int32_t ldv;
    float* out; int32_t ldo;     /* [loc_cap, heads*head_dim] fp32 */
} tscd_frame_attention_args;
int tscd_frame_attention(const tscd_frame_attention_args* args, void* stream);

typedef struct {
    int32_t rows_cap, dim;
    const int32_t* n_rows;       /* device row count */
    const float* x; const float* r;
    const float *w_a, *b_a, *w_b, *b_b;
    int32_t out_dtype;
    void* out16; float* out32;   /* either may be NULL */
    /* optional fused single-output head (matcher_obj_pred, tscd_head.py:518): head_out[row] = <y_row, head_w> + head_b,
     * y = the fp32 LayerNorm output (dim 1024 only); head_w fp32 [dim], head_b fp32 [1], head_out fp32 [rows_cap] */
    const float* head_w; const float* head_b; float* head_out;
} tscd_residual_ln2_args;
int tscd_residual_ln2(const tscd_residual_ln2_args* args, void* stream);

/* ---- final per-class expansion (post_process.py:9-85) ---------------------------------------------------------
 * tscd_final_expand builds, per local frame, the two candidate lists the reference feeds to batched_nms:
 *   refined: one row per (proposal, class) with sigmoid(cls) >= thr and sigmoid(obj)*sigmoid(cls) >= thr, in
 *            row-major (proposal, class) order; box = decode_reg_preds5(deltas, still box) (tscd_head.py:914-949);
 *   still:   the unrefined rows with obj*class_conf >= thr.
 * tscd_final_rows assembles [x1,y1,x2,y2,obj,cls_score,cls_id] rows in NMS keep order. */
typedef struct {
    int32_t B, F, L, num_classes, max_keep;
    float conf_thre;             /* 0.001 */
    float xform_clip;            /* log(736/32) */
    const int32_t* sel_count;    /* [B*F] */
    const float* sel_rows;       /* [B*F, max_keep, 7+C] */
    const int32_t* lrow_off;     /* [B*L+1] */
    const float* cls_logits; int32_t ld_cls;   /* [loc_cap, >=C] */
    const float* obj_logits; int32_t ld_obj;   /* [loc_cap, >=1] */
    const float* reg_deltas; int32_t ld_reg;   /* [loc_cap, >=4] */
    /* refined candidates, capacity per frame = max_keep * num_classes */
    float* r_box; float* r_score; int32_t* r_cls; float* r_obj; float* r_cscore; int32_t* r_count;
    /* still-detector candidates, capacity per frame = max_keep */
    float* o_box; float* o_score; int32_t* o_cls; float* o_obj; float* o_cscore; int32_t* o_count;
} tscd_final_expand_args;
int tscd_final_expand(const tscd_final_expand_args* args, void* stream);

typedef struct {
    int32_t num_frames, cand_cap, keep_cap;
    const float* box; const float* obj; const float* cscore; const int32_t* cls;
    const int32_t* keep; const int32_t* keep_count;
    float* rows;                 /* [num_frames, keep_cap, 7] */
} tscd_final_rows_args;
int tscd_final_rows(const tscd_final_rows_args* args, void* stream);

/* ---- evaluator / Predictor glue (SURVEY.md section 8f-1) ---------------------------------------------------------------
 * Replaces the per-frame .cpu() + per-box Python loops of OVISEvaluator.convert_to_coco_format
 * (yolox/evaluators/ovis_evaluator_v2.py:233-289) and Predictor.to_repp_heavy (tools/val_to_imdb.py:193-218): all detections of
 * all frames as ONE packed table (one device->host copy), already divided by the per-frame resize scale and converted to
 * top-left + width / height:  packed row (12 floats) = [frame, x, y, w, h, obj * cls_score, class, obj, x2, y2, cls_score, 0];
 * offsets[f] .. offsets[f+1] are frame f's rows (in NMS keep order). */
typedef struct {
    int32_t num_frames, cap;     /* frames; row pitch of `rows` per frame */
    const float* rows;           /* [num_frames, cap, 7] stage output (x1,y1,x2,y2,obj,cls_score,cls) */
    const int32_t* count;        /* [num_frames] */
    const float* scale;          /* [num_frames] resize scale of every frame (boxes are DIVIDED by it), or NULL */
    int32_t* offsets;            /* out [num_frames + 1] */
    float* packed;               /* out [num_frames * cap, 12] */
} tscd_pack_detections_args;
int tscd_pack_detections(const tscd_pack_detections_args* args, void* stream);

/* Raw variant for the host-buffer entry (AggregationStage.forward_host): the stage's padded [num_frames, cap, 7] detection rows
 * compacted frame after frame into packed [sum n, 7] (+ offsets), so the host reads only the valid rows of ONE buffer and
 * splits it into the reference's list[Tensor[n,7]] (post_process.py:12-13,85) without a per-frame copy. */
typedef struct {
    int32_t num_frames, cap;
    const float* rows;           /* [num_frames, cap, 7] */
    const int32_t* count;        /* [num_frames] */
    int32_t* offsets;            /* out [num_frames + 1] */
    float* packed;               /* out [num_frames * cap, 7] */
} tscd_pack_rows_args;
int tscd_pack_rows(const tscd_pack_rows_args* args, void* stream);

/* ---- REPP detection linking (SURVEY.md section 8f-3) -------------------------------------------------------------------
 * Replaces REPP.get_video_pairs + solve_distances_def (tools/REPP.py:82-133) with the linking scores of distance_def /
 * distance_logreg (:52-79) and the pair features of tools/repp_utils.py:34-109: for every pair of consecutive frames the
 * n1 x n2 linking distances and the greedy minimum matching (global minimum first, ties in row-major order), as the list of
 * (index in frame f, index in frame f+1) pairs IN EXTRACTION ORDER (the tubelet builder, REPP.py:138-190, depends on it).
 * Detections of all frames are packed back to back; frame f owns [frame_off[f], frame_off[f+1]).  The one-hot class score
 * vectors of REPP.__call__ (:248-254) are passed as (score, class).  The logistic model is given by its coefficients in the
 * order (center_distances_corrected, height_rel, iou, width_rel) of tools/matching_model_logreg.pckl. */
typedef struct {
    int32_t num_frames;
    int32_t max_det;          /* pitch of `pairs` per frame pair; >= detections of any frame, <= 4096 */
    int32_t distance_func;    /* 0 = 'def', 1 = 'logreg' */
    int32_t clf_mode;         /* 0 = 'dot', 1 = 'max', 2 = 'dot_plus', 3 = 'raw' */
    double clf_thr;
    double coef[4];
    double intercept;
    const int32_t* frame_off; /* [num_frames + 1] */
    const float* bbox;        /* [N,4] x, y, width, height */
    const float* center;      /* [N,2] normalised box centre (val_to_imdb.py:211-212) */
    const double* score;      /* [N] obj * cls_score */
    const int32_t* cls;       /* [N] */
    int32_t* pairs;           /* out [num_frames - 1, max_det, 2] */
    int32_t* pair_count;      /* out [num_frames - 1] */
    double* ws_dist;          /* workspace [num_frames - 1, ws_pitch] candidate distances */
    int32_t* ws_idx;          /* workspace [num_frames - 1, ws_pitch] */
    int32_t ws_pitch;         /* >= number of finite distances of any frame pair (n1 * n2 always suffices) */
    int32_t* status;          /* optional [1]: TSCD_ERR_CAPACITY when a frame exceeds max_det or ws_pitch */
} tscd_repp_link_args;
int tscd_repp_link(const tscd_repp_link_args* args, void* stream);

/* ---- long-clip mode: exchange of the global-frame bank rows between ranks (SURVEY.md section 8e) ----------------------
 * One clip sharded by frame: every rank runs K1-K3 on its own frames [n_local_frames local | n_global_frames global], then the
 * ranks all-gather ONE packed buffer each (ncclAllGather, issued by the host) and every rank builds the virtual clip
 * [own local frames | all ranks' global frames, rank-major] whose local rows it attends from.  Replaces nothing in the
 * reference (single-GPU only); it is the exchange step BASELINE.json configs[3] names.
 *   tscd_bank_pack_bytes  size of one rank's buffer: 1 KB header (per-frame counts, up to 256 global frames per rank) + n_global_frames * kmax rows of
 *                         (cls 256 | reg 256 16-bit values | score fp32 + pad) = 1040 bytes;
 *   tscd_bank_pack        bank rows of the rank's global frames -> send buffer (frames padded to kmax rows: static layout);
 *   tscd_bank_unpack      gathered buffers [world, rank_bytes] + own bank -> per-frame counts, prefix offsets and the compacted
 *                         16-bit bank of the virtual clip (two kernels, no host sync). */
typedef struct {
    int32_t n_local_frames, n_global_frames, kmax;
    int32_t dtype;               /* TSCD_F16 / TSCD_BF16 bank element type */
    const int32_t* sel_count;    /* [n_local_frames + n_global_frames] */
    const int32_t* row_off;      /* [.. + 1] */
    const void* bank_cls;        /* [rows, 256] */
    const void* bank_reg;
    const float* bank_score;     /* [rows] */
    void* send;                  /* [tscd_bank_pack_bytes] */
} tscd_bank_pack_args;
int64_t tscd_bank_pack_bytes(int32_t n_global_frames, int32_t kmax);
int tscd_bank_pack(const tscd_bank_pack_args* args, void* stream);

typedef struct {
    int32_t world, n_local_frames, n_global_frames, kmax;
    int32_t dtype;
    int64_t rank_bytes;          /* pitch of one rank's buffer inside recv */
    const void* recv;            /* [world, rank_bytes] all-gathered buffers */
    const int32_t* sel_count;    /* own selection (local frames are read) */
    const int32_t* row_off;
    const void* bank_cls; const void* bank_reg; const void* bank_edge; const float* bank_score;
    int32_t* v_count;            /* out [n_local_frames + world * n_global_frames] */
    int32_t* v_row_off;          /* out [.. + 1] */
    void* v_bank_cls; void* v_bank_reg;   /* out [rows_cap, 256] */
    void* v_bank_edge;           /* out, local rows only (may be NULL) */
    float* v_bank_score;         /* out [rows_cap] */
} tscd_bank_unpack_args;
int tscd_bank_unpack(const tscd_bank_unpack_args* args, void* stream);

/* ---- frame store: K1-K3 once per video frame, clips assembled from it on the device ---------------------------------------
 * Replaces the per-clip repetition of K1-K3 over the frames of tools/tscd_demo.py:223-241 / vid.py:601-683 (each clip = lframe
 * consecutive local frames + gframe frames drawn from the rest of the video, so a frame appears in many clips).  A caller-owned
 * store (tscd_b200/frames.py FrameStore) keeps one frame's K1-K3 result per slot at a fixed pitch of kmax rows:
 *   tscd_frame_scatter   the packed tscd_gather output of N frames (+ tscd_edge_combine's bank_edge) -> slots frame_slots[0..N);
 *   tscd_clip_assemble   clip_slots [B*F] (clip-major; a slot may repeat, within a clip too) -> exactly the packed clip arrays
 *                        tscd_gather would have written for those frames: sel_count, row_off (exclusive prefix), bank rows,
 *                        sel_idx (optional) and the sel_rows of the first L frames of every clip.  Two kernels, no host sync.
 * A clip slot outside [0, frames) or never written (count -1) sets status to TSCD_ERR_FRAME_SLOT and contributes 0 rows; a slot
 * written by a call whose status was set passes that code on (K1 / K2 report capacity per call, not per frame).  A frame slot
 * outside [0, frames) in tscd_frame_scatter sets slot_error to TSCD_ERR_FRAME_SLOT and is skipped (status is only read, so
 * every written slot carries the same K1-K3 flag whatever the launch order of the blocks).
 * Banks: 256 16-bit channels per row (TSCD-L); all pointers 16-byte aligned. */
typedef struct {
    int32_t frames, kmax, num_classes;
    int32_t dtype;               /* TSCD_F16 / TSCD_BF16 bank element type */
    int32_t* count;              /* [frames] kept rows of the frame in the slot, -1 = never written */
    int32_t* status;             /* [frames] status of the call that wrote the slot (0 = ok) */
    void* bank_cls; void* bank_reg; void* bank_edge;   /* [frames * kmax, 256] */
    float* bank_score;           /* [frames * kmax] */
    int32_t* sel_idx;            /* [frames, kmax] anchor ids */
    float* sel_rows;             /* [frames, kmax, 7 + num_classes] reference rows */
} tscd_frame_store;

typedef struct {
    tscd_frame_store store;
    int32_t num_frames;          /* N */
    const int32_t* frame_slots;  /* [N] distinct slots */
    const int32_t* sel_count; const int32_t* row_off;   /* tscd_gather outputs over the N frames (max_keep == store.kmax) */
    const int32_t* sel_idx; const float* sel_rows;
    const void* bank_cls; const void* bank_reg; const void* bank_edge; const float* bank_score;
    const int32_t* status;       /* [1] the flag K1-K3 of these frames wrote (read only; copied into every slot written) */
    int32_t* slot_error;         /* [1] optional: set to TSCD_ERR_FRAME_SLOT when a frame slot is outside [0, frames) */
} tscd_frame_scatter_args;
int tscd_frame_scatter(const tscd_frame_scatter_args* args, void* stream);

typedef struct {
    tscd_frame_store store;
    int32_t B, F, L;
    int64_t row_cap;             /* rows of the output banks, >= B * F * kmax */
    const int32_t* clip_slots;   /* [B * F] */
    int32_t* sel_count;          /* out [B * F] */
    int32_t* row_off;            /* out [B * F + 1] */
    void* bank_cls; void* bank_reg; void* bank_edge;   /* out [row_cap, 256] */
    float* bank_score;           /* out [row_cap] */
    int32_t* sel_idx;            /* out [B * F, kmax] or NULL */
    float* sel_rows;             /* out [B * F, kmax, 7 + C]: rows of the local frames written */
    int32_t* status;             /* [1] */
} tscd_clip_assemble_args;
int tscd_clip_assemble(const tscd_clip_assemble_args* args, void* stream);

/* Debug aid: cycles block 0 of the last tscd_cafm_chain launches spent per phase
 * (0 assignment re-index, 1 query input, 2 q projection, 3 normalise, 4 attention, 5 norms/state, 6 state carry). */
int tscd_debug_chain_clocks(long long* host_out8, int reset);

/* Library / build information (also proves the .so was loaded). */
const char* tscd_version(void);
const char* tscd_last_cuda_error(void); /* text of the last CUDA runtime error seen by a TSCD_ERR_CUDA return */
int tscd_device_ok(void); /* 1 if the current device is compute capability 10.x */

#ifdef __cplusplus
}
#endif
#endif /* TSCD_B200_H_ */
