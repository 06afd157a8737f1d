/*
 * monoloco_b200 -- C ABI of the B200-native monoloco hot path (libmonoloco_b200.so).
 *
 * The reference (vita-epfl/monoloco @ f5e82c4) has no FFI on this path: its boundary is the Python API
 * monoloco/network/net.py:30-133 (Loco.__init__/forward), architectures.py:48-71,135-145 (nn.Module.forward)
 * and train/losses.py:59-73 (MultiTaskLoss.forward).  The entry points below are what a ctypes binding under
 * that Python API binds (INTEGRATION.md shows the stub); every function cites the reference code it replaces.
 *
 * Conventions: plain C, no exceptions, int return codes (0 = ok, <0 = error, text via mlb_last_error()),
 * caller-owned buffers, explicit cudaStream_t passed as void*.  All tensors are fp32 row-major.
 * Thread-safety: one handle may be used from one thread at a time; distinct handles are independent.
 */
#ifndef MONOLOCO_B200_H_
#define MONOLOCO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MLB_ABI_VERSION 2
#define MLB_MAX_OPS 32
#define MLB_MAX_PEERS 8
#define MLB_GATHER_LD 20   /* floats per gathered row: raw at [0,out), dec at [12,20) */
#define MLB_GATHER_DEC 12
#define MLB_GATHER_FLAG_STRIDE 32   /* uint32 between the per-rank completion flags (one 128-byte line each) */

/* ---- layer program: one entry per Linear(+BN+ReLU+Dropout)(+residual) of architectures.py ---- */
enum { MLB_OP_GEMM = 0, /* L-wide Linear, weights streamed through the TMA ring                    */
       MLB_OP_HEAD = 1  /* narrow head Linear (w_fin / w_aux / MonolocoModel.w2), N <= 16          */ };

enum { MLB_F_RELU     = 1,  /* nn.ReLU after the affine                                            */
       MLB_F_SAVE_RES = 2,  /* output is the `x` of the next MyLinearSimple (architectures.py:88)  */
       MLB_F_ADD_RES  = 4,  /* out = x + y                                   (architectures.py:100) */
       MLB_F_DROPOUT  = 8,  /* top-level self.dropout site (architectures.py:53,66; net.py:141)    */
       MLB_F_IN_XIN   = 16  /* reads the network input (first layer w1, architectures.py:50)       */ };

typedef struct mlb_op {
    int32_t type;      /* MLB_OP_*                                                                  */
    int32_t K;         /* in_features                                                               */
    int32_t Kpad;      /* K rounded up to the weight-chunk depth (zero padded)                      */
    int32_t N;         /* out_features                                                              */
    int32_t flags;     /* MLB_F_*                                                                   */
    int32_t out_col;   /* HEAD: first column of the raw [B,out] output it writes                    */
    int64_t w_off;     /* float offset into the packed blob: GEMM = chunked W^T, HEAD = W [N][K]    */
    int64_t scale_off; /* GEMM: per-feature scale [N]  (folded BatchNorm1d eval, eps 1e-5)          */
    int64_t shift_off; /* GEMM: per-feature shift [N]; HEAD: bias [N]                               */
} mlb_op;

enum { MLB_DECODE_NONE = 0,
       MLB_DECODE_LOCO = 1,  /* process.py:231-278 extract_outputs (monoloco_pp / monstereo)        */
       MLB_DECODE_MONO = 2,  /* process.py:330-360 extract_outputs_mono (legacy monoloco_p)         */
       MLB_DECODE_DB   = 3   /* net.py:95-100 legacy monoloco: d = o0, bi = exp(o1)*o0              */ };

typedef struct mlb_model_desc {
    int32_t abi_version;  /* MLB_ABI_VERSION                                                        */
    int32_t input_size;   /* 34 mono | 68 stereo                     (net.py:45-58)                 */
    int32_t output_size;  /* raw output columns: 2 | 9 | 10                                         */
    int32_t linear_size;  /* hidden width L (zero-padded by the packer): multiple of 128; <= 1024, or a     */
                          /* multiple of 256 <= 2048 (tensor-core kernel only)  (net.py:30, hyp_tuning.py:52) */
    int32_t n_ops;
    int32_t decode_kind;  /* MLB_DECODE_*                                                           */
    float   p_dropout;    /* nn.Dropout p (architectures.py:46)                                     */
    int32_t reserved;
} mlb_model_desc;

typedef struct mlb_model* mlb_handle;

/* Build a device-resident model from a host blob packed by monoloco_b200/packing.py (replaces
 * Loco.__init__'s load_state_dict + .to(device), net.py:68-81).  `device` is the CUDA ordinal. */
int mlb_create(const mlb_model_desc* desc, const mlb_op* ops, const float* packed_host, size_t n_floats,
               int device, mlb_handle* out);
/* Re-upload the packed blob (same layout) -- e.g. after an optimizer step. */
int mlb_update_weights(mlb_handle h, const float* packed_host, size_t n_floats, void* stream);
void mlb_destroy(mlb_handle h);
const char* mlb_last_error(void);
int mlb_abi_version(void);
/* number of SMs / resident CTAs the forward uses on this handle's device */
int mlb_num_sms(mlb_handle h);
/* which kernel the most recent mlb_forward on this handle launched (bench.py labels its roofline with it) */
enum { MLB_KERNEL_TILE = 0,    /* loco_forward_kernel: one CTA per row tile, FFMA2                              */
       MLB_KERNEL_CLUSTER = 1, /* loco_forward_cluster_kernel: 8-CTA cluster per 16 rows, FFMA2                 */
       MLB_KERNEL_WIDE = 2,    /* loco_forward_wide_kernel: the whole grid on <= 32 rows                        */
       MLB_KERNEL_TC = 3,      /* loco_forward_tc_kernel: tcgen05 kind::tf32, 3 MMAs per fp32 product           */
       MLB_KERNEL_WIDE2 = 4    /* loco_forward_wide2_kernel: 4-CTA clusters, K x N split, <= 16 rows            */ };
int mlb_last_kernel(mlb_handle h);
/* per-wave kernel times measured on this device when the handle was created (ms): [0] one wave of FFMA clusters, [1] + [2] * TM
 * one wave of FFMA row tiles, [3] one wave of tensor-core tiles -- mlb_forward picks the kernel family with them (no constants
 * from another box).  Returns 1 if measured, 0 if the defaults are in use (MLB_NO_CALIBRATE). */
int mlb_kernel_times(mlb_handle h, double out_ms[4]);
/* co-resident clusters of the tensor-core kernel on this device (= its persistent grid size), 0 if unavailable */
int mlb_tc_resident_clusters(mlb_handle h);
/* device error word of this handle (mapped host memory; read it after a stream synchronisation): 0 = none,
 * 1 = a TMA/mbarrier wait timed out, 3 = grid-barrier time-out (whole-grid kernel), 4 = fused all-gather: a peer
 * rank did not signal its epoch within 20 s. */
int mlb_device_error(mlb_handle h);

/* ---- inference ---- */
enum { MLB_IN_X = 0,          /* pre-processed network input [B, input_size] (nn.Module.forward)    */
       MLB_IN_KPS = 1,        /* raw keypoints [B,3,17] (u,v,conf rows): process.py:47-67 fused      */
       MLB_IN_KPS_STEREO = 2  /* left [L,3,17] + right [R,3,17], all-vs-all rows l*R+r: :25-44 fused */ };

/* At most one MLB_FWD_FORCE_* may be set, and it must name a kernel this handle has for this many rows (otherwise
 * mlb_forward fails).  A forced kernel ignores rows_per_group. */
enum { MLB_FWD_ZERO_CENTER = 1, /* preprocess_monoloco(zero_center=True) (net.py:96, legacy)        */
       MLB_FWD_DROPOUT     = 2, /* MC-dropout pass: top-level dropout sites active (net.py:141)     */
       MLB_FWD_RES_TMEM    = 4, /* stash the residual x of MyLinearSimple in Tensor Memory (default) */
       MLB_FWD_FORCE_TILE    = 8,  /* always use the throughput kernel (one CTA per row tile)        */
       MLB_FWD_FORCE_CLUSTER = 16, /* always use the small-batch kernel (8-CTA cluster per 16 rows)  */
       MLB_FWD_RES_SCRATCH   = 32, /* stash the residual in the L2-resident global scratch instead   */
       MLB_FWD_FORCE_WIDE    = 64, /* always use the whole-grid latency kernel (one launch / 32 rows)*/
       MLB_FWD_FORCE_TC      = 128, /* always use the tensor-core kernel (error-compensated TF32, 128-row tiles) */
       MLB_FWD_FORCE_WIDE2   = 256  /* always use the second-generation latency kernel (<= 16 rows)             */ };

typedef struct mlb_forward_args {
    int32_t input_kind;     /* MLB_IN_*                                                             */
    int32_t flags;          /* MLB_FWD_*                                                            */
    int32_t n_rows;         /* B; for MLB_IN_KPS_STEREO must equal n_left * n_right                 */
    int32_t n_left;         /* stereo only                                                          */
    int32_t n_right;        /* stereo only                                                          */
    int32_t rows_per_group; /* 0 = auto; else 8,10,..,16 (tile = 2*rows_per_group detections / CTA)  */
    float kinv[9];          /* K^-1 row-major (camera.py:25), only for MLB_IN_KPS*                  */
    float z_met;            /* camera.py:27 scale; 0 -> 10 (process.py:59-60)                       */
    const float* x;         /* input (see input_kind); left keypoints for stereo                    */
    const float* x_right;   /* right keypoints [R,3,17] (stereo)                                    */
    float* out_raw;         /* [B, output_size]            required                                 */
    float* out_dec;         /* [B, 8] = x,y,z,d,bi,yaw_pred,yaw_orig,sigmoid(aux)   or NULL         */
    float* out_xyzc;        /* [B, 4] = xyz_from_distance(d, K^-1[u_c,v_c,1]) (camera.py:161-177,
                               net.py:192-213) and its norm; MLB_IN_KPS* (left pose), or NULL       */
    float* out_x;           /* [B, input_size] the pre-processed network input, or NULL             */
    const uint8_t* drop_mask; /* [sites][B][L] keep-mask (1 keep) for MLB_FWD_DROPOUT, or NULL      */
    uint64_t drop_seed;     /* in-kernel counter RNG seed when drop_mask == NULL                    */
    /* fused all-gather (multi-GPU, one process per GPU): the decode epilogue additionally stores every row as
     * [raw(out) | pad | dec(8)] (MLB_GATHER_LD floats, dec at MLB_GATHER_DEC) into n_gather buffers -- this
     * rank's and its NVLink peers' (pointers from mlb_ipc_open) -- at row gather_row0 + i.                  */
    float* gather[MLB_MAX_PEERS];
    int32_t n_gather;       /* 0 = off                                                              */
    int32_t gather_rank;    /* index of this rank's own buffer in gather[] / gather_flags[]         */
    int64_t gather_row0;    /* first global row of this rank's shard                                */
    /* device-side completion of the fused all-gather (no collective library in the data plane): when gather_epoch != 0
     * the last CTA of the launch to finish its peer stores writes gather_epoch (st.release.sys) into slot gather_rank of
     * EVERY rank's flag array, then spins (ld.acquire.sys) on this rank's own array until all n_gather slots have reached
     * gather_epoch -- the kernel retires only when every shard has landed in this rank's buffer.  gather_flags[r] = rank
     * r's flag array (MLB_GATHER_FLAG_STRIDE uint32 between slots, zero-initialised, in peer-mapped memory); epochs must
     * increase by one per step on every rank.  gather_epoch == 0: no protocol, the caller synchronises the ranks.     */
    uint32_t* gather_flags[MLB_MAX_PEERS];
    uint32_t gather_epoch;
    int32_t reserved0;
} mlb_forward_args;

/* Fused pre-process -> MLP -> heads -> decode on DEVICE buffers (replaces net.py:92-124 body:
 * preprocess_*, self.model(inputs), extract_outputs). Asynchronous on `stream`. */
int mlb_forward(mlb_handle h, const mlb_forward_args* args, void* stream);
/* Same with HOST buffers: H2D of the inputs, kernel, D2H of every non-NULL output, then stream sync
 * (replaces net.py:92-93 `.to(device)` + process.py:261-263 `.detach().cpu()`). */
int mlb_forward_host(mlb_handle h, const mlb_forward_args* host_args, void* stream);

/* pre-process only: [B,3,17] -> [B,34] (process.py:47-67), for callers such as
 * prep/preprocess_kitti.py:193 that never run the network.  Device buffers. */
int mlb_preprocess(const float* kps, int n_rows, const float kinv[9], float z_met, int zero_center,
                   float* out_x, void* stream);

/* monstereo arg-max filter (process.py:307-327): rows [n_left*n_right, out] viewed [n_left, n_right, out];
 * keeps, per left pose, every row whose last column >= the max over its right poses (ties kept, row-major
 * order).  Gathers raw (and dec / xyzc if non-NULL) rows into sel_*; writes the kept-row count to *n_sel_dev
 * and the kept flat row indices to sel_idx (capacity n_left*n_right).  One warp per left pose, two launches (count,
 * ordered scatter), no host synchronisation; cnt_scratch [n_left] int32 and best_scratch [n_left] fp32 are caller-owned
 * device scratch.  Device buffers. */
int mlb_stereo_filter(const float* raw, const float* dec, const float* xyzc, int n_left, int n_right, int out_size,
                      float* sel_raw, float* sel_dec, float* sel_xyzc, int32_t* sel_idx, int32_t* n_sel_dev,
                      int32_t* cnt_scratch, float* best_scratch, void* stream);

/* ---- Loco.post_process for a BATCH of images on the device (net.py:164-248; utils/iou.py:6-29,44-64,87-101;
 * utils/camera.py:10-29,82-96,161-177).  Detections / ground truths of all images are concatenated; det_off / gt_off are
 * CSR offsets.  One CTA per image: bbox-centre / shoulder / head pixels (rounded half-even like Python round()), bbox-
 * centre ray K^-1[u_c,v_c,1], xyz_from_distance(d, ray), conf = 0.035 * box_conf / (bi / |xyz|) in fp64, greedy IoU
 * matching in decreasing box confidence (fp64, first maximum, each ground truth used once), the output order (matches
 * first -- left to right by box x1 when `reorder` -- then the rest by index) and xyz_real of the matches.
 * All pointers are device pointers. */
typedef struct mlb_post_args {
    int32_t n_img;
    int32_t max_det;           /* largest number of detections in one image (shared-memory sizing)              */
    int32_t max_gt;            /* largest number of ground-truth boxes in one image                              */
    int32_t reorder;           /* net.py:185-186                                                                 */
    double iou_min;            /* net.py:164 default 0.3                                                         */
    const int32_t* det_off;    /* [n_img + 1]                                                                    */
    const int32_t* gt_off;     /* [n_img + 1] or NULL (no ground truth)                                          */
    const double* boxes;       /* [n_det][5] x1, y1, x2, y2, confidence (Python floats = fp64)                   */
    const float* kps;          /* [n_det][3][17]                                                                 */
    const float* kinv;         /* [n_img][9] K^-1 row-major, fp32                                                */
    const float* dec;          /* [n_det][8] decoded network outputs (mlb_forward out_dec): d at 3, bi at 4      */
    const double* gt_boxes;    /* [n_gt][4]                                                                      */
    const double* gt_d;        /* [n_gt] ground-truth distances (dic_gt['ys'][j][3])                             */
    float* xyz;                /* out [n_det][3] xyz_pred                                                        */
    float* ray;                /* out [n_det][4] bbox-centre ray (x, y, z) and sqrt(1 + x^2 + y^2)               */
    double* conf;              /* out [n_det]                                                                    */
    int32_t* uv;               /* out [n_det][6] rounded centre, shoulder, head pixels                           */
    int32_t* match_gt;         /* out [n_det] image-local index of the matched ground truth, or -1              */
    int32_t* order;            /* out [n_det] per image: image-local detection index at every output position   */
    int32_t* n_match;          /* out [n_img]                                                                    */
    float* xyz_real;           /* out [n_det][3] xyz_from_distance(gt distance, ray) of matched detections       */
} mlb_post_args;
int mlb_post_process(const mlb_post_args* args, void* stream);

/* KITTI label rows (eval/generate_kitti.py:202-253, nets monoloco_pp / monstereo): rows [n][15] fp64 =
 * [alpha, x1, y1, x2, y2, h, w, l, x, y, z, ry, conf, bi, epi] with conf = conf_scale * box_conf / (bi / |xyz|)
 * (conf_scale 0.035 monoloco_pp, 0.033 monstereo); the host only formats "%f".  boxes [n][5] fp64, raw [n][out_size],
 * dec [n][8], epi [n] or NULL.  Device buffers. */
int mlb_kitti_rows(int n, int out_size, double conf_scale, const double* boxes, const float* raw, const float* dec,
                   const float* epi, double* rows, void* stream);

/* decode only (process.py:231-278 / 330-360 on a raw tensor that did not come from mlb_forward):
 * raw [B, out_size] -> dec [B, 8] as in mlb_forward_args.out_dec.  Device buffers. */
int mlb_decode(const float* raw, int n_rows, int out_size, int decode_kind, float* dec, void* stream);

/* MC-dropout epistemic spread (net.py:135-161, process.py:101-122): d_bi [n_pass, n_rows, 2] = (d, bi) of
 * n_pass stochastic forwards (MLB_FWD_DROPOUT); for every row draws n_samples Laplace(d, |bi|) samples per pass
 * (counter RNG, `seed`) and writes the unbiased std over all n_pass*n_samples draws to out_std [n_rows]. */
int mlb_laplace_std(const float* d_bi, int n_pass, int n_rows, int n_samples, uint64_t seed, float* out_std,
                    void* stream);

/* ---- training step (trainer.py:153-161: model(inputs) in train mode, mt_loss, loss.backward()) -------------
 * One persistent cooperative kernel per direction: forward (train-mode BatchNorm1d = batch statistics with a
 * grid-wide reduction per layer, Dropout with a counter RNG or explicit masks, running-stat update) and backward
 * (dL/dout -> every parameter gradient); mlb_train_step fuses forward + MultiTaskLoss + backward in ONE launch.
 * All pointers are device pointers to fp32 tensors in the reference's native layouts (nn.Linear.weight [out,in]).
 * LocoModel topology only (architectures.py:48-71), which is what Trainer builds (trainer.py:115-122). */
#define MLB_MAX_BLOCKS 16
enum { MLB_TASK_D = 0, MLB_TASK_X = 1, MLB_TASK_Y = 2, MLB_TASK_H = 3, MLB_TASK_W = 4, MLB_TASK_L = 5,
       MLB_TASK_ORI = 6, MLB_TASK_AUX = 7 };  /* trainer.py:40, losses.py:76-101 */

typedef struct mlb_train_block {   /* one L-wide Linear (+BatchNorm1d+ReLU+Dropout) in forward order           */
    int32_t K;                     /* in_features                                                              */
    int32_t has_bn;                /* 0 only for LocoModel.w2 (architectures.py:59)                            */
    int32_t res_src;               /* index of the block whose output is added to this one's (x + y), or -1   */
    int32_t reserved;
    const float* W;                /* [L, K]                                                                   */
    const float* b;                /* [L]                                                                      */
    const float* gamma;            /* BatchNorm1d.weight [L]                                                   */
    const float* beta;             /* BatchNorm1d.bias   [L]                                                   */
    float* running_mean;           /* updated in place with momentum (may be NULL)                             */
    float* running_var;
    float* dW;                     /* gradient outputs, overwritten: [L, K], [L], [L], [L]                     */
    float* db;
    float* dgamma;
    float* dbeta;
} mlb_train_block;

typedef struct mlb_train_args {
    int32_t n_rows, input_size, output_size, linear_size, n_blocks;
    int32_t aux_block;             /* block whose output feeds w_aux (LocoModel.w2); w_fin reads the last block */
    int32_t update_running_stats;  /* 1 in training (nn.BatchNorm1d momentum update, unbiased variance)         */
    int32_t rows_per_group;        /* 0 = auto                                                                  */
    float p_dropout, bn_eps, bn_momentum;
    int32_t flags;                 /* reserved, must be 0                                                       */
    uint64_t drop_seed;            /* counter-RNG seed (must be the same in forward and backward)               */
    const uint8_t* drop_mask;      /* optional explicit keep masks [n_bn_blocks][B][L] (parity tests)           */
    const float* x;                /* [B, input_size] pre-processed inputs                                      */
    float* out;                    /* [B, output_size]                                                          */
    const float* g_out;            /* backward only: dL/d(out) [B, output_size]                                 */
    const float* W_aux; const float* b_aux; const float* W_fin; const float* b_fin;   /* [1,L],[1],[out-1,L],[out-1] */
    float* dW_aux; float* db_aux; float* dW_fin; float* db_fin;
    /* fused MultiTaskLoss / AutoTuneMultiTaskLoss (losses.py:28-73), mlb_train_step only */
    const float* labels;           /* [B, label_ld]  Y = [theta, psi, z, r, h, w, l, sin, cos, yaw(, s_match)]   */
    int32_t label_ld, n_tasks;
    int32_t tasks[8];              /* MLB_TASK_*                                                                */
    float task_scale[8];           /* lambda_t (MultiTaskLoss) or lambda_t / (2 exp(log_sigma_t)^2) (AutoTune)  */
    float* loss_vals;              /* [8] unweighted per-task means (device)                                    */
    const float* task_scale_dev;   /* optional device copy of task_scale[] (overrides it): lets AutoTune's       */
                                   /* lambda_t / (2 exp(log_sigma_t)^2) stay on the device, no host sync         */
} mlb_train_args;

typedef struct mlb_train* mlb_train_handle;
/* workspace for up to max_rows detections: saved activations, pre-BN outputs, gradients, transposed weights. */
int mlb_train_create(int device, int max_rows, int input_size, int linear_size, int n_blocks, mlb_train_handle* out);
void mlb_train_destroy(mlb_train_handle h);
int mlb_train_forward(mlb_train_handle h, const mlb_train_args* a, const mlb_train_block* blocks, void* stream);
int mlb_train_backward(mlb_train_handle h, const mlb_train_args* a, const mlb_train_block* blocks, void* stream);
int mlb_train_step(mlb_train_handle h, const mlb_train_args* a, const mlb_train_block* blocks, void* stream);
/* profiling aid: wall time (ns) of every phase of the most recent launch (synchronises the device);
 * returns the number of phases written. types: 0 PACK, 1 FWD, 2 FWD_FINAL, 3 BWD_INIT, 4 BWD_HEAD, 5 BWD, 6 DW. */
int mlb_train_phase_times(mlb_train_handle h, int max_n, double* out_ns, int* types, int* blks);
/* profiling aid: out_ns[(ph*3 + s)*8 + k] = ns since the start of phase ph at which CTA s (0 first, 1 middle, 2 last
 * active) passed point k (0 input tile ready, 1 GEMM done, 2 epilogue done, 3 left the grid barrier,
 * 4 batch statistics loaded, 5 tile rows finished, 6-7 spare); 0 where unset. */
int mlb_train_subphase_times(mlb_train_handle h, int max_n, double* out_ns);

/* ---- optimizer side of the train step (trainer.py:159-160): clip_grad_norm_(params, max_norm) + Adam.step() over a
 * list of fp32 tensors (device pointers, host arrays of pointers / sizes), two multi-tensor launches, no host sync.
 * clip_mask[i] != 0: tensor i takes part in the gradient norm and is scaled by the clip coefficient (the reference clips
 * model.parameters() only; AutoTune's log_sigmas are optimised but not clipped).  max_norm <= 0 disables clipping.
 * `step` is Adam's 1-based step count; sqnorm_scratch_dev is one device double. */
int mlb_adam_clip_step(int n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                       float* const* exp_avg_sq, const int64_t* sizes, const int32_t* clip_mask, float max_norm, float lr,
                       float beta1, float beta2, float eps, float weight_decay, int64_t step, double* sqnorm_scratch_dev,
                       void* stream);

/* ---- NVLink peer buffers for the fused all-gather (cudaIpc*, one process per GPU) ---- */
#define MLB_IPC_HANDLE_BYTES 64
/* cudaMalloc `bytes` on `device` (zero-filled) and export an IPC handle for the other ranks. */
int mlb_ipc_alloc(int device, size_t bytes, void** dev_ptr, unsigned char handle[MLB_IPC_HANDLE_BYTES]);
/* map a peer rank's buffer into this process (cudaIpcOpenMemHandle, peer access over NVLink). */
int mlb_ipc_open(int device, const unsigned char handle[MLB_IPC_HANDLE_BYTES], void** dev_ptr);
int mlb_ipc_close(void* dev_ptr);
int mlb_ipc_free(void* dev_ptr);

/* FP32-FFMA throughput probe (roofline denominator for the fp32-bound regime): every thread of
 * `blocks` x 512 threads runs |iters| x 128 FMAs in 16 independent chains (iters < 0: packed fma.rn.f32x2).
 * Returns flops launched via *flops. */
int mlb_probe_ffma(int device, int blocks, int iters, double* flops, void* stream);

/* number of kernels this library has launched in this process (bench.py "gpu_launches") */
uint64_t mlb_launch_count(void);
/* profiling aid: point the tile kernel's timestamp marks at a device buffer of >= 4*n_ops + 4 uint64 (NULL: off, the
 * default).  CTA 0 stamps %globaltimer at: [0] start, [1] input tile staged, per op i [2+4i] GEMM done, [3+4i] epilogue
 * math done, [4+4i] CTA synchronised, [5+4i] activation tile rewritten; [2+4n] heads done, [3+4n] rows stored. */
int mlb_debug_fwd_marks(void* dev_buf);

/* tensor-core feasibility probe (tools/probe_tc.py; not on the product path): D[128,128] = A[128,K] . W[128,K]^T on
 * tcgen05.mma kind::tf32 with every fp32 operand split into two TF32 terms.  mode 0: a_hi.w_hi only; 1: the three products
 * into one TMEM accumulator; 2: the cross terms a_lo.w_hi + a_hi.w_lo into a second accumulator (out_cross).  K % 32 == 0. */
int mlb_probe_tf32x3(const float* A_dev, const float* W_dev, int K, int mode, float* out_main_dev, float* out_cross_dev,
                     void* stream);
/* the same error-compensated product for one whole layer, Y[B,N] = X[B,K] . W[N,K]^T (timing probe, not on the product
 * path).  stages (bit mask): 1 = split X into TF32 hi/lo planes (x_planes_dev, 2*B*K floats), 2 = split W (w_planes_dev,
 * 2*N*K floats), 4 = the tcgen05 GEMM from the planes (4-stage TMA ring, two TMEM accumulators).  B % 128 == 0,
 * N % 256 == 0, K % 16 == 0. */
int mlb_probe_tc_layer(const float* X_dev, const float* W_dev, float* Y_dev, int B, int N, int K, float* x_planes_dev,
                       float* w_planes_dev, int stages, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MONOLOCO_B200_H_ */
