/*
 * avc_b200.h -- C-ABI of libavc_b200.so: the B200 (sm_100a) implementation of attack-vc's
 * adversarial perturbation loop.
 *
 * The reference (bbbbhrrrr/attack-vc) has no native layer: its hot path is Python calling
 * PyTorch (attack_utils.py:7-130 driving models.py:121-485).  Each entry point below therefore
 * cites the reference *Python* interface it replaces; INTEGRATION.md shows the ctypes binding a
 * maintainer adds on the reference side (this repository ships that binding as
 * attack_vc_b200/_lib.py + attack_utils.py).
 *
 * Conventions
 *   - every function returns AVC_OK (0) or a negative avc_status; avc_last_error() gives text.
 *   - all data pointers are DEVICE pointers to fp32 unless a name ends in _host.
 *   - utterance tensors use the reference's logical layout [B, 80, T] with explicit element
 *     strides (sb, sc, st), so the CLI's transposed views (attack.py:49-50) need no copy.
 *   - `stream` is a cudaStream_t passed as void*.  Calls that own temporary device memory (the
 *     one-shot attacks, avc_attack_end, the forward-only and unit-test entry points) synchronise
 *     the stream before returning; avc_attack_step only enqueues.  The library never frees caller memory and keeps no global mutable state: all
 *     state lives in the handle, one handle per (process, device).
 *   - there is no CPU fallback: without a CUDA device avc_create fails with AVC_ERR_CUDA.
 */
#ifndef AVC_B200_H_
#define AVC_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct avc_handle avc_handle;
typedef struct avc_session avc_session;   /* one attack in flight: optimiser state + captured iteration */

typedef enum avc_status {
  AVC_OK = 0,
  AVC_ERR_INVALID = -1,     /* bad argument / unsupported hyper-parameter        */
  AVC_ERR_CUDA = -2,        /* CUDA runtime error (text in avc_last_error)       */
  AVC_ERR_WEIGHTS = -3,     /* weights missing or wrong shape                    */
  AVC_ERR_STATE = -4        /* call order violated (e.g. attack before weights)  */
} avc_status;

#define AVC_MAX_BLOCKS 8
#define AVC_MAX_BANK 8

/* Hyper-parameters of one encoder (constructor args of ContentEncoder models.py:126-139 and
 * SpeakerEncoder models.py:218-232).  dropout_rate must be 0 and bank_scale 1 (SURVEY §2.2). */
typedef struct avc_encoder_desc {
  int32_t c_in, c_h, c_out, kernel_size, bank_size, c_bank;
  int32_t n_conv_blocks, n_dense_blocks;          /* n_dense_blocks = 0 for the content encoder */
  int32_t subsample[AVC_MAX_BLOCKS];
  float neg_slope;                                /* 0 = ReLU, 0.01 = "lrelu" (models.py:107-118) */
} avc_encoder_desc;

/* Decoder constructor args, models.py:351-363.  sn must be false, dropout_rate 0. */
typedef struct avc_decoder_desc {
  int32_t c_in, c_cond, c_h, c_out, kernel_size, n_conv_blocks;
  int32_t upsample[AVC_MAX_BLOCKS];
  float neg_slope;
} avc_decoder_desc;

typedef struct avc_model_desc {
  avc_encoder_desc speaker, content;
  avc_decoder_desc decoder;
} avc_model_desc;

/* One tensor of model.state_dict() (models.py:438-452): key, device pointer, PyTorch shape. */
typedef struct avc_weight_view {
  const char* name;        /* e.g. "speaker_encoder.conv_bank.3.weight" */
  const float* data;       /* contiguous fp32, device memory            */
  int32_t ndim;
  int64_t shape[4];
} avc_weight_view;

/* Arguments shared by the three attacks (attack_utils.py:7-14, 51-53, 89-96). */
typedef struct avc_attack_args {
  const float* vc_tgt;  int64_t tgt_stride[3];  int32_t B, T_tgt;   /* utterance to defend   */
  const float* adv_tgt; int64_t adv_stride[3];  int32_t T_adv;      /* adversarial target    */
  const float* vc_src;  int64_t src_stride[3];  int32_t T_src;      /* NULL for emb_attack   */
  const float* w0;      int64_t w0_stride[3];   /* initial w ~ N(0,1) (attack_utils.py:30,68,112) */
  float* adv_out;       int64_t out_stride[3];  /* vc_tgt + eps*tanh(w_final), [B,80,T_tgt]       */
  float* loss_out;      /* [n_iters] device, per-iteration loss; may be NULL                     */
  float* grad_out;      /* [B,80,T_tgt] contiguous, dL/dw of the LAST iteration; may be NULL     */
  float eps;            /* attack.py:95-100                                                      */
  int32_t n_iters;      /* attack.py:101-106                                                     */
  double inv_norm;      /* MSELoss normaliser 1/(B_global*D); <=0 means 1/(B*D) of this call.     *
                         * Sharded callers pass the GLOBAL value (SURVEY §5 sharding hazard).      */
  int32_t use_graph;    /* 1: capture one iteration into a CUDA graph and replay it               */
} avc_attack_args;

/* ---- lifetime -------------------------------------------------------------------------- */
/* replaces: AdaInVC(config["model"]).to(device)  (data_utils.py:220, models.py:438-452) */
int avc_create(avc_handle** out, const avc_model_desc* desc, int device);
void avc_destroy(avc_handle* h);
const char* avc_last_error(const avc_handle* h);   /* h may be NULL: last create() error */
/* replaces: model.load_state_dict(...) (data_utils.py:221).  Synchronous; copies + repacks. */
int avc_load_weights(avc_handle* h, const avc_weight_view* tensors, int32_t n);

/* ---- the hot path ---------------------------------------------------------------------- */
/* replaces: attack_utils.emb_attack (attack_utils.py:51-86) */
int avc_emb_attack(avc_handle* h, const avc_attack_args* a, void* stream);
/* replaces: attack_utils.e2e_attack (attack_utils.py:7-48) */
int avc_e2e_attack(avc_handle* h, const avc_attack_args* a, void* stream);
/* replaces: attack_utils.fb_attack (attack_utils.py:89-130) */
int avc_fb_attack(avc_handle* h, const avc_attack_args* a, void* stream);

/* ---- attacks over utterances of DIFFERENT lengths in one call ------------------------------
 * The same three attacks (kind 0 emb, 1 e2e, 2 fb) on B utterances of frames_host[b] frames each.  The perturbed
 * utterances only pass through the speaker encoder, which runs them as one padded batch on the tensor-core kernels
 * with per-utterance lengths; the adversarial target and the conversion source keep one length for the batch.
 * vc_tgt, w0, adv_out and grad_out are PACKED: utterance b's frames are rows [sum_{i<b} T_i, sum_{i<=b} T_i) of one
 * contiguous time-major [sum_b T_b, 80] tensor.  loss_out (summed over the batch), eps, n_iters, inv_norm and use_graph
 * mean what they mean in avc_attack_args.  Every length must pass the speaker encoder's reflect-padding rule; the
 * error names the first utterance that does not.  AVC_CONV_IMPL=1 or 3 (CUDA cores) is rejected. */
typedef struct avc_attack_varlen_args {
  const float* vc_tgt;        /* [sum T_b, 80] packed utterances to defend                        */
  const float* w0;            /* [sum T_b, 80] packed initial w                                   */
  float* adv_out;             /* [sum T_b, 80] packed result                                      */
  float* grad_out;            /* [sum T_b, 80] packed dL/dw of the last iteration; may be NULL    */
  const int32_t* frames_host; /* [B] host: frames of every utterance                              */
  int32_t B;
  const float* adv_tgt; int64_t adv_stride[3]; int32_t T_adv;   /* [B,80,T_adv], batch stride 0 allowed */
  const float* vc_src;  int64_t src_stride[3]; int32_t T_src;   /* NULL for emb                         */
  float* loss_out;            /* [n_iters] device or NULL                                         */
  float eps;
  int32_t n_iters;
  double inv_norm;
  int32_t use_graph;
} avc_attack_varlen_args;
int avc_attack_varlen(avc_handle* h, int32_t kind, const avc_attack_varlen_args* a, void* stream);

/* ---- the same attacks as a session, so a caller can interleave iterations with a progress bar
 * (the reference shows tqdm.trange, attack_utils.py:33,71,115) or time iterations precisely.
 * begin: validates, computes targets + loop invariants, captures one iteration (kind 0 emb, 1 e2e,
 * 2 fb; a->n_iters is the MAXIMUM number of iterations).  step: enqueue n more iterations.
 * end: write adv_out / loss_out / grad_out, synchronise, free the session (always frees). */
int avc_attack_begin(avc_handle* h, int32_t kind, const avc_attack_args* a, void* stream, avc_session** out);
int avc_attack_step(avc_session* s, int32_t n, void* stream);
int avc_attack_end(avc_session* s, void* stream);
/* kernels launched by one iteration of this session */
int32_t avc_session_launches(const avc_session* s);
/* measurement aid for bench.py: run ONE iteration eagerly with CUDA events around every launch.
 * Arrays hold avc_session_launches() entries: kind (0 conv,1 norm,2 dense tail,3 affine,4 loss,
 * 5 update,6 layout,7 copy), milliseconds, algorithmic FLOPs and algorithmic HBM bytes. */
int avc_session_profile(avc_session* s, int32_t cap, int32_t* kind, float* ms, double* flops, double* bytes, void* stream);

/* ---- universal perturbation header (SURVEY 8f rank 2) -------------------------------------------------
 * replaces: UniversalPerturbationHeader.optimize(source_mel, target_mel, speaker_encoder, Adam([header], lr), ...)
 * (models/header_model.py:25-68) with speaker_encoder = this handle's AdaIN-VC SpeakerEncoder applied to
 * mel.squeeze(1).  ONE perturbation [80,T] is shared by the batch: perturbed = clamp(source + header, -1, 1),
 * loss = mse(e, e_target) - lambda * mse(e, e_source), Adam step, header = clamp(header, -eps, eps). */
typedef struct avc_header_args {
  const float* source; int64_t src_stride[3]; int32_t B, T;     /* [B,80,T] (the reference's [B,1,80,T] squeezed) */
  const float* target; int64_t tgt_stride[3]; int32_t T_tgt;
  const float* header0; int64_t hdr_stride[2];                   /* [80,T] initial header (zeros, header_model.py:22) */
  float* header_out;    int64_t out_stride[2];                   /* [80,T] */
  float* loss_out;                                               /* [n_iters] or NULL */
  float* grad_out;                                               /* [80,T] contiguous, d loss / d header of the last iteration, or NULL */
  float eps, lambda, lr;                                         /* train_header.py:120-125: 0.1, 0.5, 1e-3 */
  int32_t n_iters;
  double inv_norm;                                               /* 1/(B_global*128); <= 0: this call's batch */
  int32_t use_graph;
} avc_header_args;
int avc_header_optimize(avc_handle* h, const avc_header_args* a, void* stream);
/* session form (ended with avc_attack_end).  phase 0: n whole iterations.  Sharded batches run phase 1 (forward,
 * backward, this rank's partial header gradient), all-reduce avc_header_grad_buffer() over the ranks, then phase 2
 * (Adam + projection + next perturbed batch) -- the one per-iteration collective of this workload. */
int avc_header_begin(avc_handle* h, const avc_header_args* a, void* stream, avc_session** out);
int avc_header_step(avc_session* s, int32_t n, int32_t phase, void* stream);
float* avc_header_grad_buffer(avc_session* s, int64_t* n_floats);

/* ---- speaker-embedding loss and its gradient w.r.t. a perturbed batch (SURVEY 8f rank 3) ---------------------
 * replaces: train_predictive.py:113-123 with speaker_encoder = this handle's AdaIN-VC SpeakerEncoder on mel.squeeze(1):
 *   e_s = speaker_encoder(source); e_t = speaker_encoder(target); e_p = speaker_encoder(perturbed)
 *   loss = mse(e_p, e_t) - lambda * mse(e_p, e_s); loss.backward()   -> d loss / d perturbed
 * A session binds the four device buffers once; every avc_spk_grad_step re-reads their CURRENT contents (one captured
 * graph: three encoder forwards, the loss, one backward), so a training loop refills them each step.  Ended with
 * avc_attack_end.  The encoder's own parameter gradients (an unread side effect in the reference: the optimiser only
 * owns the predictive model) are not computed. */
typedef struct avc_spk_grad_args {
  const float* perturbed; int64_t p_stride[3];  int32_t B, T;     /* [B,80,T]                                     */
  const float* source;    int64_t s_stride[3];                    /* [B,80,T]                                     */
  const float* target;    int64_t t_stride[3];  int32_t T_tgt;    /* [B,80,T_tgt]                                 */
  float* grad_out;        int64_t g_stride[3];                    /* [B,80,T]: d loss / d perturbed               */
  float* loss_out;                                                /* one float (device), may be NULL              */
  float lambda;                                                   /* train_predictive.py:181 default 0.5          */
  double inv_norm;                                                /* 1/(B_global*128); <= 0: this call's batch    */
  int32_t use_graph;
} avc_spk_grad_args;
int avc_spk_grad_begin(avc_handle* h, const avc_spk_grad_args* a, void* stream, avc_session** out);
int avc_spk_grad_step(avc_session* s, void* stream);              /* enqueues only */

/* ---- forward-only model entry points (SURVEY §8f row 1; also used by the parity tests) --- */
/* replaces: model.speaker_encoder(x) (models.py:327-343).  x [B,80,T] strided -> emb [B,c_out] */
int avc_speaker_encoder(avc_handle* h, const float* x, const int64_t stride[3], int32_t B, int32_t T,
                        float* emb, void* stream);
/* replaces: model.inference(src, tgt) (models.py:472-485) -> out [B,80,T_out] contiguous,
 * T_out = avc_decoder_frames(h, T_src). */
int avc_inference(avc_handle* h, const float* src, const int64_t src_stride[3], int32_t T_src,
                  const float* tgt, const int64_t tgt_stride[3], int32_t T_tgt, int32_t B,
                  float* out, void* stream);
int32_t avc_decoder_frames(const avc_handle* h, int32_t T_src);

/* ---- per-kernel entry points for unit tests (time-major [B,T,C] contiguous tensors) ------- */
/* replaces: pad_layer(x, nn.Conv1d(k, stride)) (models.py:10-30): reflect pad + conv + bias.
 * w is PyTorch layout [c_out, c_in, k].  y [B, ceil(T/stride), c_out]. */
int avc_conv1d_fwd(avc_handle* h, const float* x, const float* w, const float* bias, float* y,
                   int32_t B, int32_t T, int32_t c_in, int32_t c_out, int32_t k, int32_t stride,
                   int32_t impl /*0 auto, 1 fp32 CUDA cores, 2 tcgen05 (TF32 + BF16 correction MMA; kernel picked by size), 3 fp32 CUDA cores without the small-M kernel,
                                   6 tcgen05 role-swapped N=256 kernel, 7 tcgen05 N=128 kernel*/, void* stream);
/* autograd of the above w.r.t. x: dy [B,T_out,c_out] -> dx [B,T,c_in] */
int avc_conv1d_dgrad(avc_handle* h, const float* dy, const float* w, float* dx,
                     int32_t B, int32_t T, int32_t c_in, int32_t c_out, int32_t k, int32_t stride,
                     int32_t impl, void* stream);
/* autograd of the above w.r.t. the parameters: x [B,T,c_in], dy [B,T_out,c_out] -> dw [c_out,c_in,k] (PyTorch
 * layout), dbias [c_out] or NULL.  Replaces the param.grad side effect of loss.backward() (attack_utils.py:45,83,127),
 * which the attack itself never reads (SURVEY.md §8 "wgrad note"): opt-in, not part of an attack iteration. */
int avc_conv1d_wgrad(avc_handle* h, const float* x, const float* dy, float* dw, float* dbias,
                     int32_t B, int32_t T, int32_t c_in, int32_t c_out, int32_t k, int32_t stride, void* stream);
/* the same with the kernel chosen explicitly: impl 0 auto (tensor cores from 2048 GEMM rows), 1 exact fp32 on the CUDA
 * cores, 2 tcgen05: TMA-fed MN-major operands, 3xTF32 (hi/lo planes), fp32 accumulation in TMEM; stated tolerance 2e-5
 * relative per tensor against fp64 */
int avc_conv1d_wgrad_ex(avc_handle* h, const float* x, const float* dy, float* dw, float* dbias,
                        int32_t B, int32_t T, int32_t c_in, int32_t c_out, int32_t k, int32_t stride, int32_t impl, void* stream);
/* replaces: act(append_cond(InstanceNorm1d(y), cond)) [+ residual] (models.py:414-431).
 * cond [B,2C] (mean | std) or NULL; res [B,T/up,C] or NULL; stats_out [B,C,2] (mean, rstd). */
int avc_instnorm_adain_act_fwd(avc_handle* h, const float* y, const float* cond, const float* res,
                               int32_t up, float* out, float* stats_out, int32_t B, int32_t T,
                               int32_t C, float neg_slope, void* stream);
/* its backward: g [B,T,C] -> gy [B,T,C] (may be NULL), gcond [B,2C] (d mean | d std) */
int avc_instnorm_adain_act_bwd(avc_handle* h, const float* g, const float* y, const float* stats,
                               const float* cond, float* gy, float* gcond, int32_t B, int32_t T,
                               int32_t C, float neg_slope, void* stream);
/* replaces: adv = x + eps*tanh(w); tanh backward; torch.optim.Adam([w]).step()
 * (attack_utils.py:40,44-46; torch/optim/adam.py _single_tensor_adam).  step is 1-based. */
int avc_adam_tanh_step(avc_handle* h, const float* g_adv, const float* x, float* w, float* m,
                       float* v, float* adv, int64_t n, float eps, int32_t step, void* stream);

/* Measurement aid for the three HBM-bound unit entry points above (bench.py's roofline legs; SURVEY.md 8d): with reps > 0 each
 * call runs its kernel once and then `reps` more times back to back, timing those with events recorded on `stream` behind the
 * first run, so no host time sits inside the bracket.  avc_unit_last_ms = device milliseconds per repetition of the last call.
 * (The Adam step entry point then applies 1 + reps updates: time it on scratch tensors.)  reps = 0 restores single runs. */
int avc_unit_timing(avc_handle* h, int32_t reps);
float avc_unit_last_ms(const avc_handle* h);

/* ---- VSMask PredictiveModel (SURVEY.md 8a row P; reference models/predictive_model.py:53-110) ------------
 * Own handle: the model is independent of AdaIN-VC.  x is the reference's [B,1,F,T] tensor (contiguous),
 * out [B,1,F',T'] with (F',T') = avc_pm_out_shape(F,T) -- (95,63) for the (80,100) windows of vsmask.py. */
typedef struct avc_pm_handle avc_pm_handle;
/* replaces: PredictiveModel() (predictive_model.py:54-85) */
int avc_pm_create(avc_pm_handle** out, int device);
void avc_pm_destroy(avc_pm_handle* h);
const char* avc_pm_last_error(const avc_pm_handle* h);
/* replaces: load_state_dict (vsmask.py:27-30): the 69 tensors of PredictiveModel.state_dict() by name */
int avc_pm_load_weights(avc_pm_handle* h, const avc_weight_view* tensors, int32_t n);
int avc_pm_out_shape(int32_t F, int32_t T, int32_t* F_out, int32_t* T_out);
/* replaces: PredictiveModel.forward (predictive_model.py:87-110); training != 0 uses BatchNorm batch
 * statistics like model.train() (train_predictive.py:64), 0 the running statistics (vsmask.py:30). */
int avc_pm_forward(avc_pm_handle* h, const float* x, float* out, int32_t B, int32_t F, int32_t T, int32_t training, void* stream);
/* replaces: model.train(); out = model(x); loss = out.square().mean(); loss.backward()  (BASELINE config 5:
 * "predictive_model forward/backward").  out (may be NULL) receives the forward result, loss one float,
 * grad_x (may be NULL) d loss / d x; grads[i].name is a state_dict key, grads[i].data the device buffer of
 * that tensor's shape that receives its gradient ("...running_mean"/"...running_var" receive the updated
 * running statistics instead). */
int avc_pm_train_step(avc_pm_handle* h, const float* x, int32_t B, int32_t F, int32_t T, float* out, float* loss,
                      float* grad_x, const avc_weight_view* grads, int32_t n_grads, void* stream);
int64_t avc_pm_kernel_launches(const avc_pm_handle* h);
/* ---- data-parallel training of the PredictiveModel (SURVEY 8e, BASELINE config 5 "across 2/4/8 GPUs") ---------
 * One process per GPU, each with its own handle and its slice of the global batch.  The sums that couple the ranks --
 * BatchNorm2d batch statistics (sum, sum of squares per channel, predictive_model.py:23) in the forward pass, the two
 * per-channel sums of its backward, and the parameter gradients -- are written into `comm` and handed to the caller's
 * all-reduce (SUM over ranks, in place, ordered on `stream`; the Python host passes torch.distributed.all_reduce over
 * NCCL), so N ranks x B windows compute exactly what one device computes on N*B windows.  world_size 1 / fn NULL
 * switches it off.  The library itself links no communication library. */
typedef int (*avc_allreduce_fn)(void* ctx, float* comm, int64_t n_floats, void* stream);   /* 0 = ok */
int avc_pm_set_allreduce(avc_pm_handle* h, avc_allreduce_fn fn, void* ctx, float* comm, int64_t comm_floats, int32_t world_size);
/* floats `comm` must hold for the gradient all-reduce (= number of trainable parameters, 6 088 904) */
int64_t avc_pm_param_count(const avc_pm_handle* h);

/* ---- VSMask predictor training step (SURVEY 8f rank 3) ---------------------------------------------------------
 * replaces: the loop body of train_predictive_model (train_predictive.py:92-126) with utils/audio.py:77-116
 * (apply_weighted_constraint) and speaker_encoder = the AdaIN-VC SpeakerEncoder of `se` on mel.squeeze(1):
 *   pert = model(source)                                   [B,1,F',T'] = (95,63) for (80,100) windows
 *   delta[:, :, :, fs:fe] = pert[:, :, :F, :fe-fs]          fs = future_steps, fe = min(fs + T', T)   (crop: see below)
 *   delta = clamp per band (bins < int(.3F): eps1, < int(.7F): eps2, else eps3) of (source + delta) - source
 *   perturbed = source + delta
 *   loss = mse(SE(perturbed), SE(target)) - lambda * mse(SE(perturbed), SE(source)); backward; Adam(model.parameters(), lr)
 * The reference as shipped raises at :102 ([B,1,80,63] += [B,1,95,63]) and at utils/audio.py:93 (3-D unpack of a 4-D
 * tensor); this entry point DEFINES the two repairs a maintainer has to make for the loop to run at all: the
 * prediction is cropped to its first F mel rows, and the constraint acts on the mel axis of the 4-D tensor.
 * The handle's weights, BatchNorm running statistics and Adam moments are updated in place on the device. */
typedef struct avc_pm_trainer avc_pm_trainer;
typedef struct avc_pm_trainer_args {
  int32_t B, F, T;                 /* windows [B,1,F,T]; F must equal the speaker encoder's c_in (80)               */
  int32_t future_steps;            /* train_predictive.py:173, default 10                                           */
  float eps1, eps2, eps3;          /* :178-183, 0.1 / 0.05 / 0.08                                                   */
  float lambda;                    /* :184, 0.5                                                                      */
  float beta1, beta2, adam_eps;    /* torch.optim.Adam defaults 0.9 / 0.999 / 1e-8 (:57)                            */
  double inv_norm;                 /* MSELoss normaliser 1/(B_global*128); <= 0: this rank's batch                   */
} avc_pm_trainer_args;
int avc_pm_trainer_begin(avc_pm_handle* pm, avc_handle* se, const avc_pm_trainer_args* a, void* stream, avc_pm_trainer** out);
/* one optimiser step on (source, target) [B,1,F,T] contiguous device tensors; lr is this step's learning rate (the
 * reference's ReduceLROnPlateau, :58-60,131, stays on the host).  loss_out: one device float or NULL (with sharding:
 * this rank's part of the global loss).  Synchronises `stream` before returning (the step's activations go back to the
 * handle's pool). */
int avc_pm_trainer_step(avc_pm_trainer* t, const float* source, const float* target, float lr, float* loss_out, void* stream);
/* d loss / d (parameter) of the LAST step, by state_dict key, PyTorch shapes (test / inspection aid) */
int avc_pm_trainer_grads(avc_pm_trainer* t, const avc_weight_view* grads, int32_t n, void* stream);
int avc_pm_trainer_end(avc_pm_trainer* t);
/* replaces: model.state_dict() after training (train_predictive.py:137-146): copies the handle's current parameters and
 * running statistics into the caller's tensors, by state_dict key */
int avc_pm_export_weights(avc_pm_handle* h, const avc_weight_view* tensors, int32_t n, void* stream);


/* ---- mel front-end and Griffin-Lim back-end (SURVEY.md 8f rank 4; reference data_utils.py:16-31, 65-197) ---------------
 * Own handle: depends only on the preprocessing constants (the reference reads them from config.yaml, data_utils.py:214-220).
 * librosa.load / librosa.effects.trim (file I/O, silence trimming: data_utils.py:93-96) stay on the host. */
typedef struct avc_audio_handle avc_audio_handle;
typedef struct avc_audio_desc {
  int32_t sample_rate, n_fft, hop_length, win_length, n_mels;   /* AdaIN-VC: 24000, 2048, 300, 1200, 80 (BASELINE) / 512 */
  float preemph, ref_db, max_db;                                /* 0.97, 20, 100                                        */
} avc_audio_desc;
int avc_audio_create(avc_audio_handle** out, const avc_audio_desc* d, int device);
void avc_audio_destroy(avc_audio_handle* h);
const char* avc_audio_last_error(const avc_audio_handle* h);
int32_t avc_audio_frames(const avc_audio_handle* h, int64_t n_samples);    /* 1 + n_samples / hop_length (librosa.stft, center=True) */
int64_t avc_audio_samples(const avc_audio_handle* h, int32_t n_frames);    /* hop_length * (n_frames - 1)     (librosa.istft)         */
/* replaces: file2mel from the trimmed waveform on (data_utils.py:99-114): pre-emphasis, |librosa.stft|, mel basis, dB, clip.
 * wav [n] device fp32 -> mel [avc_audio_frames(n)][n_mels] (the reference's mel.T).  Synchronises the stream. */
int avc_audio_wav2mel(avc_audio_handle* h, const float* wav, int64_t n, float* mel, void* stream);
/* replaces: mel2wav (data_utils.py:149-164) incl. griffin_lim (:168-197, n_iter = 100 there) and the de-emphasis lfilter.
 * mel [n_frames][n_mels] -> wav [avc_audio_samples(n_frames)].  Synchronises the stream. */
int avc_audio_mel2wav(avc_audio_handle* h, const float* mel, int32_t n_frames, int32_t n_iter, float* wav, void* stream);
/* the same for B utterances of EQUAL length laid end to end (wav [B][n], mel [B][n_frames][n_mels]): the B*n_frames frames are
 * the rows of one GEMM per transform */
int avc_audio_wav2mel_batch(avc_audio_handle* h, const float* wav, int32_t B, int64_t n, float* mel, void* stream);
int avc_audio_mel2wav_batch(avc_audio_handle* h, const float* mel, int32_t B, int32_t n_frames, int32_t n_iter, float* wav, void* stream);
/* the same for B utterances of ANY lengths laid end to end, in one call: utterance u is samples [s_off[u], s_off[u] + n[u]) of
 * wav and frames [f_off[u], f_off[u] + F[u]) of mel, F[u] = avc_audio_frames(n[u]) (wav2mel) / n_samples = avc_audio_samples(F[u])
 * (mel2wav), the offsets being the prefix sums of the host lengths.  All frames are the rows of one GEMM per transform.
 * mean / std ([n_mels] device fp32, both or neither): wav2mel then writes the speaker-normalised mel (mel - mean) / std, mel2wav
 * reads x * std + mean (data_utils.py:35-47), both correctly rounded and unfused; NULL keeps the plain mel.  Every length is
 * validated as by the equal-length calls.  Synchronises the stream. */
int avc_audio_wav2mel_varlen(avc_audio_handle* h, const float* wav, const int64_t* n_host, int32_t B, const float* mean, const float* std,
                             float* mel, void* stream);
int avc_audio_mel2wav_varlen(avc_audio_handle* h, const float* mel, const int32_t* frames_host, int32_t B, int32_t n_iter, const float* mean,
                             const float* std, float* wav, void* stream);
int64_t avc_audio_kernel_launches(const avc_audio_handle* h);

/* ---- introspection ----------------------------------------------------------------------- */
int64_t avc_kernel_launches(const avc_handle* h);   /* kernels launched (graph nodes x replays) */
int32_t avc_launches_per_iter(const avc_handle* h); /* kernels in the last captured iteration  */
const char* avc_version(void);

#ifdef __cplusplus
}
#endif
#endif /* AVC_B200_H_ */
