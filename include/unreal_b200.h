/*
 * unreal_b200.h -- C ABI of libunreal_b200.so, the B200-native (sm_100a) implementation of
 * the UNREAL rollout-and-target hot path of kvas7andy/unreal.
 *
 * The reference is pure Python and has no FFI of its own; its boundary is the Python class
 * API of Environment / Experience / Trainer / RMSPropApplier (SURVEY.md 8b).  Each entry
 * point below names the reference function (path:line under /root/reference) whose
 * arithmetic it replaces; unreal_b200/_lib.py is the ctypes binding and INTEGRATION.md shows
 * the stub a reference maintainer would add.
 *
 * Conventions
 *   - every function returns UNREAL_OK (0) or a negative UNREAL_E* code and never throws;
 *     unreal_last_error() returns a thread-local message for the last failure.
 *   - all array arguments are caller-owned DEVICE pointers (e.g. torch.Tensor.data_ptr())
 *     unless the name ends in _host; "nullable" arguments may be NULL.
 *   - functions only enqueue work on `stream` (a cudaStream_t passed as void*, NULL = the
 *     legacy default stream); they do not synchronise, allocate, or keep caller pointers.
 *     The only library-owned memory is what *_create() returns handles to.
 *   - layouts are C-contiguous; [T, N] means time-major (one row per rollout step).
 *   - a handle must not be used from two host threads at once; distinct handles are independent.
 *   - work runs on the current device; the maze map is process-wide and applies on every device,
 *     and the library's lazy set-up (kernel attributes, device queries, the map upload) is per device.
 */
#ifndef UNREAL_B200_H_
#define UNREAL_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UNREAL_OK 0
#define UNREAL_EINVAL (-1) /* bad argument (null, size, dtype, alignment) */
#define UNREAL_ECUDA (-2)  /* a CUDA runtime call or launch failed */
#define UNREAL_ESTATE (-3) /* call not valid in the handle's current state */
#define UNREAL_ENOMEM (-4)

/* element type tags for observation / frame buffers */
#define UNREAL_F32 0
#define UNREAL_U8 1 /* 1.0 is stored as 255; loaders divide by 255 (lab/indoor/gym convention) */
#define UNREAL_BF16 2 /* activations between the dense layers (K7); as a maze obs_dtype: the frame in
                         conv1's space-to-depth plane layout x'' [6][441][8] (see unreal_s2d_frames) */

#define UNREAL_MAZE_GRID 7
#define UNREAL_FRAME_HW 84
#define UNREAL_PC_CELLS 20
#define UNREAL_MT_WORDS 624

/* ---- library ------------------------------------------------------------------------ */
const char* unreal_last_error(void);
int unreal_abi_version(void);
/* sm count, compute capability of the current device; fails if it is not sm_100. */
int unreal_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* tunables used by the benchmarks to A/B kernel variants: "maze_render_variant" (0 direct
 * 128-bit stores, 1 TMA bulk store from a shared-memory frame template), ... */
int unreal_set_tunable(const char* name, int value);
int unreal_get_tunable(const char* name, int* value);

/* ---- maze: environment/maze_environment.py --------------------------------------------
 * map49_host: the 49-character map of maze_environment.py:18-25 ('+' wall, 'S', 'G'); it is
 * parsed like _setup (:30-48) and copied to __constant__ memory.  NULL selects the
 * reference map.  Must be called before any other unreal_maze_* call. */
int unreal_maze_set_map(const char* map49_host);
/* start / goal cell of the current map (host ints). */
int unreal_maze_get_layout(int* start_x, int* start_y, int* goal_x, int* goal_y, uint8_t* walls49_host);

/* reset() (:50-55) for every env with mask[i] != 0 (all when mask is NULL):
 * pos <- start, last_action <- 0, last_reward <- 0. */
int unreal_maze_reset(int32_t* pos /*[N,2] x,y*/, int32_t* last_action /*[N]*/, float* last_reward /*[N]*/,
                      const uint8_t* mask /*[N] nullable*/, int n, void* stream);

/* K1: process(action) (:98-128) for N mazes in one launch: _move/_clamp/_is_wall (:66-91),
 * reward/terminal (:114-122), render (_get_current_image :93-96, _put_pixel :57-60) and the
 * pixel change against the previous frame (environment.py:88-99, evaluated in closed form
 * from the old and new cell; see DESIGN.md).  Updates pos / last_action / last_reward in
 * place like :125-127.
 *   active     [N] u8, nullable: envs with 0 are skipped (their rollout already ended);
 *              they get reward 0, terminal 0, an invalid frame record, obs/pc untouched.
 *   obs        [N,84,84,3] of obs_dtype, nullable: env.last_state['image'] AFTER the call,
 *              i.e. the new frame, or the start frame if auto_reset reset the env.
 *   pc         [N,20,20] f32, nullable.
 *   frame_rec  [N] u64, nullable: packed ExperienceFrame (experience.py:10-18) of this step
 *              for unreal_replay_add; layout in DESIGN.md ("frame record").
 *   auto_reset != 0: an env that reached the goal is reset inside the call, which is what
 *              the caller does at trainer.py:201-204, :279-296. */
int unreal_maze_step(int32_t* pos, const int32_t* action /*[N]*/, const uint8_t* active,
                     float* reward /*[N]*/, uint8_t* terminal /*[N]*/, int32_t* last_action,
                     float* last_reward, void* obs, int obs_dtype, float* pc, uint64_t* frame_rec,
                     int n, int auto_reset, void* stream);

/* Window form of unreal_maze_step: T <= 32 process() calls of every env in one launch, for callers that hold the T
 * actions up front (BASELINE configs[1]: the actions are an input of the pass).  action / reward / terminal / frame_rec
 * are [T,N], obs [T,N,84,84,3] (f32 or u8, nullable), pc [T,N,20,20] (nullable), all time-major; pos / last_action /
 * last_reward [N] are advanced by the T steps.  Same results as T unreal_maze_step calls without an `active` mask. */
int unreal_maze_window(int32_t* pos, const int32_t* action, float* reward, uint8_t* terminal, int32_t* last_action,
                       float* last_reward, void* obs, int obs_dtype, float* pc, uint64_t* frame_rec, int n, int t,
                       int auto_reset, void* stream);

/* _get_current_image (:93-96) for M cells: pos [M,2] -> obs [M,84,84,3]. Used to
 * re-materialise frames sampled from the compact replay ring. */
int unreal_maze_render(const int32_t* pos, void* obs, int obs_dtype, int m, void* stream);

/* closed-form pixel change between two cells: pos0, pos1 [M,2] -> pc [M,20,20]. */
int unreal_maze_pixel_change(const int32_t* pos0, const int32_t* pos1, float* pc, int m, void* stream);
/* Trainer._process_pc on replayed MAZE frames (trainer.py:339-380) in one pass: unreal_maze_pixel_change + unreal_pc_targets
 * without the [t,n,20,20] maps between them.  pos0 / pos1 int32 [t,n,2] time-major (the frame's cell and the next frame's),
 * len int32 [n] nullable (valid steps per env; later rows of tgt are zero), boot f32 [n,20,20], tgt f32 [t,n,20,20]. */
int unreal_maze_pc_targets(const int32_t* pos0, const int32_t* pos1, const int32_t* len, const float* boot, float gamma_pc,
                           float* tgt, int t, int n, void* stream);
/* The targets of a maze rollout pass in one launch, from the frame records K1 wrote: the reverse loops of
 * Trainer._process_base (trainer.py:298-324) and Trainer._process_pc (:352-372).  Equal, bit for bit, to
 * unreal_nstep_returns on the pass's rewards / terminals + unreal_pc_targets on its pixel-change maps, which it never
 * reads: the maps are evaluated from the two cells of each record.  A record whose valid bit is 0 counts as reward 0,
 * not terminal and map 0.  rec u64 [t,n], values [t,n] f32, boot_value [n], boot_q [n,20,20] -> out_R, out_adv [t,n]
 * and pc_tgt [t,n,20,20] f32; all time-major. */
int unreal_maze_rollout_targets(const uint64_t* rec, const float* values, const float* boot_value, const float* boot_q,
                                float gamma, float gamma_pc, float* out_R, float* out_adv, float* pc_tgt, int t, int n,
                                void* stream);

/* ---- K2: Environment._calc_pixel_change + _subsample (environment.py:88-99) ------------
 * literal |cur-prev| over the 2-pixel-cropped frame, mean over channels, 4x4 mean.
 * cur, prev: [M,H,W,C] of dtype (u8 values are divided by 255); pc: [M,(H-4)/4,(W-4)/4] f32. */
int unreal_pixel_change(const void* cur, const void* prev, int dtype, float* pc, int m, int h, int w,
                        int c, void* stream);
/* Device self-check of the division-free roundings K2's u8 kernel uses in place of `/ 3` and `/ 255`:
 * mismatches[0] = floats s in [2^-100, 2^100] (all 2^31 - ... of them, and 0) whose two-instruction s/3 differs from the
 * correctly rounded quotient; mismatches[1] = (byte value, byte lane) pairs whose v/255 differs.  Both must be 0. */
int unreal_selfcheck_arith(unsigned long long* mismatches, void* stream);
/* Environment._subsample (environment.py:88-91) on its own: a [M,H,W] f32 -> out [M,H/width,W/width] f32, the mean
 * over width x width blocks taken like numpy's reshape(...).mean(-1).mean(1): columns of a block row first (left to
 * right, then / width), then the block's rows (top to bottom, then / width).  H and W must be multiples of width. */
int unreal_subsample(const float* a, float* out, int m, int h, int w, int width, void* stream);
/* stream form: frames [S, L+1, H,W,C]; pc [S, L, ph, pw] with pc[s,i] = change(frames[s,i+1],
 * frames[s,i]).  Every frame is read from HBM once. */
int unreal_pixel_change_stream(const void* frames, int dtype, float* pc, int s, int l, int h, int w,
                               int c, void* stream);

/* ---- K3: n-step returns and advantages, Trainer._process_base (trainer.py:298-324) -----
 * R_t = r_t + gamma * (term_t ? 0 : R_{t+1}), R_T = boot; adv_t = R_t - v_t.
 * r, v, out_R, out_adv: [T,N] f32; term [T,N] u8; boot [N] f32 (ignored where the last
 * step is terminal).  out_adv / v nullable together (that is Trainer._process_vr's scan,
 * trainer.py:394-403, on time-major data). */
int unreal_nstep_returns(const float* r, const float* v, const uint8_t* term, const float* boot,
                         float gamma, float* out_R, float* out_adv, int t, int n, void* stream);
/* env-major form for sequences gathered from the replay ring: r [N,L] f32, len [N] i32
 * (number of target steps, <= L), boot [N]; one warp per sequence, shuffle scan. */
int unreal_sequence_returns(const float* r, const int32_t* len, const float* boot, float gamma,
                            float* out_R /*[N,L]*/, int n, int l, void* stream);

/* ---- K4: pixel-control Q targets, Trainer._process_pc (trainer.py:352-372) ------------
 * tgt_t = pc_t + gamma_pc * (term_t ? 0 : tgt_{t+1}); tgt_{len} = boot.
 * pc, tgt [T,N,20,20] f32; term [T,N] u8 nullable; len [N] i32 nullable (steps >= len are
 * written as 0); boot [N,20,20]. */
int unreal_pc_targets(const float* pc, const uint8_t* term, const int32_t* len, const float* boot,
                      float gamma_pc, float* tgt, int t, int n, void* stream);

/* ---- RNG: numpy legacy RandomState streams, one per env --------------------------------
 * mt [624,N] u32 (word-major), mt_pos [N] i32.  seed_host: N seeds (RandomState(seed)). */
int unreal_mt_seed(uint32_t* mt, int32_t* mt_pos, const uint32_t* seeds /*[N] device*/, int n, void* stream);
/* Trainer.choose_action (trainer.py:147-148) = RandomState.choice(A, p=pi): pi [N,A] f32 ->
 * action [N] i32; consumes two words per active env. */
int unreal_choose_action(uint32_t* mt, int32_t* mt_pos, const float* pi, const uint8_t* active,
                         int32_t* action, int n, int a, void* stream);
/* raw draws for tests: out [N,K] = randint(0, high) K times per env. */
int unreal_mt_randint(uint32_t* mt, int32_t* mt_pos, uint32_t high, int32_t* out, int n, int k, void* stream);

/* ---- K5: replay ring, train/experience.py ----------------------------------------------
 * Device-resident ring of packed frame records, H slots per env (experience.py:48-60). */
typedef struct unreal_replay unreal_replay_t;
int unreal_replay_create(unreal_replay_t** out, int n_envs, int history_size);
int unreal_replay_destroy(unreal_replay_t* r);
int unreal_replay_reset(unreal_replay_t* r, void* stream);
/* add_frame (:63-93) for every env whose record is valid. */
int unreal_replay_add(unreal_replay_t* r, const uint64_t* frame_rec /*[N]*/, void* stream);
/* is_full (:96-97) per env -> full [N] u8; count/top for tests (nullable). */
int unreal_replay_state(unreal_replay_t* r, uint8_t* full, int32_t* count, int64_t* top,
                        int32_t* n_pos, int32_t* n_neg, void* stream);
/* verbatim export (direction 0) / import (direction 1) of the ring for checkpoints: rec [N,H] u64,
 * top [N] i64, count / n_pos / n_neg [N] i32 (device buffers). */
int unreal_replay_copy(unreal_replay_t* r, int direction, uint64_t* rec, int64_t* top, int32_t* count,
                       int32_t* n_pos, int32_t* n_neg, void* stream);
/* sample_sequence(L) (:100-118) with the env's own MT stream: start [N], len [N] i32 and
 * the gathered records rec [N,L] u64 (entries >= len are 0). */
int unreal_replay_sample_sequence(unreal_replay_t* r, uint32_t* mt, int32_t* mt_pos, int seq_len,
                                  int32_t* start, int32_t* len, uint64_t* rec, void* stream);
/* sample_rp_sequence() (:121-153): start [N] i32 (raw position of the first of 4 frames)
 * and rec [N,4] u64. */
int unreal_replay_sample_rp(unreal_replay_t* r, uint32_t* mt, int32_t* mt_pos, int32_t* start,
                            uint64_t* rec, void* stream);
/* unpack records (any shape, M entries) into SoA fields; every output nullable.
 * pos0 [M,2] i32 state cell, pos1 [M,2] i32 cell after the move, action/last_action [M] i32,
 * reward/last_reward [M] f32, terminal/valid [M] u8. */
int unreal_frame_unpack(const uint64_t* rec, int m, int32_t* pos0, int32_t* pos1, int32_t* action,
                        float* reward, uint8_t* terminal, int32_t* last_action, float* last_reward,
                        uint8_t* valid, void* stream);

/* ---- K5 framed mode (SURVEY.md 8f-4): payloads of generic-frame envs beside the record ring ----
 * For lab / gym / indoor / synthetic frames (environment/{lab,gym,indoor}_environment.py process())
 * the state has no closed form, so what the reference's deque keeps by reference (experience.py:10-18,
 * :71: frame.state['image'], .pixel_change, float .reward / .last_reward, state['objective']) lives in
 * caller-owned payload arrays [N, H, item] addressed by the ring slot of the record.
 * unreal_frame_pack: records for unreal_replay_add from SoA step outputs (cells 0; reward and
 *   last_reward stored as their SIGN, the only thing the ring tests :76-80; inactive envs -> invalid 0). */
int unreal_frame_pack(const int32_t* action, const float* reward, const uint8_t* terminal,
                      const int32_t* last_action /*nullable*/, const float* last_reward /*nullable*/,
                      const uint8_t* active /*nullable*/, uint64_t* rec, int n, void* stream);
/* add_frame (:63-93) that also reports where the frame went: slot [N] i32 = ring slot written, or -1
 * when the frame was discarded (invalid record, terminal directly after terminal :64-67). */
int unreal_replay_add_slots(unreal_replay_t* r, const uint64_t* frame_rec, int32_t* slot, void* stream);
/* payload [N,H,item_bytes] <- src [N,item_bytes] at slot[e] (skipped for slot[e] < 0).  item_bytes a
 * multiple of 4; 128-bit accesses when it is a multiple of 16 and both pointers are 16-byte aligned. */
int unreal_ring_store(void* payload, const void* src, const int32_t* slot, int n_envs, int history_size,
                      long long item_bytes, void* stream);
/* Frame-producer helper of the generic-frame env adapter (environment/frame_environment.py): the new frames of the envs
 * that stepped.  out[e, :] <- src[idx ? idx[e] : e, :] for every env with mask[e] != 0 (mask NULL: all envs, idx NULL:
 * row e); rows of item_bytes bytes (a multiple of 4).  What `image = frames[k]` / the masked upload of a simulator's
 * frame does per env in the reference's env classes (lab_environment.py:99-102, indoor_environment.py:102-103). */
int unreal_rows_select(void* out, const void* src, const int64_t* idx, const uint8_t* mask, int n, long long item_bytes,
                       void* stream);
/* The payloads of a sampled sequence (sample_sequence :109-117 / sample_rp_sequence :146-151 collecting
 * self._frames[start+i]): out item (e,t) <- payload[e, (top[e]+start[e]+t) % H] for t < len[e] (len NULL:
 * all seq_len), zeros beyond and for start[e] < 0.  out is [L,N,item] when time_major else [N,L,item]. */
int unreal_replay_gather(unreal_replay_t* r, const void* payload, long long item_bytes, const int32_t* start,
                         const int32_t* len /*nullable*/, int seq_len, int time_major, void* out, void* stream);

/* ---- rollout bookkeeping (Trainer._process_base, trainer.py:228-296), fused ------------------------------------
 * unreal_rollout_lar: ExperienceFrame.concat_action_and_reward (experience.py:34-46) for every env:
 *   lar [N, A+1+G] f32 = one-hot(last_action, A) ++ [last_reward] ++ objective [N,G] (G = 0: objective NULL).
 * unreal_rollout_post: what follows env.process() in the rollout loop (:265-296), terminal handling as masked
 *   arithmetic so the window never returns to the host: term_now = terminal & active; last_rec = frame_rec where
 *   active; episode_reward += reward; stats [2] f64 += (episodes finished, sum of their scores); for finished envs
 *   ended = 1, active = 0, episode_reward = 0 and their LSTM state rows (lstm_c / lstm_h [N,256] f32, both nullable)
 *   are zeroed (local_network.reset_state :293).  active / ended [N] u8, last_rec [N] u64 in / out. */
int unreal_rollout_lar(const int32_t* last_action, const float* last_reward, const float* objective, int n, int a, int g,
                       float* lar, void* stream);
int unreal_rollout_post(const float* reward, const uint8_t* terminal, const uint64_t* frame_rec, int n, uint8_t* active,
                        uint8_t* ended, uint64_t* last_rec, float* episode_reward, float* lstm_c, float* lstm_h,
                        double* stats, void* stream);

/* ---- evaluation of a frozen policy on the maze (Evaluator, unreal_b200/train/evaluator.py) -----------------------
 * Everything of one evaluation step after the policy, for N mazes in one launch (per-env logic in csrc/eval_core.cuh).
 * For every env with active[e] != 0:
 *   action    greedy != 0: argmax of pi [N,a] f32 (lowest index on ties), no draw; else RandomState.choice(a, p=pi) on
 *             the env's stream mt [624,N] / mt_pos [N] (trainer.py:147-148, two words, as unreal_choose_action);
 *   step      maze_environment.py:98-128 on the map of unreal_maze_set_map; pos [N,2], last_action, last_reward [N]
 *             updated like :125-127;
 *   episode   ep_score [N] += reward, ep_length [N] += 1; at a terminal or at max_steps steps the result row
 *             (e, ep_index[e]) of res_score / res_length / res_finished [N,episodes] is written (finished = terminal),
 *             ep_index advances, the env is reset as after a terminal (trainer.py:201-202, :279-296: start cell, last
 *             action / reward 0, lstm_c / lstm_h rows [N,256] f32 zeroed, local_network.reset_state :293), and after its
 *             `episodes`-th episode active[e] = 0;
 *   operand   row e of the next step's GEMM operand xh bf16 [N, ld_xh] is written: columns [0,256) = fc_tab [49,256]
 *             bf16 row of the new cell, [256, kx) = one-hot(last_action, a) ++ [last_reward] ++ zeros (objective size 0),
 *             [kx, kx+256) = lstm_h row rounded to bf16 (nearest even).
 * Inactive envs are not touched: no draw, no state, result, LSTM or operand write. */
int unreal_maze_eval_act(const float* pi, int a, int greedy, uint32_t* mt, int32_t* mt_pos, int32_t* pos,
                         int32_t* last_action, float* last_reward, float* ep_score, int32_t* ep_length, int32_t* ep_index,
                         uint8_t* active, float* res_score, int32_t* res_length, uint8_t* res_finished, int episodes,
                         int max_steps, float* lstm_c, float* lstm_h, const void* fc_tab_bf16, void* xh_bf16, int64_t ld_xh,
                         int kx, int n, void* stream);

/* ---- K6: shared RMSProp with global-norm clip, train/rmsprop_applier.py ---------------
 * _apply_gradients (:109-132): g <- grad * clip / max(||grad||, clip)  (tf.clip_by_global_norm :121)
 * _apply_dense (:83-93) = TF ApplyRMSProp:  ms += (g*g - ms)*(1-decay);
 *                         mom = momentum*mom + lr*g/sqrt(ms+eps);  var -= mom.
 * All of var/rms/mom/grad are flat [P] f32 (the 20 variables concatenated).
 *   unreal_grad_sumsq   : sumsq[0] += sum(grad^2)  (caller zeroes it; fp32 tree + fp64 atomics)
 *   unreal_rmsprop_update: mom nullable iff momentum == 0; sumsq is the (all-reduced) sum of
 *                         squares on device; clip_norm <= 0 disables clipping; grad_scale
 *                         multiplies grad first (1/world for an averaged all-reduce);
 *                         writes grad_norm[0] (nullable). */
int unreal_grad_sumsq(const float* grad, int64_t p, double* sumsq, void* stream);
int unreal_rmsprop_update(float* var, float* rms, float* mom, const float* grad, int64_t p,
                          const double* sumsq, float grad_scale, float lr, float decay, float momentum,
                          float eps, float clip_norm, float* grad_norm, void* stream);
/* same, with the learning rate read from device memory (lr_dev [1] f32) when the kernel runs: a CUDA graph
 * that captured the update keeps following the annealed rate of trainer.py:140-144. */
int unreal_rmsprop_update_dlr(float* var, float* rms, float* mom, const float* grad, int64_t p,
                              const double* sumsq, float grad_scale, const float* lr_dev, float decay, float momentum,
                              float eps, float clip_norm, float* grad_norm, void* stream);

/* ---- K7: dense layers of UnrealModel (model/model.py:281-598) on the tcgen05 tensor path ------
 * C[M,N] (=|+=) act(A*B + bias + add), bf16 operands, fp32 accumulation in TMEM.
 *   a_mn_major 0: A is row-major [M,K] (lda >= K);  1: A is row-major [K,M] (lda >= M)
 *   b_mn_major 0: B is row-major [N,K] (ldb >= K);  1: B is row-major [K,N] (ldb >= N) -- TF's
 *              [in,out] weight layout (model.py:752-783) is b_mn_major = 1 for tf.matmul(x, W).
 *   c_dtype    UNREAL_GEMM_OUT_F32 / UNREAL_GEMM_OUT_BF16; ldc in elements.
 *   bias [N] f32 nullable; add [M,N] f32 (ld = ldc) nullable; relu != 0 applies max(.,0).
 *   accumulate != 0 or split_k > 1: C (f32) += result with red.global.add (caller zeroes C).
 * lda / ldb must be multiples of 8 elements and all pointers 16-byte aligned (TMA). */
#define UNREAL_GEMM_OUT_F32 0
#define UNREAL_GEMM_OUT_BF16 1
int unreal_gemm_bf16(const void* a, int64_t lda, int a_mn_major, const void* b, int64_t ldb, int b_mn_major,
                     void* c, int64_t ldc, int c_dtype, const float* bias, const float* add, int relu,
                     int accumulate, int split_k, int m, int n, int k, void* stream);

/* tf.nn.conv2d / conv2d_transpose with VALID padding around the GEMM (model.py:786-787, :803-820).
 * in [S,H,W,C] of in_dtype (UNREAL_F32 / UNREAL_U8 (/255) / UNREAL_BF16) ->
 * out bf16 [S*OH*OW, KH*KW*C], column (ky*KW + kx)*C + c, i.e. the row-major order of an HWIO
 * filter.  (H-KH) and (W-KW) must be multiples of the stride. */
int unreal_im2col(const void* in, int in_dtype, void* out_bf16, int s, int h, int w, int c, int kh, int kw,
                  int stride, void* stream);
/* inverse scatter as a gather: out[s,y,x,c] = act(bias[c] + sum of the taps that cover (y,x)).
 * cols [S*OH*OW, KH*KW*C] f32/bf16, out [S,H,W,C] f32/bf16, bias [C] nullable, relu flag. */
int unreal_col2im(const void* cols, int cols_dtype, void* out, int out_dtype, const float* bias, int relu, int s,
                  int h, int w, int c, int kh, int kw, int stride, void* stream);
/* contrib.rnn.BasicLSTMCell(256) pointwise part (model.py:110): gates [N,1024] f32 hold the
 * pre-activations i|j|f|o on entry and their activations on return (forget_bias 1.0);
 * c = c_prev*f + i*j, h = tanh(c)*o; h16 is the bf16 copy fed to the next step's GEMM. */
int unreal_lstm_cell_fwd(float* gates, const float* c_prev, float* c_out, float* h_out, void* h16_out, int n,
                         void* stream);
/* same; h16_out rows are h16_ld elements apart (>= 256): the bf16 h is written straight into columns of the next
 * step's concatenated [x_t, h_{t-1}] GEMM operand, so each step is ONE GEMM over K = |x| + 256 that writes the gate
 * pre-activations once (no separate x-part GEMM, no read-modify-write accumulation). */
int unreal_lstm_cell_fwd_ld(float* gates, const float* c_prev, float* c_out, float* h_out, void* h16_out, int h16_ld,
                            int n, void* stream);
/* acting step (run_base_policy_and_value, model.py:630-660): the cell applied in place to the persistent state
 * c_state / h_state [N,256] f32 of the envs with active[e] != 0 (active NULL: all); h_out [N,256] (nullable) = the
 * state's h afterwards (unchanged for inactive envs). */
int unreal_lstm_cell_act(const float* gates, float* c_state, float* h_state, float* h_out, const uint8_t* active, int n,
                         void* stream);
/* The same cell steps with the gates stored as bf16 [N,1024] (the step GEMM writes the pre-activations as bf16, the
 * activations kept for the backward pass are bf16): fwd = unreal_lstm_cell_fwd_ld, act = unreal_lstm_cell_act,
 * bwd = unreal_lstm_cell_bwd2 (dh_rec nullable).  The cell kernels are HBM-bound on that buffer. */
int unreal_lstm_cell_fwd_g16(void* gates_bf16, const float* c_prev, float* c_out, float* h_out, void* h16_out, int h16_ld,
                             int n, void* stream);
int unreal_lstm_cell_act_g16(const void* gates_bf16, float* c_state, float* h_state, float* h_out, const uint8_t* active,
                             int n, void* stream);
/* unreal_lstm_cell_act_g16 + the acting heads of unreal_a3c_head_loss (model.py:343-377 for one step, run_base_policy_and_value
 * :630-660) in one launch: the warp that computes an env's row of h also reduces softmax(h . Wp + bp) -> pi_out [N,A] and
 * h . Wv + bv -> v_out [N]; wp f32 [256,A], wv f32 [256], a in 1..7.  Inactive envs keep c / h and report the heads of
 * the h they hold. */
int unreal_lstm_cell_act_heads(const void* gates_bf16, float* c_state, float* h_state, const uint8_t* active, int n,
                               const float* wp, const float* bp, const float* wv, const float* bv, int a, float* pi_out,
                               float* v_out, void* stream);
int unreal_lstm_cell_bwd_g16(const void* gates_act_bf16, const float* c_prev, const float* c, const float* dh,
                             const float* dh_rec, float* dc, void* dgates_bf16, int n, void* stream);
/* One LSTM step as ONE launch: the step GEMM over [x_t, h_{t-1}] with the BasicLSTMCell arithmetic in its epilogue
 * (model/model.py:110, :343-351; a tile holds all four gates of 64 units, the pre-activations never reach HBM).
 *   xh [N, k] bf16, rows ld_xh apart (k = lstm input + padding + 256); w [k,1024] bf16 (i | j | f | o columns); bias [1024]
 *   c_prev -> c_out [N,256] f32 (may alias: the acting step updates the persistent state in place); h_out [N,256] f32
 *   (nullable); h16_out bf16 rows h16_ld apart (nullable: the next step's operand columns); acts [N,1024] bf16
 *   (nullable: the gate activations the backward pass reads); active [N] (nullable): rows with 0 keep c / h, and
 *   h_copy [N,256] (nullable, needs h_out) receives every row's h -- the new one, or what h_out held.
 *   tiled != 0: c_prev, c_out and acts are in the 32-row tiled layout the epilogue accesses contiguously (rows padded
 *   to a multiple of 32; 16-byte chunk ch of row r at 16 * ((r / 32 * chunks_per_row + ch) * 32 + r % 32)); these are
 *   buffers only this kernel and unreal_lstm_step_bwd touch.
 * Replaces unreal_gemm_bf16 + unreal_lstm_cell_fwd_g16 / unreal_lstm_cell_act_g16. */
int unreal_lstm_step_fwd(const void* xh, int64_t ld_xh, const void* w, const float* bias, const float* c_prev, float* c_out,
                         float* h_out, float* h_copy, void* h16_out, int h16_ld, void* acts, const uint8_t* active, int tiled,
                         int n, int k, void* stream);
/* One backward LSTM step as ONE launch: dh_rec = dgates_next [N,1024] bf16 x wh [256,1024]^T bf16 (the h rows of the
 * cell's kernel, rows ld_wh apart) on the tensor cores, and in its epilogue the cell's backward pass of step t on
 * dh [N,256] + dh_rec (the gradient of tf.nn.dynamic_rnn's unroll, model.py:343-351): acts [N,1024] bf16 step t's gate
 * activations, c_prev / c [N,256]; dc [N,256] in: wrt c_t, out: wrt c_{t-1}; dgates [N,1024] bf16 out (row-major).
 * dgates_next NULL = the unroll's last step: no product, dh2 [N,256] (nullable) is added to dh instead.
 * tiled != 0: acts, c_prev, c and dc are in unreal_lstm_step_fwd's tiled layout.
 * Replaces unreal_gemm_bf16 + unreal_lstm_cell_bwd_g16. */
int unreal_lstm_step_bwd(const void* dgates_next, const void* wh, int64_t ld_wh, const void* acts, const float* c_prev,
                         const float* c, const float* dh, const float* dh2, float* dc, void* dgates, int tiled, int n,
                         void* stream);
/* backward of the above: dh [N,256] total gradient wrt h_t; dc [N,256] in: wrt c_t, out: wrt
 * c_{t-1}; dgates bf16 [N,1024] wrt the pre-activations. */
int unreal_lstm_cell_bwd(const float* gates_act, const float* c_prev, const float* c, const float* dh, float* dc,
                         void* dgates_bf16, int n, void* stream);
/* same with the gradient w.r.t. h_t given as two addends, dh + dh_rec (heads' gradient and the recurrent one from
 * step t+1; dh_rec nullable): saves the element-wise add between the steps of the backward unroll. */
int unreal_lstm_cell_bwd2(const float* gates_act, const float* c_prev, const float* c, const float* dh,
                          const float* dh_rec, float* dc, void* dgates_bf16, int n, void* stream);

/* Fused convolutions of the encoder (model.py:281-289) as implicit GEMMs whose im2col is done by
 * the TMA engine (multi-dimensional boxes over a space-to-depth view; no patch matrix in memory).
 *   unreal_s2d_frames: frames [S,84,84,3] f32 / u8 (/255) -> x'' bf16 [S,6,441,8] (plane-major):
 *                      x''[s, q, Y*21+X, e] = frame[4Y+dy, 4X+dx, c], dy*12 + dx*3 + c = q*8 + e.
 *   unreal_conv_fwd  : layer 1: in = x'' -> out bf16 [S,20,20,16] = relu(conv 8x8 s4 + bias);
 *                        w bf16 [4 taps][6 chunks][16 out][8]: tap t = by*2+bx, W[4by+dy, 4bx+dx, c, o].
 *                      layer 2: in = h1 bf16 [S,20,20,16] -> out bf16 [S,9,9,32] = relu(conv 4x4 s2 + bias);
 *                        w bf16 [32 out, 256]: column (ky*4 + kx)*16 + c holds W[ky, kx, c, o] (HWIO transposed). */
int unreal_s2d_frames(const void* frames, int dtype, void* out_bf16, int s, void* stream);
int unreal_conv_fwd(const void* in_bf16, int layer, const void* w_taps_bf16, const float* bias, void* out_bf16, int s,
                    void* stream);
/* conv2's geometry (4x4 stride 2 VALID over [S,20,20,16] -> [S,9,9,32]) without bias and ReLU: the input gradient of
 * the pixel-control head's transposed convolution (model.py:418-430 backward) is this convolution of d loss / d y
 * (padded to 16 channels) with the deconv filter; w as in unreal_conv_fwd layer 2. */
int unreal_conv2_fwd_linear(const void* in_bf16, const void* w_taps_bf16, void* out_bf16, int s, void* stream);

/* ReLU backward fused with the bias gradient (tf.nn.relu / bias_add gradients of the dense layers):
 * out_bf16 = dy * (y > 0) and db[c] += sum_rows out[:, c]; y_bf16 NULL: no mask; out / db nullable.
 * dy [rows, cols] bf16 or f32 (contiguous), cols a multiple of 8; the caller zeroes db. */
int unreal_relu_grad(const void* dy, int dy_dtype, const void* y_bf16, void* out_bf16, float* db, int64_t rows,
                     int cols, int out_planes /* 1: out is [cols/8][rows][8] */, void* stream);
/* conv1 filter gradient on the tensor path, reading the forward's x'' and the masked dY planes
 * ([2][S*400][8] bf16 from unreal_relu_grad with out_planes = 1) once each:
 * dw_taps f32 [4 taps][16 out][48 (dy,dx,c)] += sum_pixels dY * x' (caller zeroes dw_taps). */
int unreal_conv1_wgrad(const void* xpp_bf16, const void* dy_planes_bf16, float* dw_taps, int s, void* stream);
/* same, with the dY planes on the x'' grid's 21-pixel row pitch ([2][S*420][8], column ox = 20 zero; written by
 * unreal_conv2_dgrad_relu with pitch21 = 1): one 1680-byte bulk copy per plane and work item instead of five
 * 320-byte ones. */
/* Render-fused conv1 for the maze env type: pos [S,2] i32 (agent cell x, y of each frame) instead of frames.
 * The kernels synthesise each work item's x'' tile in shared memory from the cell and the wall map set by
 * unreal_maze_set_map (maze_environment.py:30-41, :57-60, :93-96: the frame is a pure function of the position),
 * bit-identical to what unreal_maze_render(dtype bf16) would have written: no frame is written to or read from
 * HBM for the forward pass or the filter gradient.  out / dw_taps / dy planes as in unreal_conv_fwd (layer 1) /
 * unreal_conv1_wgrad_p21. */
int unreal_conv1_fwd_maze(const int32_t* pos, const void* w_taps_bf16, const float* bias, void* out_bf16, int s,
                          void* stream);
int unreal_conv1_wgrad_maze(const int32_t* pos, const void* dy_planes21_bf16, float* dw_taps, int s, void* stream);
/* Split-bf16 ("bf16x3") encoder forward, for reference-grade (fp32-like) products on the bf16 tensor path: every fp32
 * operand a is carried as a_hi = bf16(a) and a_lo = bf16(a - a_hi), and a.b is accumulated as
 * a_hi.b_hi + a_hi.b_lo + a_lo.b_hi in fp32.  Layouts are those of the bf16 entry points above; *_lo filters are the
 * same tap layouts of bf16(W - bf16(W)).
 *   unreal_s2d_frames_split    : as unreal_s2d_frames, plus the lo planes.
 *   unreal_conv1_fwd_split     : x'' hi / lo planes (xpp_lo NULL: the input is exactly bf16, two passes)
 *                                -> h1 = relu(conv + bias) as a hi / lo pair of bf16 [S,20,20,16].
 *   unreal_conv1_fwd_maze_split: render-fused (the rendered frames are exactly 0 / 1: two passes) -> h1 hi / lo.
 *   unreal_conv2_fwd_split     : h1 hi / lo -> h2 bf16 [S,9,9,32] = relu(conv + bias).
 * With zero lo filters and a zero (or NULL) lo input the results equal the bf16 entry points bit for bit. */
int unreal_s2d_frames_split(const void* frames, int dtype, void* out_hi_bf16, void* out_lo_bf16, int s, void* stream);
int unreal_conv1_fwd_split(const void* xpp_hi_bf16, const void* xpp_lo_bf16, const void* w_hi_bf16, const void* w_lo_bf16,
                           const float* bias, void* out_hi_bf16, void* out_lo_bf16, int s, void* stream);
int unreal_conv1_fwd_maze_split(const int32_t* pos, const void* w_hi_bf16, const void* w_lo_bf16, const float* bias,
                                void* out_hi_bf16, void* out_lo_bf16, int s, void* stream);
int unreal_conv2_fwd_split(const void* h1_hi_bf16, const void* h1_lo_bf16, const void* w_hi_bf16, const void* w_lo_bf16,
                           const float* bias, void* out_bf16, int s, void* stream);
int unreal_conv1_wgrad_p21(const void* xpp_bf16, const void* dy_planes21_bf16, float* dw_taps, int s, void* stream);
/* conv2 filter gradient from h1 [S,20,20,16] bf16 and the masked dY2 [S*81,32] bf16, both read once through
 * TMA boxes: dw_taps f32 [4 ky][64 (kx,c)][32 out] = HWIO [4,4,16,32] += ... (caller zeroes dw_taps). */
int unreal_conv2_wgrad(const void* h1_bf16, const void* dy_bf16, float* dw_taps, int s, void* stream);
/* conv2 input gradient (transposed convolution) as a 4-tap implicit GEMM over zero-filling TMA boxes:
 * dy [S*81,32] bf16, w_dtaps bf16 [4 taps][64 (dy,dx,c)][32 out] = W2[2by+dy, 2bx+dx, c, o]
 * -> dh1 bf16 [S,20,20,16] (un-masked; unreal_relu_grad applies conv1's ReLU mask). */
int unreal_conv2_dgrad(const void* dy_bf16, const void* w_dtaps_bf16, void* dh1_bf16, int s, void* stream);
/* unreal_conv2_dgrad fused with the ReLU gradient of the layer below (conv1, model.py:285: h1 = relu(...)):
 * the transposed convolution's result is masked by h1 > 0, rounded to bf16 and written as the two
 * 8-channel planes [2][S*400][8] that unreal_conv1_wgrad consumes (pitch21 != 0: [2][S*420][8] on a 21-pixel row
 * pitch with a zero column, for unreal_conv1_wgrad_p21); db1 [16] f32 (caller-zeroed, atomically
 * accumulated, nullable) receives conv1's bias gradient.  Replaces unreal_conv2_dgrad + unreal_relu_grad. */
int unreal_conv2_dgrad_relu(const void* dy_bf16, const void* w_dtaps_bf16, const void* h1_bf16,
                            void* dy1_planes_bf16, float* db1, int s, int pitch21, void* stream);
/* The pixel-control head's two transposed convolutions as ONE 8-channel deconv, forward (model.py:418-430,
 * :803-820 conv2d_transpose 4x4 stride 2 VALID + bias + ReLU): h bf16 [S,9,9,32], w_dtaps bf16
 * [4 taps, 32 (dy,dx,c8), 32 in] (the merged [kh,kw,8,32] filter in unreal_conv2_dgrad's tap order),
 * bias8 f32 [8] (nullable) -> y8 f32 [S,20,20,8].  Same tcgen05 kernel as unreal_conv2_dgrad with 8 channels. */
int unreal_pc_deconv_fwd(const void* h_bf16, const void* w_dtaps_bf16, const float* bias8, float* y8, int s,
                         void* stream);

/* Policy / value heads and the A3C losses in one pass over h [M,256] f32 (model.py:358-377 heads; :499-527 base
 * policy + entropy + value loss; :556-565 value-replay loss): logits = h Wp + bp, pi = softmax, v = h Wv + bv
 * (Wp [256,A], Wv [256]: TF [in,out] layouts, fp32).  Every output is nullable:
 *   pi_out [M,A], v_out [M]                       the acting outputs of run_base_policy_and_value / run_base_value
 *   sums [3] f64 += (policy loss, value loss, entropy) with act [M] i32, adv, r, mask [M] f32 (mask NULL: all ones):
 *     policy = -sum mask (log pi[a] adv + entropy_beta H), value = value_coef sum mask (r - v)^2, pi clamped to [1e-20,1]
 *   dz [M,A] = d policy / d logits, dv [M] = d value / d v   (consumed by unreal_a3c_head_bwd)
 * act NULL: no policy loss (value replay); r NULL: no value loss; a = 0 / wp NULL: value head only.
 * a <= 15 (a <= 7 runs the 8-output build, a = 8..15 the 16-output one; unreal_a3c_head_bwd alike). */
int unreal_a3c_head_loss(const float* h, const float* wp, const float* bp, const float* wv, const float* bv,
                         const int32_t* act, const float* adv, const float* r, const float* mask, int64_t m, int a,
                         float entropy_beta, float value_coef, float* pi_out, float* v_out, double* sums, float* dz,
                         float* dv, void* stream);
/* backward of the two heads: go2 [2] f32 on the device = incoming gradients of (policy, value) losses;
 * dh [M,256] = go_p dz Wp^T + go_v dv Wv^T (written), dwp [256,A] / dbp [A] / dwv [256] / dbv [1] += (caller-zeroed). */
int unreal_a3c_head_bwd(const float* h, const float* wp, const float* wv, const float* dz, const float* dv,
                        const float* go2, int64_t m, int a, float* dh, float* dwp, float* dbp, float* dwv, float* dbv,
                        void* stream);
/* Maze-cell de-duplication of the encoder: a maze frame is a pure function of the agent cell (maze_environment.py:93-96),
 * so conv1 -> conv2 -> fc1 (model.py:281-289, :332-340) over all samples of an update is a lookup in a 49-row table
 * (cell index y*7+x) and its backward pass a segment sum by cell.  pos [S,2] i32 = the samples' agent cells (x, y).
 *   gather:       out[s, 0:d] = table[cell(s), 0:d]                 bf16; out rows are ld_out elements apart
 *   segment_sum:  out[cell, 0:256] += sum_{s: cell(s)=cell} dy[s]   dy f32 / bf16 [S,256], out f32 [49,256] (caller-zeroed) */
int unreal_cell_gather(const void* table_bf16, const int32_t* pos, void* out_bf16, int64_t ld_out, int64_t s, int d,
                       void* stream);
int unreal_cell_segment_sum(const void* dy, int dy_dtype, const int32_t* pos, float* out, int64_t s, int d, void* stream);
/* Pixel-control head with its loss fused into the deconv (unreal_pc_deconv_fwd + unreal_pc_loss + unreal_pc_loss_grad16 in
 * one kernel; model.py:418-441, :531-546): h bf16 [S,9,9,32] -> loss (double, accumulated) and d loss / d (pre-ReLU deconv
 * output) as conv2-geometry input dy16 bf16 [S,400,16] (channels 8..15 zero), NOT yet multiplied by the upstream
 * gradient, plus the deconv bias gradient db8 [8] (caller-zeroed, nullable).  The f32 head output is never materialised.
 * unreal_conv2_fwd_linear_scaled = unreal_conv2_fwd_linear with the accumulators multiplied by *scale (device scalar):
 * the backward convolution applying that upstream gradient. */
int unreal_pc_deconv_loss(const void* h_bf16, const void* w_dtaps_bf16, const float* bias8, const int32_t* act,
                          const float* target, const float* mask, int a, float lam, int s, double* loss, void* dy16_bf16,
                          float* db8, void* stream);
int unreal_conv2_fwd_linear_scaled(const void* in_bf16, const void* w_taps_bf16, const float* scale, void* out_bf16, int s,
                                   void* stream);
/* unreal_conv2_fwd_linear_scaled + the ReLU gradient of the layer its result flows into (pc_fc1, model.py:424, whose
 * output [S,2592] is the deconv's input [S,9,9,32]): the epilogue zeroes the result where mask_y_bf16 [S,9,9,32] <= 0,
 * rounds to bf16 and adds the rounded values summed over samples to db [2592] (pc_fc1's bias gradient; caller-zeroed,
 * nullable) -- replaces unreal_relu_grad over the dense [S,2592] gradient.  scale nullable (1). */
int unreal_conv2_fwd_linear_masked(const void* in_bf16, int c_in, const void* w_taps_bf16, const float* scale,
                                   const void* mask_y_bf16, void* out_bf16, float* db, int s, void* stream);
/* The same pixel-control backward pass on the loss gradient WITHOUT its 8 zero padding channels (half the bytes of the
 * largest tensor of the update, written once and read twice): unreal_pc_deconv_loss_c8 writes dy8 bf16 [S,400,8];
 * unreal_conv2_fwd_linear_masked takes it with c_in = 8 (in_bf16 [S,20,20,c_in], w_taps [32, 16*c_in]);
 * unreal_conv2_wgrad_c8 = unreal_conv2_wgrad over an 8-channel activation x8 [S,20,20,8] -> dw [4,4,8,32] (accumulated). */
int unreal_pc_deconv_loss_c8(const void* h_bf16, const void* w_dtaps_bf16, const float* bias8, const int32_t* act,
                             const float* target, const float* mask, int a, float lam, int s, double* loss, void* dy8_bf16,
                             float* db8, void* stream);
int unreal_conv2_wgrad_c8(const void* x8_bf16, const void* dy_bf16, float* dw_taps, int s, void* stream);
/* ... and on the PLANE-MAJOR loss gradient, the layout the agent runs: unreal_pc_deconv_loss_planes writes the gradient as
 * four parity planes of the 10 x 10 space-to-depth grid, dy_planes bf16 [S][4 = (dy,dx)][100 = (Y,X)][8]: element
 * (y, x, c) of the [20,20,8] gradient sits at plane (y&1, x&1), row (y>>1)*10 + (x>>1).  A sample is then ONE 6400-byte bulk
 * copy for both backward kernels instead of four overlapping TMA boxes (which bound the kernels above by the TMA engine's
 * row rate, not by HBM):
 *   unreal_pc_planes_conv  = unreal_conv2_fwd_linear_masked (w_planes bf16 [4 taps (by,bx)][2 dy][2 dx][32 o][8 c] =
 *                            W8[2by+dy][2bx+dx][c][o] of the merged deconv filter; scale nullable; db [2592] nullable);
 *   unreal_pc_planes_wgrad = unreal_conv2_wgrad_c8 (hp bf16 [S,9,9,32] -> dw8 f32 [4,4,8,32] HWIO, accumulated). */
int unreal_pc_deconv_loss_planes(const void* h_bf16, const void* w_dtaps_bf16, const float* bias8, const int32_t* act,
                                 const float* target, const float* mask, int a, float lam, int s, double* loss,
                                 void* dy_planes_bf16, float* db8, void* stream);
int unreal_pc_planes_conv(const void* dy_planes_bf16, const void* w_planes_bf16, const float* scale, const void* mask_y_bf16,
                          void* out_bf16, float* db, int s, void* stream);
int unreal_pc_planes_wgrad(const void* dy_planes_bf16, const void* hp_bf16, float* dw8, int s, void* stream);
/* The bootstrap of Trainer._process_pc (run_pc_q_max, model.py:707-712; :431-441): the same deconv with the dueling combine
 * and the max over actions in its epilogue -> qmax f32 [S,20,20]; the head output itself is not written. */
int unreal_pc_deconv_qmax(const void* h_bf16, const void* w_dtaps_bf16, const float* bias8, int a, int s, float* qmax,
                          void* stream);
/* The 16-channel pixel-control head for 8..15 actions (model.py:411-441 head and dueling combine, :531-546 loss, :707-712
 * run_pc_q_max): the merged deconv filter [4,4,16,32] holds the value in channel 0 and the advantages in channels 1..a
 * (the rest zero); w_dtaps bf16 [4 taps, 64 (dy,dx,c), 32] (conv2's transposed-convolution tap layout), bias16 f32 [16].
 *   unreal_pc_deconv_loss16: h bf16 [S,9,9,32] -> loss (double, accumulated) += lam 0.5 sum mask (R - Q_act)^2,
 *     dy16 bf16 [S,400,16] = d loss / d (pre-ReLU deconv output), every channel real and not yet multiplied by the upstream
 *     gradient (unreal_conv2_fwd_linear_masked with c_in 16 and unreal_conv2_wgrad take it), db16 f32 [16] += the
 *     bias gradient (caller-zeroed, nullable); act [S] i32, target [S,20,20] f32, mask [S] f32.
 *   unreal_pc_deconv_qmax16: qmax f32 [S,20,20] = max over actions of the dueling combine.
 * a outside 8..15 is an argument error (a <= 7 is the 8-channel head above). */
int unreal_pc_deconv_loss16(const void* h_bf16, const void* w_dtaps_bf16, const float* bias16, const int32_t* act,
                            const float* target, const float* mask, int a, float lam, int s, double* loss, void* dy16_bf16,
                            float* db16, void* stream);
int unreal_pc_deconv_qmax16(const void* h_bf16, const void* w_dtaps_bf16, const float* bias16, int a, int s, float* qmax,
                            void* stream);
/* Reward-prediction head after its fc GEMM (model.py:482-488 softmax, :571-575 loss).  logits8 [N,8] f32: columns 0..2 =
 * features . W_rp (the bf16 tcgen05 GEMM on the weight shadow padded to 8 columns), bias [3] added here.
 *   p_out (nullable) [N,3] = softmax(logits + bias)                                  (run_rp_c, model.py:723-728)
 *   loss  (nullable, double, accumulated) += -sum c log(clip(p, 1e-20, 1)) with c [N,3] f32 ([zero, positive, negative])
 *   dz16  (nullable) bf16 [N,8] = *go * d loss / d logits (columns 3..7 zero: the GEMM operand of the backward pass),
 *   db [3] += column sums of dz (caller-zeroed).  go: device scalar, nullable = 1. */
int unreal_rp_loss(const float* logits8, const float* bias, const float* c, int64_t n, float* p_out, double* loss,
                   void* dz16, float* db, const float* go, void* stream);
/* Pixel-control head: dueling combine, Q(a) gather and L2 loss in one pass (model.py:431-441, :531-546).
 * y8 [samples*px, 8] f32 = merged deconv output after ReLU (channel 0 V, 1..A advantages, rest padding);
 * act [samples] i32; target [samples*px] f32; mask [samples] f32.
 * loss (nullable, double, accumulated): lam * 0.5 * sum mask * (target - Q[act])^2.
 * dy8 (nullable): d loss / d (pre-ReLU output) scaled by *go (device scalar, nullable = 1). */
int unreal_pc_loss(const float* y8, const int32_t* act, const float* target, const float* mask, int a, float lam,
                   int64_t samples, int px_per_sample, double* loss, float* dy8, const float* go, void* stream);
/* gradient only, written as the conv2-geometry input of the deconv's backward: dy16 bf16 [S*px, 16] (channels 8..15
 * zero) and the deconv bias gradient db8 [8] f32 (caller-zeroed, atomically accumulated, nullable). */
int unreal_pc_loss_grad16(const float* y8, const int32_t* act, const float* target, const float* mask, int a, float lam,
                          int64_t samples, int px_per_sample, void* dy16_bf16, float* db8, const float* go, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* UNREAL_B200_H_ */
