/*
 * gnnpp_b200.h -- C ABI of libgnnpp_b200.so: the B200 (sm_100a) implementation of the
 * DecentralPlannerNet forward path of proroklab/gnn_pathplanning.
 *
 * The reference has no FFI of its own: its boundary for this path is the PyTorch
 * nn.Module API (SURVEY.md section 8b).  This header is the C-level boundary a
 * reference maintainer binds to (ctypes stub in INTEGRATION.md); every entry point
 * names the reference code it replaces.  Plain pointers and sizes only -- no torch
 * types.  All functions return 0 on success, a negative gpp_status otherwise;
 * gpp_last_error() returns a thread-local human-readable message.
 *
 * Conventions
 *   B batch (episodes), N agents (graph nodes), G input / F output features,
 *   K filter taps, E = 1 edge feature (the only value the reference path constructs,
 *   graphs/models/decentralplanner.py:209).
 *   `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   "dev" pointers are device memory, "host" pointers are host memory (pinned for
 *   full copy speed); neither is retained after the call returns unless stated.
 */
#ifndef GNNPP_B200_H
#define GNNPP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum gpp_status {
    GPP_OK = 0,
    GPP_ERR_INVALID = -1,     /* bad argument / shape (the reference raises AssertionError) */
    GPP_ERR_UNSUPPORTED = -2, /* valid in the reference but outside this library's envelope */
    GPP_ERR_CUDA = -3,        /* CUDA runtime error (message has the cudaError string) */
    GPP_ERR_NODEVICE = -4     /* no sm_100 device visible */
} gpp_status;

/* Tensor layouts of the node-signal tensors x / y. */
typedef enum gpp_layout {
    GPP_FEATURE_MAJOR = 0, /* [B, G, N]: the reference API layout (graphML.py:2298-2306) */
    GPP_NODE_MAJOR = 1     /* [B, N, G]: the native layout between the fused stages */
} gpp_layout;

const char* gpp_last_error(void);
int gpp_abi_version(void);
/* Fills SM count and compute capability of the current device. */
int gpp_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------
 * Graph filter  (replaces BatchLSIGF, utils/graphUtils/graphML.py:2273-2367, as called
 * by GraphFilterBatch.forward :2458-2477)
 *
 *   z_0 = x ; z_k = z_{k-1} . S_b  (right multiplication, :2350)
 *   y[b,f,n] = sum_{k,g} w[f,0,k,g] z_k[b,g,n] + bias[f]          (:2361-2366)
 *
 *   x      dev f32, layout x_layout, B*G*N
 *   S      dev [B,N,N], f32 or (s_is_f64 != 0) f64 -- cast to f32 per element exactly as
 *          `S.float()` does at :2350
 *   w      dev f32 [F,1,K,G]  (the module's `weight`, untouched layout)
 *   bias   dev f32 [F] or NULL
 *   y      dev f32, layout y_layout, B*F*N
 *   fuse_relu  apply max(.,0) in the epilogue (the nn.ReLU that follows the filter in
 *          DecentralPlannerNet.GFL, decentralplanner.py:221)
 *   workspace  dev scratch of gpp_graph_filter_workspace_bytes() bytes (holds the
 *          k-major transposed taps); may be NULL only if that size is 0
 * ---------------------------------------------------------------------------------- */
size_t gpp_graph_filter_workspace_bytes(int G, int F, int K);

int gpp_graph_filter_forward(const float* x, const void* S, int s_is_f64,
                             const float* w, const float* bias, float* y,
                             int B, int N, int G, int F, int K,
                             int x_layout, int y_layout, int fuse_relu,
                             void* workspace, void* stream);

/* Backward of the same filter (replaces autograd through graphML.py:2342-2366).
 *   dy   dev f32 [B,F,N]/[B,N,F] (y_layout) upstream gradient
 *   y    dev f32, the forward OUTPUT (needed only when fuse_relu, for the mask), else NULL
 *   dx   dev f32 out, x_layout         (NULL to skip)
 *   dw   dev f32 out [F,1,K,G]         (NULL to skip; overwritten, not accumulated)
 *   dbias dev f32 out [F]              (NULL to skip; overwritten)
 *   workspace: gpp_graph_filter_backward_workspace_bytes() bytes of dev scratch.
 * S receives no gradient (the reference's GSO never requires grad). */
size_t gpp_graph_filter_backward_workspace_bytes(int B, int N, int G, int F, int K);

int gpp_graph_filter_backward(const float* dy, const float* y, const float* x,
                              const void* S, int s_is_f64, const float* w,
                              float* dx, float* dw, float* dbias,
                              int B, int N, int G, int F, int K,
                              int x_layout, int y_layout, int fuse_relu,
                              void* workspace, void* stream);

/* ------------------------------------------------------------------------------------
 * Whole-planner inference  (replaces DecentralPlannerNet.addGSO + forward in eval mode,
 * graphs/models/decentralplanner.py:266-318: per-agent CNN + compress MLP -> K-tap graph
 * filter + ReLU -> per-agent action MLP)
 * ---------------------------------------------------------------------------------- */
typedef struct gpp_planner gpp_planner;

/* All pointers use the reference's state_dict shapes (SURVEY.md section 8 a1):
 *   conv_w[l]  [C_{l+1}, C_l, 3, 3]   conv_b[l] [C_{l+1}]     C = 3,32,32,64,64,128
 *   bn_w/bn_b/bn_mean/bn_var[l] [C_{l+1}]   (eval-mode BatchNorm2d, eps 1e-5)
 *   compress_w [128,128] compress_b [128]; gf_w [128,1,K,128] gf_b [128] (from [128,1]);
 *   action_w [5,128] action_b [5] */
typedef struct gpp_planner_weights {
    const float* conv_w[5];
    const float* conv_b[5];
    const float* bn_w[5];
    const float* bn_b[5];
    const float* bn_mean[5];
    const float* bn_var[5];
    const float* compress_w;
    const float* compress_b;
    const float* gf_w;
    const float* gf_b;
    const float* action_w;
    const float* action_b;
} gpp_planner_weights;

/* K = number of graph-filter taps (config.nGraphFilterTaps, decentralplanner.py:131). */
int gpp_planner_create(gpp_planner** out, int K);
void gpp_planner_destroy(gpp_planner* p);

/* Copies/re-lays-out the parameters into the planner's private device arena
 * (k-major conv/linear weights, BatchNorm folded to per-channel scale/shift).
 * `on_device` != 0: the pointers are device pointers, work is enqueued on `stream`;
 * == 0: host pointers (synchronous). Call again whenever the parameters change. */
int gpp_planner_set_weights(gpp_planner* p, const gpp_planner_weights* w, int on_device,
                            void* stream);

/* Device-resident forward.
 *   x       dev f32 [B,N,3,11,11]
 *   S       dev [B,N,N] f32 / f64 (s_is_f64)
 *   logits  dev f32 out [N,B,5]  -- agent-major, so that the reference's Python list of N
 *           tensors [B,5] (decentralplanner.py:303-318) is N contiguous views
 *   features_out  optional dev f32 [B,N,128] node-major CNN+compress features (may be NULL)
 */
int gpp_planner_forward(gpp_planner* p, const float* x, const void* S, int s_is_f64,
                        float* logits, float* features_out, int B, int N, void* stream);

/* Host-buffer forward: H2D copies of x and S, the forward, and the D2H copy of the logits
 * all run on the planner's own stream; returns after the logits are in `logits_host`.
 * This is the call a rollout loop makes once per step (agents/decentralplannerlocal.py
 * :563-580 does the same with .to(device) + model(...)). */
int gpp_planner_forward_host(gpp_planner* p, const float* x_host, const void* S_host,
                             int s_is_f64, float* logits_host, int B, int N);

/* ------------------------------------------------------------------------------------
 * Whole-planner TRAINING forward / backward (replaces DecentralPlannerNet.forward in train mode,
 * decentralplanner.py:278-318, and the autograd pass behind loss.backward(),
 * agents/decentralplannerlocal.py:297-314).  All pointers are device pointers.
 *
 * BatchNorm follows the reference's per-agent semantics: the reference calls ConvLayers once per agent, so
 * batch statistics are over (B,H,W) of one agent's slice and the running statistics receive N sequential
 * momentum updates per forward, in agent order (bn == NULL or NULL members: no running-stat update).
 *   logits   out [N,B,5]                         dlogits  in [N,B,5]  (gradient of the loss)
 *   workspace: gpp_planner_train_workspace_bytes(B,N,K) bytes; written by the forward (saved activations),
 *              read and scribbled on by the backward of the SAME step.
 *   grads: every member is overwritten (not accumulated) with the gradient of the matching parameter.
 * ---------------------------------------------------------------------------------- */
typedef struct gpp_planner_bn_state {
    float* running_mean[5];
    float* running_var[5];
} gpp_planner_bn_state;

typedef struct gpp_planner_grads {
    float* conv_w[5];
    float* conv_b[5];
    float* bn_w[5];
    float* bn_b[5];
    float* compress_w;
    float* compress_b;
    float* gf_w;      /* [128,1,K,128] */
    float* gf_b;      /* [128] */
    float* action_w;
    float* action_b;
} gpp_planner_grads;

size_t gpp_planner_train_workspace_bytes(int B, int N, int K);
int gpp_planner_train_forward(const gpp_planner_weights* w, const gpp_planner_bn_state* bn, float momentum,
                              const float* x, const void* S, int s_is_f64, float* logits, void* workspace,
                              int B, int N, int K, void* stream);
int gpp_planner_train_backward(const gpp_planner_weights* w, const float* x, const void* S, int s_is_f64,
                               const float* dlogits, void* workspace, const gpp_planner_grads* g,
                               int B, int N, int K, void* stream);

/* Fused training loss (replaces the per-agent loop of agents/decentralplannerlocal.py:305-312 and its autograd graph):
 *   loss = (1/N) sum_i CrossEntropy(logits[i], argmax_a target[:, i, a])          (mean over the batch per agent)
 *   dlogits[i,b,:] = grad_scale * (softmax(logits[i,b,:]) - onehot) / (N*B)       (NULL to skip)
 *   logits dev f32 [N,B,5] (as gpp_planner_forward / _train_forward write them); target_onehot dev [B,N,5], int64
 *   (target_is_i64 != 0, the dataloader's format) or f32; loss dev f32 [1].  One launch, deterministic. */
int gpp_planner_ce_loss(const float* logits, const void* target_onehot, int target_is_i64, float* loss,
                        float* dlogits, float grad_scale, int B, int N, void* stream);

/* ------------------------------------------------------------------------------------
 * GPU-resident rollout step, B episodes in lock-step (what surrounds the forward in the reference's
 * rollout loop, agents/decentralplannerlocal.py:560-592; the reference runs it on the host, one episode
 * at a time).  All pointers are device pointers; positions are integer cells (x, y) and never leave the
 * device between steps.
 *
 * gpp_rollout_build_inputs replaces multiRobotSim.getCurrentState (utils/multirobotsim_dcenlocal.py:425-453
 * -> AgentState.toInputTensor, dataloader/statetransformer.py:82-130) and multiRobotSim.getGSO (:367-394 ->
 * computeAdjacencyMatrix :320-365, connectivity test graphTools.py:396-423):
 *   pos, goal  [B,N,2] int32      map [B,W,W] or (map_shared) [W,W] uint8, 1 = obstacle
 *   radius     [B] f64 in/out: communication radius.  grow_radius != 0 (the reference's step 0): radius is divided by
 *              1.1 once, then multiplied by 1.1 until the graph is connected, and written back.
 *   x          out f32 [B,N,3,11,11]   S out [B,N,N] f64 (s_is_f64, as the simulator emits) or f32
 *   connected  out [B] int32 or NULL
 * Bit-exact with the reference (integer window arithmetic; the GSO is IEEE float64 sqrt / divide / multiply).
 *
 * gpp_rollout_move replaces multiRobotSim.move (:562-723) incl. interRobotCollision (:462-555):
 *   logits [N,B,5] (as the planner writes them); action = first maximum (LogSoftmax + argmax, :589-591); moves into
 *   the map edge or an obstacle become "stay"; vertex conflicts and position swaps are resolved as the reference does.
 *   Where the reference draws random.choice(collided agents), the contract here is round-robin: the c-th draw of the
 *   episode picks collided[c % len] (agent order); c is choice_counter[b].
 *   pos in/out; reached / start_step / end_step [B,N] in/out (-1 = not yet); last_action [B,N] out; maxstep [B];
 *   active [B] or NULL (0 = leave the episode untouched); flags [B,3] out = {all agents had reached their goal before
 *   this move, check_moveCollision, check_predictCollsion}; currentstep = 1-based step index (:561). */
int gpp_rollout_build_inputs(const int* pos, const int* goal, const unsigned char* map, int map_shared,
                             double* radius, int grow_radius, float* x, void* S, int s_is_f64,
                             int* connected, int B, int N, int W, void* stream);
int gpp_rollout_move(const float* logits, int* pos, const int* goal, const unsigned char* map, int map_shared,
                     const int* maxstep, const int* active, int* reached, int* start_step, int* end_step,
                     int* last_action, unsigned int* choice_counter, int* flags, int currentstep, int B, int N,
                     int W, void* stream);

/* ------------------------------------------------------------------------------------
 * Per-case evaluation of the lock-step rollout (replaces the bookkeeping of the reference's test() loop,
 * agents/decentralplannerlocal.py:484-648, that surrounds the model and the simulator's move).  Device pointers,
 * int32 unless stated.
 *
 * gpp_rollout_targets replays the expert's actions (multiRobotSim.getPathTarget, utils/multirobotsim_dcenlocal.py
 * :159-229), one warp per case:
 *   target  f32 [B,N,T,5] one-hot expert actions (the test loader's format); action = first maximum of each row
 *   start, goal [B,N,2]
 *   target_start / target_end out [B,N]: first step with a non-stop action / step + 1 of the first arrival (-1 = never)
 *   targets out [B,3] = {makespanTarget = max(end) - min(start), flowtimeTarget = sum(end - start), every agent
 *   arrived}; both metrics are 0 unless every agent arrived (an agent with start == goal counts as not arrived).
 *
 * gpp_rollout_track runs once per step after gpp_rollout_move, with the same flags / active / maxstep: for every case
 * with active[b] != 0 it ORs check_moveCollision and check_predictCollsion into status[b] (:593-598), stores the move's
 * allReachGoal and currentstep, and clears active[b] when allReachGoal || currentstep >= maxstep[b] (:600-606).
 *   status [B,4] in/out = {allReachGoal of the last move, collision happened in the loop, collision predicted in the
 *   loop, step of the last move}; zero it before the first step.
 *
 * gpp_rollout_evaluate_finish runs once after the loop, one warp per case, and writes what mutliAgent_ActionPolicy
 * returns (:611-624, with checkOptimality :825-832 and the predicted metrics of move :693-715):
 *   record out [B,10] = {allReachGoal, noReachGoalbyCollsionShielding, findOptimalSolution, check_collisionFreeSol,
 *   check_CollisionPredictedinLoop, makespanPredict, makespanTarget, flowtimePredict, flowtimeTarget,
 *   num_agents_reachgoal}, from status, targets, maxstep and gpp_rollout_move's reached / start_step / end_step. */
int gpp_rollout_targets(const float* target, const int* start, const int* goal, int* target_start, int* target_end,
                        int* targets, int B, int N, int T, void* stream);
int gpp_rollout_track(const int* flags, int* active, int* status, const int* maxstep, int currentstep, int B,
                      void* stream);
int gpp_rollout_evaluate_finish(const int* status, const int* targets, const int* maxstep, const int* reached,
                                const int* start_step, const int* end_step, int* record, int B, int N, void* stream);

/* ------------------------------------------------------------------------------------
 * Training samples from expert schedules (replaces the online expert's DataTransformer, onlineExpert/
 * DataTransformer_local_onlineExpert.py:96-305, and the train loader's per-sample scipy.io.loadmat,
 * dataloader/Dataloader_dcplocal_notTF_onlineExpert.py:142-157).  Device pointers, int32 unless stated.  C cases
 * stored as one flat row array: case c has T_c = makespan + 1 rows case_first_row[c] .. case_first_row[c+1] - 1 of
 *   pos  [R,N,2] agent cells per step, R = sum of T_c (row t of a case: the expert's cell at step t, the goal after its
 *        plan ends)
 *
 * gpp_dataset_prepare computes each case's communication threshold as computeAdjacencyMatrix(states, r0) does: start
 * at r0, multiply by 1.1 (float64) while a step is disconnected, never reset between steps; the final value is used
 * for every step.  case_first_row [C+1] (absolute row indices into pos); radius out f64 [C].  One CTA per case.
 *
 * gpp_dataset_batch builds B training samples in one launch, one CTA per sample:
 *   row_case [R]; goal [C,N,2]; map [C,W,W] or (map_shared) [W,W] uint8, 1 = obstacle; radius [C] from prepare;
 *   rows int64 [B] sample (= row) indices, a row outside [0, R) gives an all-zero sample;
 *   x out f32 [B,N,3,11,11] (toSeqInputTensor's field of view); S out f32 [B,N,N] (the float32 cast of the float64
 *   D^-1/2 A D^-1/2 with A = pdist < radius, zero diagonal); target out int64 [B,N,5] one-hot index of the move to the
 *   next row (to the goal on a case's last row) in delta = up, left, down, right, stop.
 * Both support 2 <= N <= 64 and square maps with W*W <= 327,680 cells, else GPP_ERR_UNSUPPORTED. */
int gpp_dataset_prepare(const int* pos, const int* case_first_row, double r0, double* radius, int C, int N,
                        void* stream);
int gpp_dataset_batch(const int* pos, const int* row_case, const int* case_first_row, const int* goal,
                      const unsigned char* map, int map_shared, const double* radius, const long long* rows, float* x,
                      float* S, long long* target, int B, int N, int W, int R, void* stream);

/* Asynchronous variant for pipelined rollouts over INDEPENDENT episode batches: stages the inputs on a copy stream,
 * enqueues the forward on one of the planner's four compute streams (tickets rotate over them, so the feature kernel of
 * one batch runs next to the kernels of the batches before it on the SMs they leave idle) and returns at once with a completion ticket; the
 * host buffers MUST be pinned and must stay untouched until gpp_planner_wait(ticket) returns.  Consecutive tickets may
 * complete in either order -- wait for the ticket whose logits are needed; at most 16 tickets may be outstanding. */
int gpp_planner_forward_host_async(gpp_planner* p, const float* x_host, const void* S_host,
                                   int s_is_f64, float* logits_host, int B, int N,
                                   unsigned long long* ticket);
int gpp_planner_wait(gpp_planner* p, unsigned long long ticket);

/* The same pipelining for DEVICE tensors (a driver advancing several independent episode batches whose inputs are produced on
 * the GPU): x / S must be complete in `stream` order at the time of the call (an event is recorded there), the forward
 * runs on the next compute lane, and the logits (device memory, [N][B][5]) may be consumed after
 * gpp_planner_join(p, ticket, consumer_stream) -- a device-side wait, the host does not block -- or after
 * gpp_planner_wait(ticket).  x, S and logits must stay untouched until then; tickets share the numbering and the limit of
 * 16 outstanding calls with gpp_planner_forward_host_async.  Replaces a loop of `model.addGSO(S); model(x)` calls
 * (/root/reference/agents/decentralplannerlocal.py:576-588) over independent batches. */
int gpp_planner_forward_async(gpp_planner* p, const float* x, const void* S, int s_is_f64, float* logits, int B, int N,
                              void* stream, unsigned long long* ticket);
int gpp_planner_join(gpp_planner* p, unsigned long long ticket, void* stream);

/* Which graph-filter kernel the planner uses: 0 = automatic (tensor cores once B*N >= 4096 node
 * rows), 1 = CUDA-core fp32 kernel (gf_fwd_kernel), 2 = tcgen05 3xTF32 kernel (gf_fwd_tc_kernel),
 * 3 = tcgen05 CTA-pair fp16-split kernel (gf_fwd_pair_kernel).  GPP_ERR_UNSUPPORTED at forward
 * time if N / K are outside the requested kernel's envelope. */
int gpp_planner_set_graph_filter_mode(gpp_planner* p, int mode);

/* Which feature-extractor (CNN + compress MLP) kernel the planner uses: 0 = automatic (currently always the
 * CUDA-core kernel, the faster one at every measured size), 1 = CUDA-core fp32 kernel (feature_kernel),
 * 2 = tcgen05 3xTF32 implicit-GEMM kernel (feature_tc_kernel). */
int gpp_planner_set_feature_mode(gpp_planner* p, int mode);

/* Per-kernel device timing for the roofline report: when enabled, gpp_planner_forward records
 * CUDA events before / between / after its two kernels on the launching stream (at most 8192
 * steps are kept).  gpp_planner_get_profile synchronises on the recorded events, returns the
 * summed durations in milliseconds and the number of steps they cover, and clears the log. */
int gpp_planner_set_profiling(gpp_planner* p, int enable);
int gpp_planner_get_profile(gpp_planner* p, double* feature_ms, double* graph_filter_ms, int* steps);

/* Number of kernels of this library launched by this process (any thread) since
 * the last reset (bench.py's gpu_launches claim is read from here, not guessed). */
unsigned long long gpp_launch_count(void);
void gpp_reset_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* GNNPP_B200_H */
