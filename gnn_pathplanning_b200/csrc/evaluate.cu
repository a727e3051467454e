// Per-case evaluation of B lock-step rollouts (the reference's test() loop, agents/decentralplannerlocal.py:484-648): what
// the reference computes on the HOST, one case at a time, around its rollout --
//
//   multiRobotSim.getPathTarget   utils/multirobotsim_dcenlocal.py:159-229   expert makespan / flowtime
//   mutliAgent_ActionPolicy       agents/decentralplannerlocal.py:593-624    loop flags, end-of-case branches
//   multiRobotSim.move (metrics)  utils/multirobotsim_dcenlocal.py:693-715   predicted makespan / flowtime
//   multiRobotSim.checkOptimality :825-832
//
// rollout_targets_kernel replays the expert's actions once per case, rollout_track_kernel folds each step's move flags
// into per-case loop state (and retires finished cases), rollout_finish_kernel writes the per-case record the
// reference hands to MonitoringMultiAgentPerformance.update (utils/metrics.py:104-152).  All integer arithmetic.
#include <climits>

#include "common.cuh"

namespace gpp {

constexpr int EV_MAX_N = 64;

// status[b][*] as written by rollout_track_kernel
enum { EV_ALL_REACH = 0, EV_COLLISION_HAPPENED = 1, EV_COLLISION_PREDICTED = 2, EV_FINAL_STEP = 3, EV_STATUS = 4 };
// targets[b][*] as written by rollout_targets_kernel
enum { EV_MAKESPAN_TARGET = 0, EV_FLOWTIME_TARGET = 1, EV_TARGET_ALL_REACH = 2, EV_TARGETS = 3 };
// record[b][*]: the fields of mutliAgent_ActionPolicy's result, in the order of metrics.py:106
enum {
    EV_R_ALL_REACH = 0, EV_R_NO_REACH_SH, EV_R_OPTIMAL, EV_R_COLLISION_FREE, EV_R_COLLISION_PREDICTED,
    EV_R_MP_PREDICT, EV_R_MP_TARGET, EV_R_FT_PREDICT, EV_R_FT_TARGET, EV_R_NUM_REACH, EV_RECORD
};

__device__ __forceinline__ int ev_warp_max(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ int ev_warp_min(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ int ev_warp_sum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// One warp per case, lane = agent (agents lane and lane + 32 for N > 32).  getPathTarget (:183-205) per agent: the
// action of step t is the first maximum of target[t] (torch.max(., 1)[1], :112); the start step is the first step with
// a non-stop action, the end step is step + 1 of the first arrival on the goal.  The expert path is pure arithmetic --
// the reference checks neither the map nor other agents here.  Then (:209-225) makespan = max(end) - min(start),
// flowtime = sum(end - start), computed only when every agent arrived (else both stay 0, :89-90).
__global__ void __launch_bounds__(128) rollout_targets_kernel(const float* __restrict__ target, const int* __restrict__ start,
                                                              const int* __restrict__ goal, int* __restrict__ tstart,
                                                              int* __restrict__ tend, int* __restrict__ out, int B, int N,
                                                              int T) {
    const int b = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (b >= B) return;
    int hi = INT_MIN, lo = INT_MAX, sum = 0, all = 1;
    for (int i = lane; i < N; i += 32) {
        const size_t ai = (size_t)b * N + i;
        int x = start[2 * ai], y = start[2 * ai + 1];
        const int gx = goal[2 * ai], gy = goal[2 * ai + 1];
        int s = -1, e = -1;
        const float* tp = target + ai * T * 5;
        for (int t = 0; t < T && e < 0; ++t) {
            const float* r = tp + (size_t)t * 5;
            int key = 0;
            float best = r[0];
#pragma unroll
            for (int q = 1; q < 5; ++q)
                if (r[q] > best) { best = r[q]; key = q; }
            if (key != 4 && s < 0) s = t;
            x += key == 0 ? -1 : key == 2 ? 1 : 0;       // multirobotsim_dcenlocal.py:21-25 up, left, down, right, stop
            y += key == 1 ? -1 : key == 3 ? 1 : 0;
            if (x == gx && y == gy) e = t + 1;
        }
        tstart[ai] = s;
        tend[ai] = e;
        // an agent that never moved but "arrives" (start == goal) has no start step: the reference raises TypeError
        // at :218; it is reported as not arrived
        all &= (e >= 0 && s >= 0);
        hi = max(hi, e);
        lo = min(lo, s);
        sum += e - s;
    }
    all = __all_sync(0xffffffffu, all);
    hi = ev_warp_max(hi);
    lo = ev_warp_min(lo);
    sum = ev_warp_sum(sum);
    if (lane == 0) {
        out[EV_TARGETS * b + EV_MAKESPAN_TARGET] = all ? hi - lo : 0;
        out[EV_TARGETS * b + EV_FLOWTIME_TARGET] = all ? sum : 0;
        out[EV_TARGETS * b + EV_TARGET_ALL_REACH] = all;
    }
}

// After each gpp_rollout_move: for every case that was active for that move, the loop body of :593-606.
__global__ void __launch_bounds__(256) rollout_track_kernel(const int* __restrict__ flags, int* __restrict__ active,
                                                            int* __restrict__ status, const int* __restrict__ maxstep,
                                                            int currentstep, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B || !active[b]) return;
    int* st = status + (size_t)EV_STATUS * b;
    const int all_reach = flags[3 * b];
    st[EV_ALL_REACH] = all_reach;
    st[EV_COLLISION_HAPPENED] |= flags[3 * b + 1];          // check_CollisionHappenedinLoop (:593-594)
    st[EV_COLLISION_PREDICTED] |= flags[3 * b + 2];         // check_CollisionPredictedinLoop (:597-598)
    st[EV_FINAL_STEP] = currentstep;
    if (all_reach || currentstep >= maxstep[b]) active[b] = 0;      // break (:600-606)
}

// One warp per case after the loop: the branches of :611-624 and the predicted metrics of :693-715 over the state the
// final move left (every agent has an end step then: it arrived, or the final move was at maxstep, :686-691).
__global__ void __launch_bounds__(128) rollout_finish_kernel(const int* __restrict__ status, const int* __restrict__ targets,
                                                             const int* __restrict__ maxstep, const int* __restrict__ reached,
                                                             const int* __restrict__ start_step,
                                                             const int* __restrict__ end_step, int* __restrict__ record,
                                                             int B, int N) {
    const int b = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (b >= B) return;
    int hi = INT_MIN, lo = INT_MAX, sum = 0, nreach = 0;
    for (int i = lane; i < N; i += 32) {
        const size_t ai = (size_t)b * N + i;
        const int s = start_step[ai], e = end_step[ai];
        hi = max(hi, e);
        lo = min(lo, s);
        sum += e - s;
        nreach += reached[ai] != 0;
    }
    hi = ev_warp_max(hi);
    lo = ev_warp_min(lo);
    sum = ev_warp_sum(sum);
    nreach = ev_warp_sum(nreach);
    if (lane != 0) return;
    const int* st = status + (size_t)EV_STATUS * b;
    const int ms = maxstep[b];
    const bool all_reach = st[EV_ALL_REACH] != 0, happened = st[EV_COLLISION_HAPPENED] != 0;
    const bool predicted = st[EV_COLLISION_PREDICTED] != 0, at_maxstep = st[EV_FINAL_STEP] >= ms;
    const int mp_target = targets[EV_TARGETS * b + EV_MAKESPAN_TARGET], ft_target = targets[EV_TARGETS * b + EV_FLOWTIME_TARGET];
    // the metrics the case reports are the ones getOptimalityMetrics returned before the loop (:555; setup :91-92)
    // unless checkOptimality is called after it (:614, :619, :622)
    int mp = ms, ft = ms * N, optimal = 0;
    const bool collision_free = all_reach && !happened;
    if (collision_free) {                                              // :611-614  checkOptimality(True)
        mp = hi - lo;
        ft = sum;
        optimal = mp <= mp_target && ft <= ft_target;
    }
    if (at_maxstep) {                                                  // :618-619  checkOptimality(False)
        mp = hi - lo;
        ft = sum;
        optimal = 0;
    }
    int* r = record + (size_t)EV_RECORD * b;
    r[EV_R_ALL_REACH] = all_reach;
    r[EV_R_NO_REACH_SH] = at_maxstep && !all_reach && predicted && !happened;     // :621-624
    r[EV_R_OPTIMAL] = optimal;
    r[EV_R_COLLISION_FREE] = collision_free;
    r[EV_R_COLLISION_PREDICTED] = predicted;
    r[EV_R_MP_PREDICT] = mp;
    r[EV_R_MP_TARGET] = mp_target;
    r[EV_R_FT_PREDICT] = ft;
    r[EV_R_FT_TARGET] = ft_target;
    r[EV_R_NUM_REACH] = nreach;
}

}  // namespace gpp

using namespace gpp;

extern "C" int gpp_rollout_targets(const float* target, const int* start, const int* goal, int* target_start,
                                   int* target_end, int* targets, int B, int N, int T, void* stream) {
    GPP_REQUIRE(target && start && goal && target_start && target_end && targets, GPP_ERR_INVALID,
                "rollout_targets: null pointer");
    GPP_REQUIRE(B >= 0 && N >= 1 && T >= 1, GPP_ERR_INVALID, "rollout_targets: bad sizes B=%d N=%d T=%d", B, N, T);
    GPP_REQUIRE(N <= EV_MAX_N, GPP_ERR_UNSUPPORTED, "rollout_targets: N=%d > %d agents", N, EV_MAX_N);
    if (B == 0) return GPP_OK;
    rollout_targets_kernel<<<(B + 3) / 4, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        target, start, goal, target_start, target_end, targets, B, N, T);
    GPP_LAUNCH_CHECK();
    return GPP_OK;
}

extern "C" int gpp_rollout_track(const int* flags, int* active, int* status, const int* maxstep, int currentstep, int B,
                                 void* stream) {
    GPP_REQUIRE(flags && active && status && maxstep, GPP_ERR_INVALID, "rollout_track: null pointer");
    GPP_REQUIRE(B >= 0, GPP_ERR_INVALID, "rollout_track: bad size B=%d", B);
    if (B == 0) return GPP_OK;
    rollout_track_kernel<<<(B + 255) / 256, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(flags, active, status, maxstep,
                                                                                            currentstep, B);
    GPP_LAUNCH_CHECK();
    return GPP_OK;
}

extern "C" int gpp_rollout_evaluate_finish(const int* status, const int* targets, const int* maxstep, const int* reached,
                                           const int* start_step, const int* end_step, int* record, int B, int N,
                                           void* stream) {
    GPP_REQUIRE(status && targets && maxstep && reached && start_step && end_step && record, GPP_ERR_INVALID,
                "rollout_evaluate_finish: null pointer");
    GPP_REQUIRE(B >= 0 && N >= 1, GPP_ERR_INVALID, "rollout_evaluate_finish: bad sizes B=%d N=%d", B, N);
    GPP_REQUIRE(N <= EV_MAX_N, GPP_ERR_UNSUPPORTED, "rollout_evaluate_finish: N=%d > %d agents", N, EV_MAX_N);
    if (B == 0) return GPP_OK;
    rollout_finish_kernel<<<(B + 3) / 4, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        status, targets, maxstep, reached, start_step, end_step, record, B, N);
    GPP_LAUNCH_CHECK();
    return GPP_OK;
}
