// GPU-resident rollout step for B episodes in lock-step (SURVEY.md section 8 rows f1 / f2): what surrounds the planner's
// forward in the reference's rollout loop (agents/decentralplannerlocal.py:560-592), per step, on the HOST, one episode at
// a time, with python dicts of tensors:
//
//   getCurrentState  utils/multirobotsim_dcenlocal.py:425-453 -> AgentState.toInputTensor dataloader/statetransformer.py:82-130
//   getGSO           utils/multirobotsim_dcenlocal.py:367-394 -> computeAdjacencyMatrix :320-365, isConnected graphTools.py:396-423
//   move             utils/multirobotsim_dcenlocal.py:562-723 -> interRobotCollision :462-555
//
// Here: rollout_inputs_kernel builds the [B,N,3,11,11] field-of-view tensor and the [B,N,N] graph shift operator from
// integer agent positions that never leave the device; rollout_move_kernel turns the planner's logits into moves with the
// reference's edge / obstacle / inter-robot collision shielding.  Both are integer / IEEE-double restatements of the
// reference's arithmetic: bit-exact by construction (tests/test_gpu_rollout.py).
#include "step_inputs.cuh"

namespace gpp {

struct RoInputArgs {
    const int* pos;        // [B][N][2] current agent cells (x, y)
    const int* goal;       // [B][N][2]
    const unsigned char* map;   // [B][W][W] or [W][W] (map_shared) obstacle map, 1 = obstacle
    double* radius;        // [B] communication radius (updated at step 0 when grow_radius)
    float* x;              // [B][N][3][11][11] out
    void* S;               // [B][N][N] out (f32 / f64)
    int* connected;        // [B] out or null: was the communication graph connected
    int B, N, W, map_shared, grow_radius, s_is_f64;
};

// One CTA per episode.
__global__ void __launch_bounds__(128) rollout_inputs_kernel(const RoInputArgs a) {
    __shared__ unsigned long long adj[RO_MAX_N];
    __shared__ int px[RO_MAX_N], py[RO_MAX_N];
    __shared__ double dinv[RO_MAX_N];
    __shared__ double rad;
    __shared__ int is_conn;
    extern __shared__ unsigned int occ_bits[];          // ceil(W*W / 32) words: cells occupied by an agent
    const int b = blockIdx.x, tid = threadIdx.x, N = a.N, W = a.W;
    const int* pos = a.pos + (size_t)b * N * 2;
    const int* goal = a.goal + (size_t)b * N * 2;
    const unsigned char* map = a.map + (a.map_shared ? 0 : (size_t)b * W * W);
    for (int i = tid; i < (W * W + 31) / 32; i += blockDim.x) occ_bits[i] = 0u;
    if (tid < N) {
        px[tid] = pos[2 * tid];
        py[tid] = pos[2 * tid + 1];
    }
    if (tid == 0) {
        // computeAdjacencyMatrix :336-340: at step 0 the radius is divided by 1.1 once and multiplied by 1.1 until the graph
        // is connected (the first pass therefore uses r / 1.1 * 1.1, not r); later steps keep the radius found then
        rad = a.grow_radius ? a.radius[b] / 1.1 : a.radius[b];
    }
    __syncthreads();
    if (tid < N) atomicOr(&occ_bits[(px[tid] * W + py[tid]) >> 5], 1u << ((px[tid] * W + py[tid]) & 31));
    // ---- adjacency (pdist < r, zero diagonal) + connectivity, repeated with a 10 % larger radius at step 0
    for (int guard = 0; guard < 4096; ++guard) {
        if (tid == 0 && a.grow_radius) rad = rad * 1.1;
        __syncthreads();
        if (tid < N) adj[tid] = ro_adjacency_row(tid, N, px, py, rad);
        __syncthreads();
        if (tid == 0) is_conn = ro_is_connected(adj, N);
        __syncthreads();
        if (!a.grow_radius || is_conn) break;
    }
    if (tid == 0) {
        if (a.grow_radius) a.radius[b] = rad;
        if (a.connected) a.connected[b] = is_conn;
    }
    // ---- D^-1/2 A D^-1/2 with the zero-degree guard (:341-348), float64 as the reference
    if (tid < N) dinv[tid] = ro_deg_inv_sqrt(adj[tid]);
    __syncthreads();
    for (int e = tid; e < N * N; e += blockDim.x) {
        const int i = e / N, j = e - i * N;
        const double v = ro_gso_entry(adj, dinv, i, j);
        if (a.s_is_f64) reinterpret_cast<double*>(a.S)[(size_t)b * N * N + e] = v;
        else reinterpret_cast<float*>(a.S)[(size_t)b * N * N + e] = (float)v;
    }
    // ---- field-of-view tensor (statetransformer.py:82-130)
    float* xo = a.x + (size_t)b * N * RO_FOV_ELEMS;
    for (int e = tid; e < N * RO_FOV_ELEMS; e += blockDim.x) xo[e] = ro_fov_value(e, px, py, goal, map, occ_bits, W);
}

struct RoMoveArgs {
    const float* logits;   // [N][B][5]
    int* pos;              // [B][N][2] in / out
    const int* goal;       // [B][N][2]
    const unsigned char* map;
    const int* maxstep;    // [B]
    const int* active;     // [B] or null: episodes with 0 are left untouched
    int* reached;          // [B][N] in / out  (count_reachgoal)
    int* start_step;       // [B][N] in / out, -1 = None
    int* end_step;         // [B][N] in / out, -1 = None
    int* last_action;      // [B][N] out: the action each agent ended up taking this step (4 = stay)
    unsigned int* choice_counter;   // [B] in / out: number of "who may move" choices made so far in the episode
    int* flags;            // [B][3] out: allReachGoal (before the move), check_moveCollision, check_predictCollsion
    int B, N, W, map_shared, currentstep;
};

// interRobotCollision (:462-555) for one episode; `cur` = positions before the step, `nxt` = proposed, `act` = last action.
// Where the reference draws random.choice(collided_agents), this library's contract is round-robin: the c-th draw of
// the episode picks collided[c % len(collided)] (collided in agent order); the counter lives in the episode state.
__device__ bool ro_inter_robot_collision(int N, const int* cx, const int* cy, int* nx, int* ny, int* act, unsigned int& counter) {
    bool collision = false;
    int ox[RO_MAX_N], oy[RO_MAX_N], lx[RO_MAX_N], ly[RO_MAX_N];
    for (int i = 0; i < N; ++i) {            // allagents_pos (never updated) and list_pos (updated as agents are stopped)
        ox[i] = lx[i] = nx[i];
        oy[i] = ly[i] = ny[i];
    }
    for (int i = 0; i < N; ++i) {
        const int qx = lx[i], qy = ly[i];
        int count = 0;
        for (int j = 0; j < N; ++j) count += (lx[j] == qx && ly[j] == qy);
        if (count > 1) {
            collision = true;
            int coll[RO_MAX_N], nc = 0;
            for (int j = 0; j < N; ++j)
                if (ox[j] == qx && oy[j] == qy) coll[nc++] = j;
            // (nc can be 0: `pos` may be an updated entry nobody proposed originally; random.choice([]) raises
            //  IndexError in the reference -- with nc == 0 nothing below executes and no draw is consumed)
            int mover = -1;
            if (nc > 0) {
                mover = coll[counter % (unsigned int)nc];
                ++counter;
            }
            for (int t = 0; t < nc; ++t) {
                const int name = coll[t];
                if (act[name] == 4) {
                    for (int t2 = 0; t2 < nc; ++t2) {       // one of them has stopped: every collided agent stays
                        const int n2 = coll[t2];
                        act[n2] = 4;
                        nx[n2] = cx[n2]; ny[n2] = cy[n2];
                        lx[n2] = nx[n2]; ly[n2] = ny[n2];
                    }
                } else if (name != mover) {
                    act[name] = 4;
                    nx[name] = cx[name]; ny[name] = cy[name];
                    lx[name] = nx[name]; ly[name] = ny[name];
                }
            }
        }
    }
    // position swaps: two agents exchanging cells both stay (:516-553); list_nextpos is a snapshot
    int sx[RO_MAX_N], sy[RO_MAX_N];
    for (int i = 0; i < N; ++i) { sx[i] = nx[i]; sy[i] = ny[i]; }
    for (int i = 0; i < N; ++i) {
        int sw = -1;
        for (int j = 0; j < N; ++j)
            if (sx[j] == cx[i] && sy[j] == cy[i]) { sw = j; break; }      // list.index: first match
        if (sw >= 0 && sw != i && cx[sw] == nx[i] && cy[sw] == ny[i]) {
            nx[i] = cx[i]; ny[i] = cy[i];
            nx[sw] = cx[sw]; ny[sw] = cy[sw];
            act[i] = 4; act[sw] = 4;
            collision = true;
        }
    }
    return collision;
}

// One thread per episode: the reference's algorithm is sequential over agents (later agents see earlier decisions).
__global__ void __launch_bounds__(64) rollout_move_kernel(const RoMoveArgs a) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.B) return;
    if (a.active && !a.active[b]) return;
    const int N = a.N, W = a.W, B = a.B, step = a.currentstep, maxstep = a.maxstep[b];
    const unsigned char* map = a.map + (a.map_shared ? 0 : (size_t)b * W * W);
    int* pos = a.pos + (size_t)b * N * 2;
    const int* goal = a.goal + (size_t)b * N * 2;
    int* reached = a.reached + (size_t)b * N;
    int* sst = a.start_step + (size_t)b * N;
    int* est = a.end_step + (size_t)b * N;
    bool all_reach = true;
    for (int i = 0; i < N; ++i) all_reach = all_reach && reached[i] != 0;
    bool predict_collision = false, move_collision = false;
    if (!all_reach || step < maxstep) {                         // :570
        int cx[RO_MAX_N], cy[RO_MAX_N], nx[RO_MAX_N], ny[RO_MAX_N], act[RO_MAX_N];
        const int ddx[5] = {-1, 0, 1, 0, 0}, ddy[5] = {0, -1, 0, 1, 0};     // :21-25 up, left, down, right, stop
        for (int i = 0; i < N; ++i) {
            cx[i] = pos[2 * i]; cy[i] = pos[2 * i + 1];
            const float* lp = a.logits + ((size_t)i * B + b) * 5;
            int key = 0;                                          // argmax(LogSoftmax(.)) = first maximum of the logits (:589-591)
            float best = lp[0];
            for (int q = 1; q < 5; ++q)
                if (lp[q] > best) { best = lp[q]; key = q; }
            if (key != 4 && sst[i] < 0) sst[i] = step - 1;        // :596-600
            const int tx = cx[i] + ddx[key], ty = cy[i] + ddy[key];
            const bool edge = tx >= W || tx < 0 || ty >= W || ty < 0;          // reachEdge :305-318
            const bool obstacle = !edge && map[tx * W + ty] == 1;              // reachObstacle :281-303
            if (edge || obstacle) {
                predict_collision = true;
                act[i] = 4;
                nx[i] = cx[i]; ny[i] = cy[i];
            } else {
                act[i] = key;
                nx[i] = tx; ny[i] = ty;
            }
        }
        unsigned int counter = a.choice_counter[b];
        bool detect = ro_inter_robot_collision(N, cx, cy, nx, ny, act, counter);
        for (int r = 0; r < N; ++r) {                              // :652-660
            if (!detect) break;
            detect = ro_inter_robot_collision(N, cx, cy, nx, ny, act, counter);
            predict_collision = true;
        }
        move_collision = ro_inter_robot_collision(N, cx, cy, nx, ny, act, counter);     // :662
        a.choice_counter[b] = counter;
        for (int i = 0; i < N; ++i) {
            pos[2 * i] = nx[i]; pos[2 * i + 1] = ny[i];
            a.last_action[(size_t)b * N + i] = act[i];
            if (nx[i] == goal[2 * i] && ny[i] == goal[2 * i + 1] && !reached[i]) {
                reached[i] = 1;
                est[i] = step;
            }
            if (step >= maxstep && !reached[i]) {
                est[i] = step;
                if (sst[i] < 0) sst[i] = 0;
            }
        }
    }
    a.flags[3 * b] = all_reach;
    a.flags[3 * b + 1] = move_collision;
    a.flags[3 * b + 2] = predict_collision;
}

// ---------------------------------------------------------------------------------------------------------------------
// Warp-per-episode version for N <= 32 (lane = agent, state in registers).  interRobotCollision visits the agents in
// order and later visits see earlier decisions, so the visiting loop stays sequential; what happens inside one visit
// does not depend on the order in which the collided agents are handled (if any of them had already stopped they all
// stop, otherwise all but the mover stop), so it is one ballot.  70 -> ~8 us per step of 256 episodes x 10 agents.
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool ro_collision_warp(int N, int lane, int cx, int cy, int& nx, int& ny, int& act, unsigned int& counter) {
    const unsigned int FULL = 0xffffffffu;
    const bool in = lane < N;
    bool collision = false;
    const int ox = nx, oy = ny;          // allagents_pos (never updated)
    int lx = nx, ly = ny;                // list_pos (updated as agents are stopped)
    for (int i = 0; i < N; ++i) {
        const int qx = __shfl_sync(FULL, lx, i), qy = __shfl_sync(FULL, ly, i);
        const unsigned int same = __ballot_sync(FULL, in && lx == qx && ly == qy);
        if (__popc(same) > 1) {
            collision = true;
            const unsigned int coll = __ballot_sync(FULL, in && ox == qx && oy == qy);
            const int nc = __popc(coll);
            int mover = -1;
            if (nc > 0) {
                unsigned int rest = coll;                        // the (counter mod nc)-th collided agent, in agent order
                for (unsigned int r = counter % (unsigned int)nc; r > 0; --r) rest &= rest - 1;
                mover = __ffs(rest) - 1;
                ++counter;
            }
            const bool mine = (coll >> lane) & 1u;
            const bool any_stopped = __ballot_sync(FULL, mine && act == 4) != 0;
            if (mine && (any_stopped || lane != mover)) {
                act = 4;
                nx = cx; ny = cy;
                lx = nx; ly = ny;
            }
        }
    }
    // position swaps: two agents exchanging cells both stay; the searched list is a snapshot
    const int sx = nx, sy = ny;
    for (int i = 0; i < N; ++i) {
        const int cxi = __shfl_sync(FULL, cx, i), cyi = __shfl_sync(FULL, cy, i);
        const int nxi = __shfl_sync(FULL, nx, i), nyi = __shfl_sync(FULL, ny, i);
        const unsigned int m = __ballot_sync(FULL, in && sx == cxi && sy == cyi);
        const int sw = m ? (__ffs(m) - 1) : -1;                    // list.index: first match
        const int swc = sw >= 0 ? sw : 0;
        const int cxs = __shfl_sync(FULL, cx, swc), cys = __shfl_sync(FULL, cy, swc);
        if (sw >= 0 && sw != i && cxs == nxi && cys == nyi) {
            if (lane == i || lane == sw) { nx = cx; ny = cy; act = 4; }
            collision = true;
        }
    }
    return collision;
}

__global__ void __launch_bounds__(128) rollout_move_warp_kernel(const RoMoveArgs a) {
    const unsigned int FULL = 0xffffffffu;
    const int b = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (b >= a.B) return;
    if (a.active && !a.active[b]) return;
    const int N = a.N, W = a.W, B = a.B, step = a.currentstep, maxstep = a.maxstep[b];
    const bool in = lane < N;
    const unsigned char* map = a.map + (a.map_shared ? 0 : (size_t)b * W * W);
    int* pos = a.pos + (size_t)b * N * 2;
    const int* goal = a.goal + (size_t)b * N * 2;
    int reached = in ? a.reached[(size_t)b * N + lane] : 1;
    int sst = in ? a.start_step[(size_t)b * N + lane] : 0;
    const bool all_reach = __all_sync(FULL, reached != 0);
    bool predict_collision = false, move_collision = false;
    if (!all_reach || step < maxstep) {                         // :570
        int cx = 0, cy = 0, nx = -1 - lane, ny = -1, act = 4;   // lanes without an agent sit on distinct off-map cells
        bool blocked = false;
        if (in) {
            cx = pos[2 * lane]; cy = pos[2 * lane + 1];
            const float* lp = a.logits + ((size_t)lane * B + b) * 5;
            int key = 0;                                          // first maximum of the logits (:589-591)
            float best = lp[0];
#pragma unroll
            for (int q = 1; q < 5; ++q) {
                const float v = lp[q];
                if (v > best) { best = v; key = q; }
            }
            if (key != 4 && sst < 0) sst = step - 1;              // :596-600
            const int tx = cx + (key == 0 ? -1 : key == 2 ? 1 : 0), ty = cy + (key == 1 ? -1 : key == 3 ? 1 : 0);
            const bool edge = tx >= W || tx < 0 || ty >= W || ty < 0;
            const bool obstacle = !edge && map[tx * W + ty] == 1;
            blocked = edge || obstacle;
            act = blocked ? 4 : key;
            nx = blocked ? cx : tx; ny = blocked ? cy : ty;
        }
        predict_collision = __any_sync(FULL, blocked);
        unsigned int counter = a.choice_counter[b];
        bool detect = ro_collision_warp(N, lane, cx, cy, nx, ny, act, counter);
        for (int r = 0; r < N; ++r) {                              // :652-660
            if (!detect) break;
            detect = ro_collision_warp(N, lane, cx, cy, nx, ny, act, counter);
            predict_collision = true;
        }
        move_collision = ro_collision_warp(N, lane, cx, cy, nx, ny, act, counter);     // :662
        if (lane == 0) a.choice_counter[b] = counter;
        if (in) {
            pos[2 * lane] = nx; pos[2 * lane + 1] = ny;
            a.last_action[(size_t)b * N + lane] = act;
            int est = a.end_step[(size_t)b * N + lane];
            if (nx == goal[2 * lane] && ny == goal[2 * lane + 1] && !reached) {
                reached = 1;
                est = step;
            }
            if (step >= maxstep && !reached) {
                est = step;
                if (sst < 0) sst = 0;
            }
            a.reached[(size_t)b * N + lane] = reached;
            a.start_step[(size_t)b * N + lane] = sst;
            a.end_step[(size_t)b * N + lane] = est;
        }
    }
    if (lane == 0) {
        a.flags[3 * b] = all_reach;
        a.flags[3 * b + 1] = move_collision;
        a.flags[3 * b + 2] = predict_collision;
    }
}

}  // namespace gpp

using namespace gpp;

extern "C" int gpp_rollout_build_inputs(const int* pos, const int* goal, const unsigned char* map, int map_shared,
                                        double* radius, int grow_radius, float* x, void* S, int s_is_f64,
                                        int* connected, int B, int N, int W, void* stream) {
    GPP_REQUIRE(pos && goal && map && radius && x && S, GPP_ERR_INVALID, "rollout_build_inputs: null pointer");
    GPP_REQUIRE(B >= 0 && N >= 1 && W >= 1, GPP_ERR_INVALID, "rollout_build_inputs: bad sizes B=%d N=%d W=%d", B, N, W);
    GPP_REQUIRE(N <= RO_MAX_N, GPP_ERR_UNSUPPORTED, "rollout_build_inputs: N=%d > %d agents", N, RO_MAX_N);
    if (B == 0) return GPP_OK;
    const size_t smem = sizeof(unsigned int) * ((size_t)(W * W + 31) / 32);
    GPP_REQUIRE(smem <= 40 * 1024, GPP_ERR_UNSUPPORTED, "rollout_build_inputs: map %dx%d too large", W, W);
    RoInputArgs a;
    a.pos = pos; a.goal = goal; a.map = map; a.radius = radius; a.x = x; a.S = S; a.connected = connected;
    a.B = B; a.N = N; a.W = W; a.map_shared = map_shared; a.grow_radius = grow_radius; a.s_is_f64 = s_is_f64;
    rollout_inputs_kernel<<<B, 128, smem, reinterpret_cast<cudaStream_t>(stream)>>>(a);
    GPP_LAUNCH_CHECK();
    return GPP_OK;
}

extern "C" int gpp_rollout_move(const float* logits, int* pos, const int* goal, const unsigned char* map, int map_shared,
                                const int* maxstep, const int* active, int* reached, int* start_step, int* end_step,
                                int* last_action, unsigned int* choice_counter, int* flags, int currentstep, int B, int N,
                                int W, void* stream) {
    GPP_REQUIRE(logits && pos && goal && map && maxstep && reached && start_step && end_step && last_action &&
                    choice_counter && flags,
                GPP_ERR_INVALID, "rollout_move: null pointer");
    GPP_REQUIRE(B >= 0 && N >= 1 && W >= 1, GPP_ERR_INVALID, "rollout_move: bad sizes B=%d N=%d W=%d", B, N, W);
    GPP_REQUIRE(N <= RO_MAX_N, GPP_ERR_UNSUPPORTED, "rollout_move: N=%d > %d agents", N, RO_MAX_N);
    if (B == 0) return GPP_OK;
    RoMoveArgs a;
    a.logits = logits; a.pos = pos; a.goal = goal; a.map = map; a.maxstep = maxstep; a.active = active;
    a.reached = reached; a.start_step = start_step; a.end_step = end_step; a.last_action = last_action;
    a.choice_counter = choice_counter; a.flags = flags;
    a.B = B; a.N = N; a.W = W; a.map_shared = map_shared; a.currentstep = currentstep;
    if (N <= 32)
        rollout_move_warp_kernel<<<(B + 3) / 4, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(a);
    else
        rollout_move_kernel<<<(B + 63) / 64, 64, 0, reinterpret_cast<cudaStream_t>(stream)>>>(a);
    GPP_LAUNCH_CHECK();
    return GPP_OK;
}
