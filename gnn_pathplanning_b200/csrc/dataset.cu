// Training samples built on the device from expert schedules (SURVEY.md section 8 row f3): what the reference's
// online-expert DataTransformer writes into one .mat file per case and its train loader reads back one sample at a time
// with scipy.io.loadmat --
//
//   obtainSchedule                      onlineExpert/DataTransformer_local_onlineExpert.py:154-196  positions, targets
//   computeAdjacencyMatrix(states, 5)   :256-305  one threshold grown over the whole schedule, then every step's GSO
//   AgentState.toSeqInputTensor         dataloader/statetransformer.py:133-187  per-step field of view
//   CreateDataset.load_train_data       dataloader/Dataloader_dcplocal_notTF_onlineExpert.py:142-157
//
// The dataset keeps only integer cells [R,N,2] (R = sum of the cases' T = makespan + 1 rows), goals and maps on the
// device.  dataset_prepare_kernel computes each case's threshold once; dataset_batch_kernel builds B samples -- the
// field-of-view tensor, the float32 cast of the float64 GSO and the one-hot target -- in one launch, with the same
// device functions as the rollout's inputs builder (step_inputs.cuh).  Bit-exact with the reference's files.
#include "step_inputs.cuh"

namespace gpp {

constexpr int DS_PREP_THREADS = 256;
constexpr int DS_GUARD = 4096;          // bound on the threshold's growth steps (5 * 1.1^4096 overflows long before)

// Squared length of the longest edge of a minimum spanning tree of one step's agents (Prim's algorithm, lane = agent,
// agents lane and lane + 32): the graph {pdist < r} is connected iff sqrt of it is < r, because sqrt is monotone and
// a spanning tree with every edge < r exists iff the minimax one has its longest edge < r.  One warp, N >= 2.
__device__ int ds_bottleneck_d2(const int* pos, int N, int lane) {
    const unsigned int FULL = 0xffffffffu;
    int x[2], y[2], best[2];
    bool in_tree[2];
    const int x0 = pos[0], y0 = pos[1];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int i = lane + 32 * h;
        const bool live = i < N;
        x[h] = live ? pos[2 * i] : 0;
        y[h] = live ? pos[2 * i + 1] : 0;
        best[h] = (x[h] - x0) * (x[h] - x0) + (y[h] - y0) * (y[h] - y0);
        in_tree[h] = !live || i == 0;
    }
    int longest = 0;
    for (int n = 1; n < N; ++n) {
        unsigned long long key = ~0ull;               // (squared distance to the tree, agent) of the nearest outsider
#pragma unroll
        for (int h = 0; h < 2; ++h)
            if (!in_tree[h]) key = min(key, ((unsigned long long)(unsigned)best[h] << 32) | (unsigned)(lane + 32 * h));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) key = min(key, __shfl_xor_sync(FULL, key, o));
        const int j = (int)(key & 0xffffffffu), d2 = (int)(key >> 32);
        longest = max(longest, d2);
        const int hj = j >> 5;
        const int xj = __shfl_sync(FULL, hj ? x[1] : x[0], j & 31), yj = __shfl_sync(FULL, hj ? y[1] : y[0], j & 31);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (lane + 32 * h == j) in_tree[h] = true;
            const int dx = x[h] - xj, dy = y[h] - yj;
            best[h] = min(best[h], dx * dx + dy * dy);
        }
    }
    return longest;
}

// One CTA per case, a warp per step.  computeAdjacencyMatrix multiplies the threshold by 1.1 while a step is
// disconnected and never resets it, so the final threshold is v_K (v_0 = r0, v_{k+1} = v_k * 1.1 in float64) with K the
// largest over steps of the least k at which the step is connected.
__global__ void __launch_bounds__(DS_PREP_THREADS) dataset_prepare_kernel(const int* __restrict__ pos,
                                                                          const int* __restrict__ case_first_row,
                                                                          double r0, double* __restrict__ radius, int N) {
    __shared__ int kmax;
    const int c = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) kmax = 0;
    __syncthreads();
    const int first = case_first_row[c], rows = case_first_row[c + 1] - first;
    for (int t = warp; t < rows; t += DS_PREP_THREADS / 32) {
        const int d2 = ds_bottleneck_d2(pos + (size_t)(first + t) * N * 2, N, lane);
        if (lane == 0) {
            const double d = sqrt((double)d2);          // scipy pdist (euclidean, float64) of the longest tree edge
            double v = r0;
            int k = 0;
            while (!(d < v) && k < DS_GUARD) {
                v = v * 1.1;
                ++k;
            }
            atomicMax(&kmax, k);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double v = r0;
        for (int k = 0; k < kmax; ++k) v = v * 1.1;
        radius[c] = v;
    }
}

struct DsBatchArgs {
    const int* pos;              // [R][N][2] every case's cells, case after case
    const int* row_case;         // [R] case of each row
    const int* case_first_row;   // [C + 1]
    const int* goal;             // [C][N][2]
    const unsigned char* map;    // [C][W][W] or [W][W] (map_shared)
    const double* radius;        // [C] from dataset_prepare_kernel
    const long long* rows;       // [B] samples to build
    float* x;                    // [B][N][3][11][11] out
    float* S;                    // [B][N][N] out
    long long* target;           // [B][N][5] out
    int B, N, W, R, map_shared;
};

// One CTA per sample.  The target of row t is the move to row t + 1, or to the goal on a case's last row
// (obtainSchedule :177-189); a row index outside [0, R) gives an all-zero sample.
__global__ void __launch_bounds__(128) dataset_batch_kernel(const DsBatchArgs a) {
    __shared__ unsigned long long adj[RO_MAX_N];
    __shared__ int px[RO_MAX_N], py[RO_MAX_N], nx[RO_MAX_N], ny[RO_MAX_N];
    __shared__ double dinv[RO_MAX_N];
    extern __shared__ unsigned int occ_bits[];          // ceil(W*W / 32) words: cells occupied by an agent
    const int b = blockIdx.x, tid = threadIdx.x, N = a.N, W = a.W;
    float* xo = a.x + (size_t)b * N * RO_FOV_ELEMS;
    float* So = a.S + (size_t)b * N * N;
    long long* to = a.target + (size_t)b * N * 5;
    const long long r = a.rows[b];
    if (r < 0 || r >= a.R) {
        for (int e = tid; e < N * RO_FOV_ELEMS; e += blockDim.x) xo[e] = 0.f;
        for (int e = tid; e < N * N; e += blockDim.x) So[e] = 0.f;
        for (int e = tid; e < N * 5; e += blockDim.x) to[e] = 0;
        return;
    }
    const int c = a.row_case[r];
    const int* pos = a.pos + (size_t)r * N * 2;
    const int* goal = a.goal + (size_t)c * N * 2;
    const int* next = r + 1 == a.case_first_row[c + 1] ? goal : pos + N * 2;
    const unsigned char* map = a.map + (a.map_shared ? 0 : (size_t)c * W * W);
    for (int i = tid; i < (W * W + 31) / 32; i += blockDim.x) occ_bits[i] = 0u;
    if (tid < N) {
        px[tid] = pos[2 * tid];
        py[tid] = pos[2 * tid + 1];
        nx[tid] = next[2 * tid];
        ny[tid] = next[2 * tid + 1];
    }
    __syncthreads();
    if (tid < N) {
        atomicOr(&occ_bits[(px[tid] * W + py[tid]) >> 5], 1u << ((px[tid] * W + py[tid]) & 31));
        adj[tid] = ro_adjacency_row(tid, N, px, py, a.radius[c]);
    }
    __syncthreads();
    if (tid < N) dinv[tid] = ro_deg_inv_sqrt(adj[tid]);
    __syncthreads();
    for (int e = tid; e < N * N; e += blockDim.x) {
        const int i = e / N, j = e - i * N;
        So[e] = (float)ro_gso_entry(adj, dinv, i, j);      // the loader's GSO[t].float()
    }
    for (int e = tid; e < N * 5; e += blockDim.x) {
        const int i = e / 5, q = e - i * 5;
        const int dx = nx[i] - px[i], dy = ny[i] - py[i];
        // index in delta = [[-1,0],[0,-1],[1,0],[0,1],[0,0]] (:34-38); the host rejects any other displacement
        const int key = dx == -1 && dy == 0 ? 0 : dx == 0 && dy == -1 ? 1 : dx == 1 && dy == 0 ? 2
                      : dx == 0 && dy == 1 ? 3 : dx == 0 && dy == 0 ? 4 : -1;
        to[e] = q == key ? 1 : 0;
    }
    for (int e = tid; e < N * RO_FOV_ELEMS; e += blockDim.x) xo[e] = ro_fov_value(e, px, py, goal, map, occ_bits, W);
}

}  // namespace gpp

using namespace gpp;

extern "C" int gpp_dataset_prepare(const int* pos, const int* case_first_row, double r0, double* radius, int C, int N,
                                   void* stream) {
    GPP_REQUIRE(pos && case_first_row && radius, GPP_ERR_INVALID, "dataset_prepare: null pointer");
    GPP_REQUIRE(C >= 0 && N >= 1, GPP_ERR_INVALID, "dataset_prepare: bad sizes C=%d N=%d", C, N);
    GPP_REQUIRE(N >= 2 && N <= RO_MAX_N, GPP_ERR_UNSUPPORTED, "dataset_prepare: N=%d agents outside [2, %d]", N, RO_MAX_N);
    GPP_REQUIRE(r0 > 0.0, GPP_ERR_INVALID, "dataset_prepare: radius %g <= 0", r0);
    if (C == 0) return GPP_OK;
    dataset_prepare_kernel<<<C, DS_PREP_THREADS, 0, reinterpret_cast<cudaStream_t>(stream)>>>(pos, case_first_row, r0,
                                                                                               radius, N);
    GPP_LAUNCH_CHECK();
    return GPP_OK;
}

extern "C" int gpp_dataset_batch(const int* pos, const int* row_case, const int* case_first_row, const int* goal,
                                 const unsigned char* map, int map_shared, const double* radius, const long long* rows,
                                 float* x, float* S, long long* target, int B, int N, int W, int R, void* stream) {
    GPP_REQUIRE(pos && row_case && case_first_row && goal && map && radius && rows && x && S && target, GPP_ERR_INVALID,
                "dataset_batch: null pointer");
    GPP_REQUIRE(B >= 0 && N >= 1 && W >= 1 && R >= 0, GPP_ERR_INVALID, "dataset_batch: bad sizes B=%d N=%d W=%d R=%d",
                B, N, W, R);
    GPP_REQUIRE(N >= 2 && N <= RO_MAX_N, GPP_ERR_UNSUPPORTED, "dataset_batch: N=%d agents outside [2, %d]", N, RO_MAX_N);
    const size_t smem = sizeof(unsigned int) * ((size_t)(W * W + 31) / 32);
    GPP_REQUIRE(smem <= 40 * 1024, GPP_ERR_UNSUPPORTED, "dataset_batch: map %dx%d too large", W, W);
    if (B == 0) return GPP_OK;
    DsBatchArgs a;
    a.pos = pos; a.row_case = row_case; a.case_first_row = case_first_row; a.goal = goal; a.map = map;
    a.radius = radius; a.rows = rows; a.x = x; a.S = S; a.target = target;
    a.B = B; a.N = N; a.W = W; a.R = R; a.map_shared = map_shared;
    dataset_batch_kernel<<<B, 128, smem, reinterpret_cast<cudaStream_t>(stream)>>>(a);
    GPP_LAUNCH_CHECK();
    return GPP_OK;
}
