// The planner's per-step inputs from integer agent cells, shared by the rollout's inputs builder (rollout.cu) and the
// training-batch builder (dataset.cu): the field-of-view tensor of AgentState.toInputTensor / toSeqInputTensor
// (dataloader/statetransformer.py:82-187) and the thresholded, degree-normalised adjacency of computeAdjacencyMatrix
// (utils/multirobotsim_dcenlocal.py:320-365, onlineExpert/DataTransformer_local_onlineExpert.py:256-305) at a given
// radius.  Integer window arithmetic and IEEE float64 sqrt / divide / multiply: bit-exact with the reference.
#pragma once
#include "common.cuh"

namespace gpp {

constexpr int RO_MAX_N = 64;        // agents per episode (one 64-bit adjacency mask per agent)
constexpr int RO_FOV = 9;           // statetransformer.py:11
constexpr int RO_HALF = 4;          // :12  FOV_width
constexpr int RO_WIN = 11;          // :14-15  FOV + 2 * border
constexpr int RO_CENTER = 5;        // :16,20-21
constexpr int RO_FOV_ELEMS = 3 * RO_WIN * RO_WIN;      // one agent's [3,11,11] slice

// Agent i's adjacency row: bit j set iff j != i and the float64 euclidean distance (scipy pdist) is < r.
__device__ __forceinline__ unsigned long long ro_adjacency_row(int i, int N, const int* px, const int* py, double r) {
    unsigned long long m = 0ull;
    for (int j = 0; j < N; ++j) {
        const int dx = px[i] - px[j], dy = py[i] - py[j];
        const double d = sqrt((double)(dx * dx + dy * dy));
        if (j != i && d < r) m |= 1ull << j;
    }
    return m;
}

// isConnected (graphTools.py:396-423) counts zero eigenvalues of the Laplacian = connected components; the same
// predicate by breadth-first search over the adjacency masks.
__device__ __forceinline__ bool ro_is_connected(const unsigned long long* adj, int N) {
    unsigned long long seen = 1ull, frontier = 1ull;
    while (frontier) {
        unsigned long long nxt = 0ull;
        for (int i = 0; i < N; ++i)
            if (frontier >> i & 1ull) nxt |= adj[i];
        frontier = nxt & ~seen;
        seen |= nxt;
    }
    const unsigned long long all = N >= 64 ? ~0ull : ((1ull << N) - 1ull);
    return (seen & all) == all;
}

// deg^-1/2 of one adjacency row, 0 for an isolated agent (the simulator's zero-degree guard, :341-348; the
// transformer has none, but its rows are never isolated: it grows the radius until every step is connected).
__device__ __forceinline__ double ro_deg_inv_sqrt(unsigned long long row) {
    const int deg = __popcll(row);
    return deg ? sqrt(1.0 / (double)deg) : 0.0;
}

// (D^-1/2 A D^-1/2)[i][j] in float64: (Deg @ A) @ Deg with A in {0, 1}.
__device__ __forceinline__ double ro_gso_entry(const unsigned long long* adj, const double* dinv, int i, int j) {
    return (adj[i] >> j & 1ull) ? dinv[i] * dinv[j] : 0.0;
}

// Element e of the [N,3,11,11] field-of-view tensor (statetransformer.py:82-130): channel 0 obstacle window (outside
// the map = obstacle), channel 1 goal (inside the 9x9 view, else projected onto the rim of the 11x11 window, :47-66),
// channel 2 agents.  occ_bits: bit (x * W + y) set where an agent stands.
__device__ __forceinline__ float ro_fov_value(int e, const int* px, const int* py, const int* goal,
                                              const unsigned char* map, const unsigned int* occ_bits, int W) {
    const int i = e / RO_FOV_ELEMS, rem = e - i * RO_FOV_ELEMS;
    const int ch = rem / (RO_WIN * RO_WIN), uv = rem - ch * RO_WIN * RO_WIN, u = uv / RO_WIN, v = uv - u * RO_WIN;
    const int cx = px[i], cy = py[i];
    float val = 0.f;
    if (ch != 1) {
        if (u >= 1 && u <= RO_FOV && v >= 1 && v <= RO_FOV) {
            const int gx = cx - RO_HALF + (u - 1), gy = cy - RO_HALF + (v - 1);
            const bool inside = gx >= 0 && gx < W && gy >= 0 && gy < W;
            if (ch == 0) val = inside ? (map[gx * W + gy] ? 1.f : 0.f) : 1.f;
            else val = inside && (occ_bits[(gx * W + gy) >> 5] >> ((gx * W + gy) & 31) & 1u) ? 1.f : 0.f;
        }
    } else {
        const int dx = goal[2 * i] - cx, dy = goal[2 * i + 1] - cy;
        int tx, ty;
        if (abs(dx) <= RO_HALF && abs(dy) <= RO_HALF) {
            tx = RO_CENTER + dx;
            ty = RO_CENTER + dy;
        } else if (dy != 0 && abs(dx) <= abs(dy)) {
            // bearing within [pi/4, 3pi/4] or [-3pi/4, -pi/4] (:56): |dx| <= |dy|; np.round = round half to even
            ty = RO_CENTER * ((dy > 0) - (dy < 0) + 1);
            tx = RO_CENTER + (int)rint((double)RO_CENTER * (double)dx / (double)abs(dy));
        } else {
            tx = RO_CENTER * ((dx > 0) - (dx < 0) + 1);
            ty = RO_CENTER + (int)rint((double)RO_CENTER * (double)dy / (double)abs(dx));
        }
        val = (u == tx && v == ty) ? 1.f : 0.f;
    }
    return val;
}

}  // namespace gpp
