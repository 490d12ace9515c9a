// Shared declarations for the ramannoodle_b200 CUDA library (sm_100a only).
#pragma once

#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/ramannoodle_b200.h"

namespace rn {

// ---- error plumbing ---------------------------------------------------------------
void set_error(const char* fmt, ...);
extern std::atomic<int64_t> g_launch_count;

#define RN_CUDA(expr)                                                                      \
    do {                                                                                   \
        cudaError_t err__ = (expr);                                                        \
        if (err__ != cudaSuccess) {                                                        \
            rn::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(err__), __FILE__, \
                          __LINE__);                                                       \
            return RN_ERR_CUDA;                                                            \
        }                                                                                  \
    } while (0)

#define RN_CHECK_ARG(cond, ...)              \
    do {                                     \
        if (!(cond)) {                       \
            rn::set_error(__VA_ARGS__);      \
            return RN_ERR_INVALID_ARGUMENT;  \
        }                                    \
    } while (0)

#define RN_LAUNCHED() (rn::g_launch_count.fetch_add(1, std::memory_order_relaxed))

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int device) {
        if (cudaGetDevice(&prev) != cudaSuccess) ok = false;
        if (ok && prev != device && cudaSetDevice(device) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

constexpr int kMaxDegree = 5;      // highest spline degree the dense epilogue is compiled for
constexpr int kAffineWarps = 8;    // consumer warps of the TMA affine kernel
constexpr int kAffineMaxKP = 12;   // k-step pairs per warp the TMA affine kernel is compiled for

}  // namespace rn

// ---- the model handle ---------------------------------------------------------------
struct rn_model {
    int device = 0;
    int sm_count = 0;
    int64_t num_atoms = 0;   // N
    int64_t dim = 0;         // K = 3N
    int64_t num_dofs = 0;    // J
    int64_t num_linear = 0;  // DOFs folded into the affine term
    int64_t num_dense = 0;   // DOFs evaluated by projection + spline epilogue
    int dense_degree = 0;    // max degree over dense DOFs (piece records are padded to it)
    int dense_max_pieces = 0;
    double alpha0[9] = {0};  // ref_polarizability + constant parts of the linear DOFs
    uint64_t ref_hash = 0;   // FNV-1a of the reference positions and lattice bytes (mask sweeps group on it)
    uint64_t shape_hash = 0; // ... of every creation input except the weights: equal for masked copies of a model

    // device tables (all fp64)
    double* d_ref_wrapped = nullptr;  // (K)   apply_pbc(ref positions)
    double* d_zero_ref = nullptr;     // (K)   zeros (Cartesian-displacement entry)
    double* d_g_frac = nullptr;       // (Kg,9) affine term acting on wrapped fractional displacements
    double* d_g_cart = nullptr;       // (Kg,9) affine term acting on Cartesian displacements
    double* d_v_frac = nullptr;       // (Jd_pad,Kv) dense basis with the lattice folded in
    double* d_v_cart = nullptr;       // (Jd_pad,Kv) dense basis, Cartesian
    int32_t* d_piece_off = nullptr;   // (Jd_pad+1) first piece of each dense DOF
    double* d_breaks = nullptr;       // interior break points; DOF j owns [piece_off[j]-j, piece_off[j+1]-j-1)
    double* d_pieces = nullptr;       // (pieces, 1 + 9*(dense_degree+1)): x0 then coefficients c[m][q]
    int64_t g_rows = 0;               // Kg: rows of the affine tables (K padded)
    int64_t v_cols = 0;               // Kv: columns of the dense basis (K padded to 16)
    int64_t dense_pad = 0;            // Jd_pad: dense DOFs padded to the J tile
    int affine_kp = 0;                // k-step pairs per warp for the TMA affine kernel (0 = ineligible)

    // truncated-power form of the dense DOFs (chained-DMMA epilogue): B_j(x) = const_j +
    // sum_{m=1..D} g_{j,m} (x-x0_j)^m + sum_i sum_m d_{j,i,m} max(x-b_{j,i},0)^m
    int tp_mode = 0;                  // 0 = unavailable, 1 = top power per break (true splines), 2 = all powers
    int tp_breaks = 0;                // break slots per DOF (padded with +inf)
    int tp_features = 0;              // features per DOF
    double alpha0_tp[9] = {0};        // alpha0 + sum_j const_j
    double* d_tp_x0 = nullptr;        // (Jd_pad)
    double* d_tp_brk = nullptr;       // (Jd_pad, tp_breaks)
    double* d_tp_c8 = nullptr;        // (Jd_pad, tp_features, 8) tensor components 0..7
    double* d_tp_c9 = nullptr;        // (Jd_pad, tp_features)    tensor component 8
};

namespace rn {

// Extra destinations of the polarizability series, written by the evaluation kernels themselves over
// NVLink (peer-mapped device memory).
//   broadcast (log2_period < 0): the rows are stored to ptr[0..count) — every pointer pre-offset to this
//     rank's first frame (fused all-gather);
//   routed (log2_period >= 0): ptr[r] is rank r's full (S,3,3) series buffer (null for this rank itself or
//     for ranks that own nothing); row n (global index first_frame + local row) goes to the ranks
//     owner(n) and owner(n-1), owner(n) = (n mod 2^log2_period) >> log2_width — the rank whose spectrum
//     stage consumes the difference signal n needs rows n and n+1 (rn_spectrum_dist_route).
// A subset of the local frames for one launch (pipelined multi-GPU schedule: the rows one half of the
// spectrum stage's pack needs are evaluated first, so that the pack can overlap the evaluation of the rest).
// In units of tiles of the kernel's frames-per-tile: local tile t has the global number g = tile0 + t; the
// launch processes the tiles with lo <= g mod period < lo + width, in increasing order.
struct TileSelect {
    int64_t period;  // 0: every tile
    int64_t lo, width;
    int64_t x0;      // tile0 mod period
    int64_t c0;      // selected tiles before the first period boundary
    int64_t count;   // selected tiles in all
};

struct AlphaPeers {
    double* ptr[8];
    int count;
    int log2_period;
    int log2_width;
    int64_t first_frame;
    int64_t sel_stripe;  // > 0: evaluate one phase only (rn_calc_polarizabilities_routed_phase)
    int sel_phase;
};

// local tile of the j-th selected one
__host__ __device__ inline int64_t select_tile(const TileSelect& S, int64_t j) {
    if (S.period == 0) return j;
    const int64_t first = S.x0 > S.lo ? S.x0 : S.lo;
    if (j < S.c0) return first - S.x0 + j;
    j -= S.c0;
    return (1 + j / S.width) * S.period + S.lo + (j % S.width) - S.x0;
}

// The same walk without divisions in the loop: a CTA visits the selected tiles j, j + step, j + 2 step, ...
struct TileCursor {
    int64_t j;       // index among the selected tiles
    int64_t k, r;    // j >= c0: period number (>= 1) and offset inside the window
};
__host__ __device__ inline void cursor_set(const TileSelect& S, int64_t j, TileCursor& c) {
    c.j = j;
    c.k = 0;
    c.r = 0;
    if (S.period && j >= S.c0) {
        c.k = 1 + (j - S.c0) / S.width;
        c.r = (j - S.c0) % S.width;
    }
}
__host__ __device__ inline void cursor_advance(const TileSelect& S, int64_t step, TileCursor& c) {
    const int64_t before = c.j;
    c.j += step;
    if (!S.period || c.j < S.c0) return;
    if (before < S.c0) {
        c.k = 1;
        c.r = c.j - S.c0;
    } else {
        c.r += step;
    }
    while (c.r >= S.width) {
        c.r -= S.width;
        c.k++;
    }
}
__host__ __device__ inline int64_t cursor_tile(const TileSelect& S, const TileCursor& c) {
    if (S.period == 0) return c.j;
    if (c.j < S.c0) return (S.x0 > S.lo ? S.x0 : S.lo) - S.x0 + c.j;
    return c.k * S.period + S.lo + c.r - S.x0;
}

inline TileSelect all_tiles() {
    TileSelect S;
    S.period = S.lo = S.width = S.x0 = S.c0 = S.count = 0;
    return S;
}

// selection of the tiles lo <= g mod period < lo + width among local tiles [0, num_tiles), g = tile0 + t
inline TileSelect make_tile_select(int64_t tile0, int64_t num_tiles, int64_t period, int64_t lo, int64_t width) {
    TileSelect S;
    S.period = period;
    S.lo = lo;
    S.width = width;
    S.x0 = tile0 % period;
    const int64_t first = S.x0 > lo ? S.x0 : lo;
    const int64_t in_first = std::max<int64_t>(0, std::min(lo + width, S.x0 + num_tiles) - first);
    S.c0 = in_first;
    int64_t count = in_first;
    const int64_t end = S.x0 + num_tiles;  // one past the last local tile, counted from the period start
    for (int64_t k = 1; k * period < end; k++)
        count += std::max<int64_t>(0, std::min(k * period + lo + width, end) - (k * period + lo));
    S.count = count;
    return S;
}

// the tiles (of `rows` frames, a divisor of 16) of one phase of the pipelined schedule: phase 0 = frames n with
// (n mod 2 stripe) < stripe + 16, phase 1 = the others
inline TileSelect phase_tiles(int64_t first_frame, int64_t num_frames, int64_t stripe, int phase, int rows) {
    const int64_t edge = (stripe + 16) / rows, period = 2 * stripe / rows;
    return phase == 0 ? make_tile_select(first_frame / rows, num_frames / rows, period, 0, edge)
                      : make_tile_select(first_frame / rows, num_frames / rows, period, edge, period - edge);
}

// bit r set: rows [local_row, local_row + rows) go to ptr[r] (rows <= 2^log2_width: at most two owners)
__host__ __device__ inline uint32_t alpha_peer_mask(const AlphaPeers& P, int64_t local_row, int rows) {
    if (P.log2_period < 0) return (1u << P.count) - 1u;
    const int64_t n0 = P.first_frame + local_row;
    const int64_t period_mask = ((int64_t)1 << P.log2_period) - 1;
    const int64_t a = n0 > 0 ? n0 - 1 : 0, b = n0 + rows - 1;
    return (1u << (int)((a & period_mask) >> P.log2_width)) | (1u << (int)((b & period_mask) >> P.log2_width));
}
inline AlphaPeers no_peers() {
    AlphaPeers p;
    for (int i = 0; i < 8; i++) p.ptr[i] = nullptr;
    p.count = 0;
    p.log2_period = -1;
    p.log2_width = 0;
    p.first_frame = 0;
    p.sel_stripe = 0;
    p.sel_phase = 0;
    return p;
}
// offset (doubles) of local row `local_row` in destination r
__host__ __device__ inline int64_t alpha_peer_offset(const AlphaPeers& P, int64_t local_row) {
    return (P.log2_period < 0 ? local_row : P.first_frame + local_row) * 9;
}
// the destinations of local rows f0, f0 + 1, ... as a launch that starts at local row f0 sees them
inline AlphaPeers peers_at(const AlphaPeers& P, int64_t f0) {
    AlphaPeers Q = P;
    if (P.log2_period < 0) {
        for (int p = 0; p < P.count; p++) Q.ptr[p] = P.ptr[p] + f0 * 9;
    } else {
        Q.first_frame = P.first_frame + f0;
    }
    return Q;
}

// kernels / launchers implemented in rn_polarizability.cu / rn_dense.cu.  `peers` may be null;
// *peers_done is set when the launched kernel stored to the peers itself.
int launch_affine(const rn_model* m, const double* d_in, bool wrap, int64_t num_frames, double* d_alpha,
                  cudaStream_t stream, const AlphaPeers* peers = nullptr, bool* peers_done = nullptr);
int launch_dense(const rn_model* m, const double* d_in, bool wrap, bool accumulate, int64_t num_frames,
                 double* d_alpha, cudaStream_t stream, const AlphaPeers* peers = nullptr, bool* peers_done = nullptr);
int launch_dense_v1(const rn_model* m, const double* d_in, bool wrap, bool accumulate, int64_t num_frames,
                    double* d_alpha, cudaStream_t stream);
int launch_fill_alpha0(const rn_model* m, int64_t num_frames, double* d_alpha, cudaStream_t stream);
// rn_polarizability.cu: calc_polarizabilities of `num_frames` device-resident frames with extra destinations
int eval_with_peers(const rn_model* model, const double* d_positions, int64_t num_frames, double* d_alpha,
                    cudaStream_t stream, const AlphaPeers& peers);
int make_routed_peers(double* const* peer_series, int world, int64_t first_frame, int64_t period, int64_t width,
                      AlphaPeers* peers);
// rn_dense_sweep.cu: spline part of 2..4 masked copies of one model with a shared projection; `routed`
// (null, or one entry per model) names the ranks the finished rows of each model also go to
bool dense_sweep_eligible(const rn_model* m);
bool dense_sweep_compatible(const rn_model* a, const rn_model* b);
int launch_dense_sweep(const rn_model* const* models, int count, const double* d_in, bool accumulate,
                       int64_t num_frames, double* const* d_alpha, cudaStream_t stream,
                       const AlphaPeers* routed = nullptr);
// rn_sweep.cu: mask sweep of device-resident frames; `routed` as above
constexpr int kMaxSweepModels = 64;
int sweep_eval(const rn_model* const* models, int num_models, const double* d_positions, int64_t num_frames,
               double* const* d_alpha_outputs, cudaStream_t stream, const AlphaPeers* routed);
// routed[g] = make_routed_peers(peer_series + g * world, ...) for every model
int make_sweep_peers(int num_models, double* const* peer_series, int world, int64_t first_frame, int64_t period,
                     int64_t width, AlphaPeers* routed);

}  // namespace rn
