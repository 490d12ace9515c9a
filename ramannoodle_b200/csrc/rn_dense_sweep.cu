// Mask sweeps of spline models (SURVEY.md §8f row N3): NG masked copies of one InterpolationModel
// (get_masked_model, ramannoodle/pmodel/_interpolation.py:697-708) share everything but the weights
// 1 - mask_j, so one launch of dense_kernel_tp projects every frame onto the basis ONCE
// (2*3N*J flop/frame, the expensive part of _interpolation.py:239-241) and runs the chained-DMMA
// spline epilogue once per mask against that mask's coefficient table — the amplitudes are re-used
// in registers instead of being recomputed per copy.
#include <algorithm>

#include "rn_dense_tp.cuh"

namespace rn {

constexpr int kDenseSweepMax = 4;

template <int DEG, int NBK, bool FULL, int NG>
static int launch_tp_sweep_cfg(const rn_model* const* models, const double* d_in, bool accumulate,
                               int64_t num_frames, double* const* d_alpha, cudaStream_t stream,
                               const AlphaPeers* routed) {
    const rn_model* m = models[0];
    const int K = (int)m->dim;
    constexpr int FT = 128;
    const bool align16 = (reinterpret_cast<uintptr_t>(d_in) % 16 == 0) && (K % 2 == 0);
    const int stages = tp_stages(0, align16);
    const size_t smem = tp_smem_bytes(stages);
    const int64_t tiles = (num_frames + FT - 1) / FT;
    int grid = (int)std::min<int64_t>(tiles, m->sm_count);
    // unit-balanced schedule for short trajectories, as in rn_dense.cu: launch_tp_cfg
    const int64_t jtiles = m->dense_pad / kJT2;
    const int64_t rounds = (tiles + m->sm_count - 1) / m->sm_count;
    // (not with routed stores: the peers need finished rows)
    const bool split = !routed && tiles * jtiles >= 2 && (double)(rounds * m->sm_count) > 1.04 * (double)tiles;
    if (split) {
        grid = (int)std::min<int64_t>(tiles * jtiles, m->sm_count);
        if (!accumulate) {
            for (int g = 0; g < NG; g++) {
                int rc = launch_fill_alpha0(models[g], num_frames, d_alpha[g], stream);
                if (rc != RN_OK) return rc;
            }
            accumulate = true;
        }
    }
    TpMasks<NG> mk;
    for (int g = 0; g < NG; g++) {
        const rn_model* mg = models[g];
        mk.c8[g] = mg->d_tp_c8;
        mk.c9[g] = mg->d_tp_c9;
        mk.alpha[g] = d_alpha[g];
        for (int q = 0; q < 9; q++)
            mk.a0[g].v[q] = accumulate ? (mg->alpha0_tp[q] - mg->alpha0[q]) : mg->alpha0_tp[q];
    }
    // routed: one set of destinations per mask (kernels of their own, the plain sweep's code stays as it is)
    TpPeers<1> none;
    none.mask[0] = no_peers();
    TpPeers<NG> peers;
    for (int g = 0; g < NG; g++) peers.mask[g] = routed ? routed[g] : no_peers();
#define RN_TP_SWEEP_LAUNCH(A, NP, P)                                                                            \
    {                                                                                                           \
        auto kern = dense_kernel_tp<DEG, NBK, FULL, true, A, NG, NP>;                                           \
        RN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));            \
        kern<<<grid, 384, smem, stream>>>(d_in, m->d_ref_wrapped, m->d_v_frac, m->d_tp_x0, m->d_tp_brk,         \
                                          num_frames, K, (int)m->v_cols, (int)m->dense_pad, (int)m->num_dense, accumulate ? 1 : 0, \
                                          split ? 1 : 0, stages, mk, P);                                                \
    }
    if (routed) {
        if (align16) RN_TP_SWEEP_LAUNCH(true, NG, peers) else RN_TP_SWEEP_LAUNCH(false, NG, peers)
    } else {
        if (align16) RN_TP_SWEEP_LAUNCH(true, 1, none) else RN_TP_SWEEP_LAUNCH(false, 1, none)
    }
#undef RN_TP_SWEEP_LAUNCH
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    return RN_OK;
}

template <int DEG, int NG>
static int launch_tp_sweep_deg(const rn_model* const* models, const double* d_in, bool accumulate, int64_t num_frames,
                               double* const* d_alpha, cudaStream_t stream, const AlphaPeers* routed) {
    const rn_model* m = models[0];
    const bool full = m->tp_mode == 2;
    switch (m->tp_breaks) {
        case 0: return launch_tp_sweep_cfg<DEG, 0, false, NG>(models, d_in, accumulate, num_frames, d_alpha, stream, routed);
        case 1:
            return full ? launch_tp_sweep_cfg<DEG, 1, true, NG>(models, d_in, accumulate, num_frames, d_alpha, stream, routed)
                        : launch_tp_sweep_cfg<DEG, 1, false, NG>(models, d_in, accumulate, num_frames, d_alpha, stream, routed);
        case 2:
            return full ? launch_tp_sweep_cfg<DEG, 2, true, NG>(models, d_in, accumulate, num_frames, d_alpha, stream, routed)
                        : launch_tp_sweep_cfg<DEG, 2, false, NG>(models, d_in, accumulate, num_frames, d_alpha, stream, routed);
        case 3:
            return full ? 1
                        : launch_tp_sweep_cfg<DEG, 3, false, NG>(models, d_in, accumulate, num_frames, d_alpha, stream, routed);
        default: return 1;
    }
}

template <int NG>
static int launch_tp_sweep_ng(const rn_model* const* models, const double* d_in, bool accumulate, int64_t num_frames,
                              double* const* d_alpha, cudaStream_t stream, const AlphaPeers* routed) {
    switch (models[0]->dense_degree) {
        case 1: return launch_tp_sweep_deg<1, NG>(models, d_in, accumulate, num_frames, d_alpha, stream, routed);
        case 2: return launch_tp_sweep_deg<2, NG>(models, d_in, accumulate, num_frames, d_alpha, stream, routed);
        case 3: return launch_tp_sweep_deg<3, NG>(models, d_in, accumulate, num_frames, d_alpha, stream, routed);
        default: return 1;
    }
}

// models that may share one projection: masked copies of one model (identical tables up to the weights)
bool dense_sweep_compatible(const rn_model* a, const rn_model* b) {
    return a->device == b->device && a->dim == b->dim && a->shape_hash == b->shape_hash &&
           a->num_dense == b->num_dense && a->num_linear == b->num_linear && a->dense_pad == b->dense_pad &&
           a->v_cols == b->v_cols && a->tp_mode == b->tp_mode && a->tp_breaks == b->tp_breaks &&
           a->tp_features == b->tp_features && a->dense_degree == b->dense_degree;
}

bool dense_sweep_eligible(const rn_model* m) {
    return m->num_dense > 0 && m->tp_mode != 0 && m->tp_features <= 12 && m->dense_degree >= 1 && m->dense_degree <= 3;
}

// Dense (spline) part of `count` (2 or 4) compatible models on fractional positions: accumulates onto
// d_alpha[g] when `accumulate` (their affine parts were written first), else writes alpha0 + sum; with
// `routed`, the finished rows of model g also go to the ranks routed[g] names.
// Returns 1 when no kernel configuration covers the models (caller evaluates them one by one).
int launch_dense_sweep(const rn_model* const* models, int count, const double* d_in, bool accumulate,
                       int64_t num_frames, double* const* d_alpha, cudaStream_t stream, const AlphaPeers* routed) {
    // instantiated for 2 and 4 masks (build time); the caller deals runs of 3 out as 2 + 1
    if (count == 2) return launch_tp_sweep_ng<2>(models, d_in, accumulate, num_frames, d_alpha, stream, routed);
    if (count == 4) return launch_tp_sweep_ng<4>(models, d_in, accumulate, num_frames, d_alpha, stream, routed);
    return 1;
}

}  // namespace rn
