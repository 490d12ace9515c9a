// Dense polarizability kernels (sm_100a): general splines.
//
//   alpha_s (+)= sum_{j in dense DOFs} w_j B_j( v_j . vec(wrap(p_s - p_ref) L) )
//   (ramannoodle/pmodel/_interpolation.py:233-252: one einsum + one BSpline call per DOF)
//
// One persistent CTA per SM.  A work tile is 128 frames x all dense DOFs; DOFs are walked in tiles
// of 64, K = 3N in chunks of 16 through a 4-stage cp.async ring.  The kernel is warp-specialised:
//   warps 8-11 (producers): fill the ring with cp.async, then replace the raw fractional positions
//       of a landed chunk in shared memory by their minimum-image displacements
//       (d - ceil(d - 0.5) against the wrapped reference; vectorised, once per element);
//   warps 0-7 (MMA): LDS + DMMA m8n8k4 only (the FP64 tensor path on sm_100; tcgen05 has no f64
//       kind), register double-buffered fragments, 16x64 accumulator tile per warp; two MMA warps
//       per scheduler so that one covers the other's LDS / mbarrier bubbles (the DMMA issue queue
//       is shallow: tools/dmma_occupancy.cu, tools/dmma_operands.cu).
//   Stages are handed over with mbarriers (full/empty), so MMA warps never wait on each other.
// Epilogue (once per DOF tile), chained DMMA: the amplitude accumulators are turned, in registers,
// into truncated-power features ((x-x0)^m, max(x-b,0)^m) and fed as the A operand of a second DMMA
// against the per-DOF coefficient table, accumulating the frame's 3x3 tensor directly — no shared
// memory round trip, no per-frame table walk; the (S,J) amplitude matrix never touches HBM.
// FP64-pipe bound: 2*3N*J flops per frame against the measured DMMA rate (profiles/fp64_peaks.json).
#include <algorithm>

#include "rn_dense_tp.cuh"

namespace rn {

// A/B hook (rn_debug_set_dense_config): generation 1 = rn_polarizability.cu, 3 = warp-specialised with
// the piecewise-polynomial epilogue, 4 = warp-specialised with the chained-DMMA epilogue (default)
// A/B switches (include/ramannoodle_b200_debug.h): atomics, read once per launch
static std::atomic<int> g_dense_version{4};
static std::atomic<int> g_dense_variant{0};  // A/B bits: 1 = one-DADD wrap with a branch in the producers, 2 = compute the DOF padding
static std::atomic<int> g_dense_stages{kTpStagesDefault};
static std::atomic<int> g_dense_split{1};  // 0 = never, 1 = when whole tiles would leave SMs idle, 2 = always (tests)

// ------------------------------------------------------------------------------------
// Third generation: warp-specialised.  Warps 0-3 only issue LDS + DMMA (one MMA warp per
// scheduler saturates the FP64 tensor pipe: tools/dmma_occupancy.cu), warps 4-7 are producers
// (cp.async ring fill + in-place minimum-image wrap).  Stages are handed over with mbarriers, so
// MMA warps never wait for each other or for address arithmetic.
// ------------------------------------------------------------------------------------
template <int DEG, int PB, bool WRAP, bool ALIGN16>
__global__ void __launch_bounds__(256, 1)
    dense_kernel_v3(const double* __restrict__ in, const double* __restrict__ ref, const double* __restrict__ V,
                    const int32_t* __restrict__ piece_off, const double* __restrict__ breaks,
                    const double* __restrict__ pieces, int64_t num_frames, int K, int Kv, int Jpad, int accumulate,
                    Alpha0 a0, double* __restrict__ alpha) {
    constexpr int FT = 128;  // frames per tile: 4 MMA warps x 32
    constexpr int REC = 1 + 9 * (DEG + 1);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* As = reinterpret_cast<double*>(smem_raw);          // [kStages2][FT][kRS2]
    double* Bs = As + (size_t)kStages2 * FT * kRS2;            // [kStages2][kJT2][kRS2]
    double* amp = Bs + (size_t)kStages2 * kJT2 * kRS2;         // [FT][kAmpStride]
    uint64_t* bars = reinterpret_cast<uint64_t*>(amp + (size_t)FT * kAmpStride);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + kStages2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int chunks = Kv / kKC2;
    const int jtiles = Jpad / kJT2;
    const int64_t total = (int64_t)jtiles * chunks;
    const int64_t num_tiles = (num_frames + FT - 1) / FT;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages2; s++) {
            mbar_init2(full0 + 8 * s, 128);  // every producer thread arrives after its wrap items
            mbar_init2(empty0 + 8 * s, 4);   // one arrival per MMA warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp >= 4) {
        // =========================== producers (128 threads) ===========================
        const int ptid = threadIdx.x - 128;
        constexpr int A_SEGS = ALIGN16 ? 8 : 16;
        constexpr int A_ELEMS = ALIGN16 ? 2 : 1;
        constexpr int A_ITEMS = (FT * A_SEGS) / 128;
        constexpr int A_ROWSTEP = 128 / A_SEGS;
        const int a_row0 = ptid / A_SEGS, a_seg = ptid % A_SEGS;
        const int b_row0 = ptid >> 3, b_seg = ptid & 7;
        const uint32_t a_dst0 = smem_u32(As) + (uint32_t)(a_row0 * kRS2 + a_seg * A_ELEMS) * 8u;
        const uint32_t b_dst0 = smem_u32(Bs) + (uint32_t)(b_row0 * kRS2 + b_seg * 2) * 8u;
        constexpr uint32_t A_STAGE_BYTES = FT * kRS2 * 8, B_STAGE_BYTES = kJT2 * kRS2 * 8;
        const double* v_src0 = V + (int64_t)b_row0 * Kv + b_seg * 2;
        const int w_row0 = ptid >> 3, w_seg = ptid & 7;

        uint32_t issued = 0;   // chunks issued so far (running over all tiles: ring stage / parity)
        uint32_t wrapped = 0;  // chunks handed to the MMA warps so far
        for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            const int64_t frame0 = tile * FT;
            const double* a_src_row[A_ITEMS];
#pragma unroll
            for (int r = 0; r < A_ITEMS; r++) {
                const int64_t frame = frame0 + a_row0 + r * A_ROWSTEP;
                a_src_row[r] = (frame < num_frames) ? in + frame * (int64_t)K + a_seg * A_ELEMS : nullptr;
            }
            int is_kc = 0, is_jt = 0;
            auto issue = [&]() {
                if (is_jt < jtiles) {
                    const uint32_t st = issued & (kStages2 - 1);
                    if (issued >= (uint32_t)kStages2) mbar_wait2(empty0 + 8 * st, ((issued >> 2) - 1) & 1);
                    const int col = is_kc * kKC2 + a_seg * A_ELEMS;
                    const int rem = K - col;
                    const int bytes = ALIGN16 ? (rem >= 2 ? 16 : (rem == 1 ? 8 : 0)) : (rem >= 1 ? 8 : 0);
                    const uint32_t a_dst = a_dst0 + st * A_STAGE_BYTES;
#pragma unroll
                    for (int r = 0; r < A_ITEMS; r++) {
                        const double* row = a_src_row[r];
                        const int nb = row ? bytes : 0;
                        const double* src = nb ? row + is_kc * kKC2 : in;
                        if (ALIGN16) cp_async_16(a_dst + (uint32_t)(r * A_ROWSTEP * kRS2) * 8u, src, nb);
                        else cp_async_8(a_dst + (uint32_t)(r * A_ROWSTEP * kRS2) * 8u, src, nb);
                    }
                    const uint32_t b_dst = b_dst0 + st * B_STAGE_BYTES;
                    const double* vsrc = v_src0 + ((int64_t)is_jt * kJT2) * Kv + is_kc * kKC2;
#pragma unroll
                    for (int r = 0; r < (kJT2 * 8) / 128; r++)
                        cp_async_16(b_dst + (uint32_t)(r * 16 * kRS2) * 8u, vsrc + (int64_t)r * 16 * Kv, 16);
                    if (++is_kc == chunks) {
                        is_kc = 0;
                        ++is_jt;
                    }
                    ++issued;
                }
                cp_async_commit();
            };
            issue();
            issue();
            int wr_kc = 0;
            for (int64_t c = 0; c < total; c++) {
                issue();             // chunk c+2
                cp_async_wait<2>();  // this thread's copies of chunk c have landed
                asm volatile("bar.sync 1, 128;" ::: "memory");  // ... and every producer's
                const uint32_t st = wrapped & (kStages2 - 1);
                if (WRAP) {
                    double* a = As + (size_t)st * FT * kRS2 + w_row0 * kRS2 + w_seg * 2;
                    const double2 rf = __ldg(reinterpret_cast<const double2*>(ref + wr_kc * kKC2 + w_seg * 2));
#pragma unroll
                    for (int r = 0; r < FT / 16; r++) {
                        double2* p = reinterpret_cast<double2*>(a + r * 16 * kRS2);
                        double2 v = *p;
                        v.x = wrap_disp(v.x, rf.x);
                        v.y = wrap_disp(v.y, rf.y);
                        *p = v;
                    }
                    if (++wr_kc == chunks) wr_kc = 0;
                }
                mbar_arrive2(full0 + 8 * st);  // release: this thread's stage writes are visible to waiters
                ++wrapped;
            }
            cp_async_wait<0>();
        }
        return;
    }

    // =============================== MMA warps (128 threads) ===============================
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp;  // frames 32*wm .. 32*wm+31
    uint32_t consumed = 0;
    for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int64_t frame0 = tile * FT;
        double out9[9];
#pragma unroll
        for (int q = 0; q < 9; q++) out9[q] = 0.0;
        double acc[4][8][2];
        int kc = 0, jt = 0;
        for (int64_t c = 0; c < total; c++) {
            if (kc == 0) {
#pragma unroll
                for (int mt = 0; mt < 4; mt++)
#pragma unroll
                    for (int nt = 0; nt < 8; nt++) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
            }
            const uint32_t st = consumed & (kStages2 - 1);
            mbar_wait2(full0 + 8 * st, (consumed >> 2) & 1);
            const double* a_src = As + (size_t)st * FT * kRS2 + (wm * 32 + g) * kRS2 + t;
            const double* b_src = Bs + (size_t)st * kJT2 * kRS2 + g * kRS2 + t;
            double af[2][4], bf[2][8];
#pragma unroll
            for (int mt = 0; mt < 4; mt++) af[0][mt] = a_src[mt * 8 * kRS2];
#pragma unroll
            for (int nt = 0; nt < 8; nt++) bf[0][nt] = b_src[nt * 8 * kRS2];
#pragma unroll
            for (int s = 0; s < kKC2 / 4; s++) {
                const int cur = s & 1, nxt = cur ^ 1;
                if (s + 1 < kKC2 / 4) {
#pragma unroll
                    for (int mt = 0; mt < 4; mt++) af[nxt][mt] = a_src[mt * 8 * kRS2 + 4 * (s + 1)];
#pragma unroll
                    for (int nt = 0; nt < 8; nt++) bf[nxt][nt] = b_src[nt * 8 * kRS2 + 4 * (s + 1)];
                }
#pragma unroll
                for (int nt = 0; nt < 8; nt++)
#pragma unroll
                    for (int mt = 0; mt < 4; mt++) dmma884(acc[mt][nt][0], acc[mt][nt][1], af[cur][mt], bf[cur][nt]);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive2(empty0 + 8 * st);  // stage may be refilled
            ++consumed;
            const bool last_chunk = (kc == chunks - 1);
            const int jt_now = jt;
            if (++kc == chunks) {
                kc = 0;
                ++jt;
            }
            if (last_chunk) {
                // ---- epilogue of this DOF tile (MMA warps only; producers keep prefetching) ----
                asm volatile("bar.sync 2, 128;" ::: "memory");  // previous amplitude tile fully consumed
#pragma unroll
                for (int mt = 0; mt < 4; mt++)
#pragma unroll
                    for (int nt = 0; nt < 8; nt++) {
                        double* dst = amp + (size_t)(wm * 32 + mt * 8 + g) * kAmpStride + nt * 8 + 2 * t;
                        dst[0] = acc[mt][nt][0];
                        dst[1] = acc[mt][nt][1];
                    }
                asm volatile("bar.sync 2, 128;" ::: "memory");
                const double* arow = amp + (size_t)threadIdx.x * kAmpStride;  // thread <-> frame
                const int j0 = jt_now * kJT2;
#pragma unroll 2
                for (int jj = 0; jj < kJT2; jj++) {
                    const double x = arow[jj];
                    const int p0 = __ldg(piece_off + j0 + jj);  // warp-uniform
                    int p = 0;
                    if (PB > 0) {
                        const int np = __ldg(piece_off + j0 + jj + 1) - p0;
#pragma unroll
                        for (int b = 0; b < PB; b++)
                            if (b + 1 < np) p += (x >= __ldg(breaks + p0 + b)) ? 1 : 0;
                    }
                    const double* rec = pieces + (int64_t)(p0 + p) * REC;
                    const double dx = x - __ldg(rec);
#pragma unroll
                    for (int q = 0; q < 9; q++) {
                        double r = __ldg(rec + 1 + q);
#pragma unroll
                        for (int mm = 1; mm <= DEG; mm++) r = fma(r, dx, __ldg(rec + 1 + 9 * mm + q));
                        out9[q] += r;
                    }
                }
            }
        }
        const int64_t frame = frame0 + threadIdx.x;
        if (frame < num_frames) {
#pragma unroll
            for (int q = 0; q < 9; q++) {
                const double base = accumulate ? alpha[frame * 9 + q] : a0.v[q];
                alpha[frame * 9 + q] = out9[q] + base;
            }
        }
    }
}

template <int DEG, int NBK, bool FULL>
static int launch_tp_cfg(const rn_model* m, const double* d_in, bool wrap, bool accumulate, int64_t num_frames,
                         double* d_alpha, cudaStream_t stream, const AlphaPeers& peers) {
    // constants: alpha0_tp = alpha0 + sum of the dense DOFs' constant terms.  When the affine kernel
    // already wrote alpha0 + D.G (accumulate), only the dense constants remain to be added.
    const int K = (int)m->dim;
    constexpr int FT = 128;
    const bool align16 = (reinterpret_cast<uintptr_t>(d_in) % 16 == 0) && (K % 2 == 0);
    const int stages = tp_stages(g_dense_stages.load(std::memory_order_relaxed), align16);
    const size_t smem = tp_smem_bytes(stages);
    const int64_t tiles = (num_frames + FT - 1) / FT;
    int grid = (int)std::min<int64_t>(tiles, m->sm_count);
    // Whole frame tiles per CTA leave SMs idle in the last wave when there are few tiles per SM
    // (100k STO frames: 782 tiles on 148 SMs = 5.3 -> 6 rounds; 10k frames: 79 tiles, 69 SMs idle).
    // Then the (frame tile, DOF tile) units are balanced over all SMs instead; shared tiles finish
    // with atomic adds, so the rows are pre-filled (alpha0) and the kernel runs in accumulate mode.
    // Not used with fused peer stores (the peers need finished rows).
    const int64_t jtiles = m->dense_pad / kJT2;
    const int64_t rounds = (tiles + m->sm_count - 1) / m->sm_count;
    const int split_mode = g_dense_split.load(std::memory_order_relaxed);
    const bool split = split_mode != 0 && peers.count == 0 && tiles * jtiles >= 2 &&
                       (split_mode == 2 || (double)(rounds * m->sm_count) > 1.04 * (double)tiles);
    if (split) {
        grid = (int)std::min<int64_t>(tiles * jtiles, m->sm_count);
        if (!accumulate) {
            int rc = launch_fill_alpha0(m, num_frames, d_alpha, stream);
            if (rc != RN_OK) return rc;
            accumulate = true;
        }
    }
    Alpha0 a0;
    for (int q = 0; q < 9; q++) a0.v[q] = accumulate ? (m->alpha0_tp[q] - m->alpha0[q]) : m->alpha0_tp[q];
    const double* V = wrap ? m->d_v_frac : m->d_v_cart;
    TpMasks<1> mk;
    mk.c8[0] = m->d_tp_c8;
    mk.c9[0] = m->d_tp_c9;
    mk.alpha[0] = d_alpha;
    mk.a0[0] = a0;
    TpPeers<1> tpeers;
    tpeers.mask[0] = peers;
#define RN_TP_LAUNCH(W, A)                                                                                   \
    {                                                                                                        \
        auto kern = dense_kernel_tp<DEG, NBK, FULL, W, A, 1>;                                                \
        RN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));         \
        kern<<<grid, 384, smem, stream>>>(d_in, m->d_ref_wrapped, V, m->d_tp_x0, m->d_tp_brk, num_frames, K, \
                                          (int)m->v_cols, (int)m->dense_pad, (int)m->num_dense, accumulate ? 1 : 0,             \
                                          (split ? 1 : 0) | (g_dense_variant.load(std::memory_order_relaxed) << 1), stages, mk, tpeers);                                        \
    }
    if (wrap) {
        if (align16) RN_TP_LAUNCH(true, true) else RN_TP_LAUNCH(true, false)
    } else {
        if (align16) RN_TP_LAUNCH(false, true) else RN_TP_LAUNCH(false, false)
    }
#undef RN_TP_LAUNCH
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    return RN_OK;
}

template <int DEG>
static int launch_tp_deg(const rn_model* m, const double* d_in, bool wrap, bool accumulate, int64_t num_frames,
                         double* d_alpha, cudaStream_t stream, const AlphaPeers& peers) {
    const bool full = m->tp_mode == 2;
    switch (m->tp_breaks) {
        case 0: return launch_tp_cfg<DEG, 0, false>(m, d_in, wrap, accumulate, num_frames, d_alpha, stream, peers);
        case 1:
            return full ? launch_tp_cfg<DEG, 1, true>(m, d_in, wrap, accumulate, num_frames, d_alpha, stream, peers)
                        : launch_tp_cfg<DEG, 1, false>(m, d_in, wrap, accumulate, num_frames, d_alpha, stream, peers);
        case 2:
            return full ? launch_tp_cfg<DEG, 2, true>(m, d_in, wrap, accumulate, num_frames, d_alpha, stream, peers)
                        : launch_tp_cfg<DEG, 2, false>(m, d_in, wrap, accumulate, num_frames, d_alpha, stream, peers);
        case 3:
            return full ? 1 : launch_tp_cfg<DEG, 3, false>(m, d_in, wrap, accumulate, num_frames, d_alpha, stream, peers);
        default: return 1;
    }
}

template <int DEG, int PB>
static int launch_v3_cfg(const rn_model* m, const double* d_in, bool wrap, bool accumulate, int64_t num_frames,
                         double* d_alpha, cudaStream_t stream) {
    Alpha0 a0;
    for (int q = 0; q < 9; q++) a0.v[q] = m->alpha0[q];
    const int K = (int)m->dim;
    constexpr int FT = 128;
    const bool align16 = (reinterpret_cast<uintptr_t>(d_in) % 16 == 0) && (K % 2 == 0);
    const size_t smem = ((size_t)kStages2 * (FT + kJT2) * kRS2 + (size_t)FT * kAmpStride) * sizeof(double) + 128;
    const int64_t tiles = (num_frames + FT - 1) / FT;
    const int grid = (int)std::min<int64_t>(tiles, m->sm_count);
    const double* V = wrap ? m->d_v_frac : m->d_v_cart;
#define RN_V3_LAUNCH(W, A)                                                                                     \
    {                                                                                                          \
        auto kern = dense_kernel_v3<DEG, PB, W, A>;                                                            \
        RN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));           \
        kern<<<grid, 256, smem, stream>>>(d_in, m->d_ref_wrapped, V, m->d_piece_off, m->d_breaks, m->d_pieces, \
                                          num_frames, K, (int)m->v_cols, (int)m->dense_pad, accumulate ? 1 : 0, a0,                     \
                                          d_alpha);                                                            \
    }
    if (wrap) {
        if (align16) RN_V3_LAUNCH(true, true) else RN_V3_LAUNCH(true, false)
    } else {
        if (align16) RN_V3_LAUNCH(false, true) else RN_V3_LAUNCH(false, false)
    }
#undef RN_V3_LAUNCH
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    return RN_OK;
}

template <int DEG>
static int launch_v3_deg(const rn_model* m, const double* d_in, bool wrap, bool accumulate, int64_t num_frames,
                         double* d_alpha, cudaStream_t stream) {
    const int pb = m->dense_max_pieces - 1;
    if (pb <= 0) return launch_v3_cfg<DEG, 0>(m, d_in, wrap, accumulate, num_frames, d_alpha, stream);
    if (pb <= 1) return launch_v3_cfg<DEG, 1>(m, d_in, wrap, accumulate, num_frames, d_alpha, stream);
    if (pb <= 3) return launch_v3_cfg<DEG, 3>(m, d_in, wrap, accumulate, num_frames, d_alpha, stream);
    return 1;
}

int launch_dense(const rn_model* m, const double* d_in, bool wrap, bool accumulate, int64_t num_frames,
                 double* d_alpha, cudaStream_t stream, const AlphaPeers* peers, bool* peers_done) {
    if (num_frames == 0) return RN_OK;
    int rc = 1;
    AlphaPeers fused = no_peers();
    if (peers) fused = *peers;
    if (peers_done) *peers_done = false;
    const int dense_version = g_dense_version.load(std::memory_order_relaxed);
    if (dense_version == 4 && m->tp_mode != 0 && m->tp_features <= 12) {
        switch (m->dense_degree) {
            case 1: rc = launch_tp_deg<1>(m, d_in, wrap, accumulate, num_frames, d_alpha, stream, fused); break;
            case 2: rc = launch_tp_deg<2>(m, d_in, wrap, accumulate, num_frames, d_alpha, stream, fused); break;
            case 3: rc = launch_tp_deg<3>(m, d_in, wrap, accumulate, num_frames, d_alpha, stream, fused); break;
            default: break;
        }
        if (rc == RN_OK && peers_done) *peers_done = true;  // the chained kernel stores to the peers itself
    }
    if (rc == 1 && dense_version >= 3) {
        switch (m->dense_degree) {
            case 0:
            case 1: rc = launch_v3_deg<1>(m, d_in, wrap, accumulate, num_frames, d_alpha, stream); break;
            case 2: rc = launch_v3_deg<2>(m, d_in, wrap, accumulate, num_frames, d_alpha, stream); break;
            case 3: rc = launch_v3_deg<3>(m, d_in, wrap, accumulate, num_frames, d_alpha, stream); break;
            default: break;
        }
    }
    if (rc == 1) rc = launch_dense_v1(m, d_in, wrap, accumulate, num_frames, d_alpha, stream);
    return rc;
}

}  // namespace rn

// Test / tuning hooks (not in the public header).
extern "C" void rn_debug_set_dense_config(int version, int variant) {
    // variant: bits 0-1 = A/B switches, bits 4-7 = ring slots of the chained-epilogue kernel (0 = default)
    const int stages = (variant >> 4) & 15;
    rn::g_dense_stages.store(stages, std::memory_order_relaxed);
    rn::g_dense_variant.store(variant & 3, std::memory_order_relaxed);
    rn::g_dense_version.store(version, std::memory_order_relaxed);
}
// 0 = whole frame tiles per CTA, 1 = automatic (default), 2 = always balance (frame tile, DOF tile) units
extern "C" void rn_debug_set_dense_split(int mode) { rn::g_dense_split.store(mode, std::memory_order_relaxed); }
