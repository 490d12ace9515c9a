// dense_kernel_tp: warp-specialised DMMA projection + chained-DMMA spline epilogue (see rn_dense.cu
// for the description).  Shared by rn_dense.cu (one model, NG = 1) and rn_dense_sweep.cu (mask
// sweeps: NG masked copies of one model share the projection, the epilogue runs once per mask).
#pragma once

#include <type_traits>

#include "rn_device.cuh"

namespace rn {

constexpr int kJT2 = 64;      // DOFs per J tile
constexpr int kKC2 = 16;      // K elements per pipeline chunk
constexpr int kRS2 = 20;      // padded smem row stride (doubles): conflict-free fragment loads
constexpr int kStages2 = 4;
constexpr int kAmpStride = 65;  // doubles per frame row of the amplitude tile
constexpr int kTpStagesDefault = 0;  // automatic: tp_stages()

// Ring depth (measured on the bench shapes, tools/run_dense_cases.py): 7 slots (215 KB) for 16-byte copies;
// 6 when odd row lengths force the 8-byte cp.async.ca path, which wants some L1 left beside the ring.
inline int tp_stages(int requested, bool align16) {
    if (requested >= 4 && requested <= 7) return requested;
    return align16 ? 7 : 6;
}

// shared memory of dense_kernel_tp with `stages` ring slots (128-frame tiles)
inline size_t tp_smem_bytes(int stages) {
    return ((size_t)stages * (128 + kJT2) * kRS2) * sizeof(double) + 128;
}


__device__ __forceinline__ void mbar_init2(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive2(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait2(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}

// What differs between the NG masked copies of a model that one launch evaluates: the truncated-power
// coefficient tables (the weights 1 - mask_j are folded into them), the constants, the output series.
template <int NG>
struct TpMasks {
    const double* c8[NG];  // (Jd_pad, NF, 8) tensor components 0..7
    const double* c9[NG];  // (Jd_pad, NF)    tensor component 8
    double* alpha[NG];     // (S, 9)
    Alpha0 a0[NG];
};

// Extra destinations of the finished rows: NP = 1, one set for every mask (a single model: the fused
// all-gather / routed stores of rn_calc_polarizabilities_multi / _routed; a sweep: none), or NP = NG, one
// set per mask (rn_calc_polarizabilities_sweep_routed).
template <int NP>
struct TpPeers {
    AlphaPeers mask[NP];
};

// Chained-DMMA epilogue: the amplitude accumulators of the projection are turned, in registers,
// into truncated-power features that feed a second DMMA against the per-DOF coefficient table
// (the C fragment layout of m8n8k4 is, up to the k-permutation, an A fragment layout: lane (g,t)
// holds amplitudes of frame g for DOFs 2t and 2t+1).  No shared-memory round trip, no per-frame
// table walks: one coefficient fragment is shared by 32 frames of the warp.
template <int DEG, int NBK, bool FULL, bool WRAP, bool ALIGN16, int NG, int NP = 1>
__global__ void __launch_bounds__(384, 1)
    dense_kernel_tp(const double* __restrict__ in, const double* __restrict__ ref, const double* __restrict__ V,
                    const double* __restrict__ tp_x0, const double* __restrict__ tp_brk, int64_t num_frames, int K,
                    int Kv, int Jpad, int Jreal, int accumulate, int split, int stages, TpMasks<NG> mk, TpPeers<NP> peers) {
    constexpr int FT = 128;    // frames per tile: 8 MMA warps x 16
    constexpr int MMAW = 8;    // MMA warps (two per scheduler: one covers the other's LDS / barrier bubbles)
    constexpr int MTW = 2;     // 8-frame groups per MMA warp
    constexpr int PERB = FULL ? DEG + 1 : 1;  // features per break slot
    constexpr int NF = DEG + NBK * PERB;      // features per DOF
    constexpr int NBS = NBK > 0 ? NBK : 1;    // stride of the break table
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // `stages` ring slots (4 .. 7, tp_stages()): the copies run two chunks ahead; every further slot lets the
    // producers finish a chunk's displacements that much earlier than the MMA warps need it
    double* As = reinterpret_cast<double*>(smem_raw);          // [stages][FT][kRS2]
    double* Bs = As + (size_t)stages * FT * kRS2;              // [stages][kJT2][kRS2]
    uint64_t* bars = reinterpret_cast<uint64_t*>(Bs + (size_t)stages * kJT2 * kRS2);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + stages);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int chunks = Kv / kKC2;
    const int jtiles = Jpad / kJT2;
    const int64_t num_tiles = (num_frames + FT - 1) / FT;
    // `split`: bit 0 = unit-balanced schedule; bits 1-2 = A/B variants (rn_debug_set_dense_config)
    const bool fast_wrap = (split & 2) != 0, keep_padding = (split & 4) != 0;
    split &= 1;
    // Work units are (frame tile, DOF tile) pairs; CTA b owns the contiguous range [u0, u1).  Normally
    // the ranges are whole frame tiles.  With `split` (few frame tiles per SM: short trajectories)
    // they are balanced to the unit, a frame tile shared by two CTAs is finished with atomic adds
    // into rows the caller pre-filled, and no SM idles through a partial last wave.
    int64_t u0, u1;
    if (split) {
        const int64_t units = num_tiles * jtiles;
        u0 = units * blockIdx.x / gridDim.x;
        u1 = units * (blockIdx.x + 1) / gridDim.x;
    } else {
        u0 = (num_tiles * blockIdx.x / gridDim.x) * jtiles;
        u1 = (num_tiles * (blockIdx.x + 1) / gridDim.x) * jtiles;
    }
    const int64_t tile_begin = u0 / jtiles, tile_end = (u1 + jtiles - 1) / jtiles;

    if (threadIdx.x == 0) {
        for (int s = 0; s < stages; s++) {
            mbar_init2(full0 + 8 * s, 128);  // every producer thread arrives after its wrap items
            mbar_init2(empty0 + 8 * s, MMAW);  // one arrival per MMA warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp >= MMAW) {
        // =========================== producers (128 threads) ===========================
        const int ptid = threadIdx.x - MMAW * 32;
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

        // ring positions (running over all tiles): slot and round parity of the next chunk to issue / to wrap
        uint32_t is_st = 0, is_round = 0, wr_st = 0;
        for (int64_t tile = tile_begin; tile < tile_end; tile++) {
            const int64_t frame0 = tile * FT;
            const int jt_lo = (int)(max(u0, tile * jtiles) - tile * jtiles);
            const int jt_hi = (int)(min(u1, (tile + 1) * jtiles) - tile * jtiles);
            const int64_t total = (int64_t)(jt_hi - jt_lo) * chunks;
            const double* a_src_row[A_ITEMS];
#pragma unroll
            for (int r = 0; r < A_ITEMS; r++) {
                const int64_t frame = frame0 + a_row0 + r * A_ROWSTEP;
                a_src_row[r] = (frame < num_frames) ? in + frame * (int64_t)K + a_seg * A_ELEMS : nullptr;
            }
            int is_kc = 0, is_jt = jt_lo;
            auto issue = [&]() {
                if (is_jt < jt_hi) {
                    const uint32_t st = is_st;
                    if (is_round > 0) {  // the slot's previous occupant (one round earlier) must have been consumed
                        mbar_wait2(empty0 + 8 * st, (is_round - 1) & 1);
                    }
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
                    if (++is_st == (uint32_t)stages) {
                        is_st = 0;
                        ++is_round;
                    }
                }
                cp_async_commit();
            };
            issue();
            issue();
            int wr_kc = 0;
            // reference positions of the chunk to wrap: fetched one iteration ahead (off the critical path)
            double2 rf_next = make_double2(0.0, 0.0);
            if (WRAP) rf_next = __ldg(reinterpret_cast<const double2*>(ref + w_seg * 2));
            for (int64_t c = 0; c < total; c++) {
                const double2 rf = rf_next;
                if (WRAP) {
                    const int nkc = (wr_kc + 1 == chunks) ? 0 : wr_kc + 1;
                    rf_next = __ldg(reinterpret_cast<const double2*>(ref + nkc * kKC2 + w_seg * 2));
                }
                issue();             // chunk c+2
                cp_async_wait<2>();  // this thread's copies of chunk c have landed
                asm volatile("bar.sync 1, 128;" ::: "memory");  // ... and every producer's
                const uint32_t st = wr_st;
                if (WRAP) {
                    double* a = As + (size_t)st * FT * kRS2 + w_row0 * kRS2 + w_seg * 2;
#pragma unroll
                    for (int r = 0; r < FT / 16; r++) {
                        double2* p = reinterpret_cast<double2*>(a + r * 16 * kRS2);
                        double2 v = *p;
                        v.x = fast_wrap ? wrap_disp_fast(v.x, rf.x) : wrap_disp(v.x, rf.x);
                        v.y = fast_wrap ? wrap_disp_fast(v.y, rf.y) : wrap_disp(v.y, rf.y);
                        *p = v;
                    }
                    if (++wr_kc == chunks) wr_kc = 0;
                }
                mbar_arrive2(full0 + 8 * st);  // release: this thread's stage writes are visible to waiters
                if (++wr_st == (uint32_t)stages) wr_st = 0;
            }
            cp_async_wait<0>();
        }
        return;
    }

    // =============================== MMA warps (128 threads) ===============================
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp;  // frames 16*wm .. 16*wm+15
    uint32_t co_st = 0, co_round = 0;  // ring slot and round parity of the next chunk to consume
    // DOF padding is not computed: the last DOF tile runs only the 8-DOF column groups that hold real DOFs
    const int nt_last = keep_padding ? 8 : (Jreal - (jtiles - 1) * kJT2 + 7) >> 3;
    for (int64_t tile = tile_begin; tile < tile_end; tile++) {
        const int64_t frame0 = tile * FT;
        const int jt_lo = (int)(max(u0, tile * jtiles) - tile * jtiles);
        const int jt_hi = (int)(min(u1, (tile + 1) * jtiles) - tile * jtiles);
        const int64_t total = (int64_t)(jt_hi - jt_lo) * chunks;
        const bool shared_tile = (jt_lo != 0) || (jt_hi != jtiles);  // other CTAs add to the same rows
        double out[NG][MTW][2], o9[NG][MTW];
#pragma unroll
        for (int m = 0; m < NG; m++)
#pragma unroll
            for (int mt = 0; mt < MTW; mt++) out[m][mt][0] = out[m][mt][1] = o9[m][mt] = 0.0;
        double acc[MTW][8][2];
        int kc = 0, jt = jt_lo;
        for (int64_t c = 0; c < total; c++) {
            if (kc == 0) {
#pragma unroll
                for (int mt = 0; mt < MTW; mt++)
#pragma unroll
                    for (int nt = 0; nt < 8; nt++) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
            }
            const uint32_t st = co_st;
            mbar_wait2(full0 + 8 * st, co_round & 1);
            const double* a_src = As + (size_t)st * FT * kRS2 + (wm * 8 * MTW + g) * kRS2 + t;
            const double* b_src = Bs + (size_t)st * kJT2 * kRS2 + g * kRS2 + t;
            const int ntc = (jt == jtiles - 1) ? nt_last : 8;
            // One copy of the chunk's MMA loop per number of live 8-DOF column groups (the last DOF tile skips
            // its groups of pure padding): every copy is unrolled without predicates — a predicated DMMA costs
            // a WARPSYNC and its issue slot.  K padding (< one 16-element chunk) is computed: zeros.
            auto mma_chunk = [&](auto groups) {
                constexpr int NTC = decltype(groups)::value;
                double af[2][MTW], bf[2][NTC];
#pragma unroll
                for (int mt = 0; mt < MTW; mt++) af[0][mt] = a_src[mt * 8 * kRS2];
#pragma unroll
                for (int nt = 0; nt < NTC; nt++) bf[0][nt] = b_src[nt * 8 * kRS2];
#pragma unroll
                for (int s = 0; s < kKC2 / 4; s++) {
                    const int cur = s & 1, nxt = cur ^ 1;
                    if (s + 1 < kKC2 / 4) {
#pragma unroll
                        for (int mt = 0; mt < MTW; mt++) af[nxt][mt] = a_src[mt * 8 * kRS2 + 4 * (s + 1)];
#pragma unroll
                        for (int nt = 0; nt < NTC; nt++) bf[nxt][nt] = b_src[nt * 8 * kRS2 + 4 * (s + 1)];
                    }
#pragma unroll
                    for (int nt = 0; nt < NTC; nt++)
#pragma unroll
                        for (int mt = 0; mt < MTW; mt++)
                            dmma884(acc[mt][nt][0], acc[mt][nt][1], af[cur][mt], bf[cur][nt]);
                }
            };
            switch (ntc) {
                case 8: mma_chunk(std::integral_constant<int, 8>{}); break;
                case 7: mma_chunk(std::integral_constant<int, 7>{}); break;
                case 6: mma_chunk(std::integral_constant<int, 6>{}); break;
                case 5: mma_chunk(std::integral_constant<int, 5>{}); break;
                case 4: mma_chunk(std::integral_constant<int, 4>{}); break;
                case 3: mma_chunk(std::integral_constant<int, 3>{}); break;
                case 2: mma_chunk(std::integral_constant<int, 2>{}); break;
                default: mma_chunk(std::integral_constant<int, 1>{}); break;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive2(empty0 + 8 * st);  // stage may be refilled
            if (++co_st == (uint32_t)stages) {
                co_st = 0;
                ++co_round;
            }
            const bool last_chunk = (kc == chunks - 1);
            const int jt_now = jt;
            if (++kc == chunks) {
                kc = 0;
                ++jt;
            }
            if (last_chunk) {
                // ---- chained-DMMA epilogue of this DOF tile ----
#pragma unroll
                for (int nt = 0; nt < 8; nt++) {
                    if (nt >= ntc) continue;  // column groups of pure padding
#pragma unroll
                    for (int c = 0; c < 2; c++) {
                        const int jl = jt_now * kJT2 + nt * 8 + 2 * t + c;  // DOF in this lane's k-slot
                        const int jb = jt_now * kJT2 + nt * 8 + 2 * g + c;  // n.b. B rows are indexed by k-slot = lane&3
                        (void)jb;
                        const double x0 = __ldg(tp_x0 + jl);
                        double brk[NBS];
#pragma unroll
                        for (int i = 0; i < NBK; i++) brk[i] = __ldg(tp_brk + (int64_t)jl * NBS + i);
                        // features of this lane's two frames (one per 8-frame group), shared by all masks
                        double feat[MTW][NF];
#pragma unroll
                        for (int mt = 0; mt < MTW; mt++) {
                            const double x = acc[mt][nt][c];
                            const double u = x - x0;
                            double pw = u;
#pragma unroll
                            for (int mm = 1; mm <= DEG; mm++) {
                                feat[mt][mm - 1] = pw;
                                if (mm < DEG) pw *= u;
                            }
#pragma unroll
                            for (int i = 0; i < NBK; i++) {
                                const double d = x - brk[i];
                                const double v = fmax(d, 0.0);
                                if (FULL) {
                                    double pv = (d >= 0.0) ? 1.0 : 0.0;  // (x - b)_+^0
#pragma unroll
                                    for (int mm = 0; mm <= DEG; mm++) {
                                        feat[mt][DEG + i * PERB + mm] = pv;
                                        pv = (mm == 0) ? v : pv * v;
                                    }
                                } else {
                                    double pv = v;
#pragma unroll
                                    for (int mm = 1; mm < DEG; mm++) pv *= v;
                                    feat[mt][DEG + i] = pv;
                                }
                            }
                        }
#pragma unroll
                        for (int m = 0; m < NG; m++) {
                            // coefficient fragments: B[k = lane&3][n = lane>>2] = c8[DOF of k-slot][f][n]
                            double b2[NF], c9[NF];
#pragma unroll
                            for (int f = 0; f < NF; f++) {
                                b2[f] = __ldg(mk.c8[m] + ((int64_t)jl * NF + f) * 8 + g);
                                c9[f] = __ldg(mk.c9[m] + (int64_t)jl * NF + f);
                            }
#pragma unroll
                            for (int mt = 0; mt < MTW; mt++) {
#pragma unroll
                                for (int f = 0; f < NF; f++) {
                                    dmma884(out[m][mt][0], out[m][mt][1], feat[mt][f], b2[f]);
                                    o9[m][mt] = fma(feat[mt][f], c9[f], o9[m][mt]);
                                }
                            }
                        }
                    }
                }
            }
        }
        // ---- store: lane (g,t) holds components 2t, 2t+1 of frames 8*mt+g; component 8 is summed over t ----
#pragma unroll
        for (int m = 0; m < NG; m++) {
            const Alpha0& a0 = mk.a0[m];
            double* alpha = mk.alpha[m];
#pragma unroll
            for (int mt = 0; mt < MTW; mt++) {
                double v9 = o9[m][mt];
                v9 += __shfl_xor_sync(0xffffffffu, v9, 1);
                v9 += __shfl_xor_sync(0xffffffffu, v9, 2);
                const int64_t frame = frame0 + wm * 8 * MTW + mt * 8 + g;
                if (frame < num_frames && shared_tile) {
                    // split schedule: the rows were pre-filled by the caller; the CTA holding DOF tile 0 adds
                    // the constant on top of its partial sum
                    double* dst = alpha + frame * 9;
                    const bool first = (jt_lo == 0);
                    atomicAdd(dst + 2 * t, out[m][mt][0] + (first ? a0.v[2 * t] : 0.0));
                    atomicAdd(dst + 2 * t + 1, out[m][mt][1] + (first ? a0.v[2 * t + 1] : 0.0));
                    if (t == 0) atomicAdd(dst + 8, v9 + (first ? a0.v[8] : 0.0));
                } else if (frame < num_frames) {
                    double* dst = alpha + frame * 9;
                    // a0 holds what must be added on top of the running value (see launch_tp_cfg)
                    const double b0 = (accumulate ? dst[2 * t] : 0.0) + a0.v[2 * t];
                    const double b1 = (accumulate ? dst[2 * t + 1] : 0.0) + a0.v[2 * t + 1];
                    const double r0 = out[m][mt][0] + b0, r1 = out[m][mt][1] + b1;
                    const double r8 = v9 + ((accumulate ? dst[8] : 0.0) + a0.v[8]);
                    dst[2 * t] = r0;
                    dst[2 * t + 1] = r1;
                    if (t == 0) dst[8] = r8;
                    // fused all-gather: the same row goes to every peer GPU's series over NVLink
                    const AlphaPeers& P = peers.mask[NP == 1 ? 0 : m];
                    if (P.count > 0) {
                        const uint32_t mask = alpha_peer_mask(P, frame, 1);
                        const int64_t off = alpha_peer_offset(P, frame);
                        for (int p = 0; p < P.count; p++) {
                            if (!((mask >> p) & 1u) || !P.ptr[p]) continue;
                            double* pd = P.ptr[p] + off;
                            pd[2 * t] = r0;
                            pd[2 * t + 1] = r1;
                            if (t == 0) pd[8] = r8;
                        }
                    }
                }
            }
        }
    }
}

}  // namespace rn
