// Mask sweeps (SURVEY.md §8f row N3): several masked copies of one model evaluated on the same
// trajectory in one pass.
//
// The reference's masking workflow (InterpolationModel.get_masked_model,
// ramannoodle/pmodel/_interpolation.py:697-708; ARTModel.get_dof_indexes, pmodel/_art.py:335-365)
// builds G deep copies of a model that differ only in `mask` and runs calc_polarizabilities
// (`_interpolation.py:191-252`) once per copy, i.e. G passes over the (S,N,3) trajectory.  For
// models whose DOFs are all single-piece linear (every ARTModel) each copy collapses to
// alpha0_g + D.G_g, so the G copies are one contraction of the displacement rows with the stacked
// table [G_0 | G_1 | ...] (K x 9G): the trajectory is streamed and wrapped once, the FP64 tensor
// pipe does 9G columns per row instead of 9.
//
//   affine_sweep_kernel<KP,NT,WRAP,MASKED>   8 warps, one CTA per SM.  Frames arrive as 8-row
//       tiles of TMA bulk copies (same staging as affine_tma_kernel); every warp owns a K-slice
//       (8*KP elements) and keeps its DMMA B fragments of all NT 8-column tiles in registers
//       (up to 180 of the 255 registers); the NT accumulator chains per warp are independent.
//       Cross-warp partials go through a double-buffered smem block and are reduced at the head
//       of the next tile.  FP64-tensor-pipe bound (DMMA 2*K*8*NT flop per frame); measured
//       0.47-0.59 of the DMMA peak: the wrap (DADDs on the same pipe, in front of every DMMA
//       group of an in-order warp) and the per-tile reduction leave the pipe idle — two variants
//       that moved them to extra warps (setmaxnreg 232/40) were slower because DADDs of other
//       warps starve behind the DMMA stream.
//
// Spline models: masked copies share the projection onto the basis (rn_dense_sweep.cu: one
// dense_kernel_tp launch, the chained-DMMA epilogue once per mask).  Anything else is evaluated one
// model after the other on the resident positions; results agree to rounding either way.
#include <algorithm>

#include "rn_common.cuh"
#include "rn_device.cuh"

extern "C" int rn_calc_polarizabilities(const rn_model* model, const double* d_positions, int64_t num_frames,
                                        double* d_alpha_out, void* stream);

namespace rn {

constexpr int kSweepWarps = 8;
constexpr int kSweepMaxMasks = 4;  // per launch: 36 columns = NT 5 column tiles (B fragments fill the register file)
constexpr int kSweepMaxTiles = 5;

struct SweepTables {
    const double* g[kSweepMaxMasks];  // (g_rows, 9) affine tables of the masks of this launch
};

struct SweepOut {
    double* alpha[kSweepMaxMasks];
    double a0[8 * kSweepMaxTiles];  // constant term per stacked column
    int columns;                    // 9 * masks
};

// routed destinations of the masks of one launch (rn_calc_polarizabilities_sweep_routed)
struct SweepPeers {
    AlphaPeers mask[kSweepMaxMasks];
};

// stacked[e][c] = G_{c/9}[e][c%9] for c < columns, 0 in the padding columns
__global__ void sweep_stack_kernel(SweepTables tabs, int64_t rows, int columns, int padded, double* __restrict__ stacked) {
    const int64_t total = rows * padded;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = idx / padded;
        const int c = (int)(idx % padded);
        stacked[idx] = (c < columns) ? __ldg(tabs.g[c / 9] + e * 9 + c % 9) : 0.0;
    }
}

template <int NT>
struct SweepSmem {
    static constexpr int kRed = 8 * NT + 4;  // doubles per (warp, row) slot
};

// wrap_disp with the rounding decided on the bit pattern: for |d| < 1.5 the result is d - n with
// n in {-1, 0, +1} chosen exactly as ceil(d - 0.5) would (d == +0.5 stays, d == -0.5 becomes +0.5),
// which leaves two DADDs on the FP64 pipe the DMMAs occupy instead of three plus an FRND.
// `far` reports |d| >= 1.5 (or NaN/Inf): the caller then takes the general formula.
__device__ __forceinline__ double wrap_disp_sel(double pos, double ref, bool& far) {
    const double d = pos - ref;
    const int hi = __double2hiint(d);
    const int lo = __double2loint(d);
    const unsigned mag = (unsigned)hi & 0x7fffffffu;
    far = mag >= 0x3ff80000u;
    const bool up = (hi > 0x3fe00000) || (hi == 0x3fe00000 && lo != 0);  // d > 0.5
    const bool down = (hi < 0) && (mag >= 0x3fe00000u);                  // d <= -0.5
    const int nhi = up ? 0x3ff00000 : (down ? (int)0xbff00000 : 0);
    return d - __hiloint2double(nhi, 0);
}

// 8 warps, one CTA per SM (the B fragments of all column tiles fill the register file).
// ROUTED: every finished element is also stored to the ranks that own its row (plain peer stores).
template <int KP, int NT, bool WRAP, bool MASKED, bool ROUTED>
__global__ void __launch_bounds__(kSweepWarps * 32, 1)
    affine_sweep_kernel(const double* __restrict__ in, const double* __restrict__ ref,
                        const double* __restrict__ stacked, int64_t num_frames, int K, int row_stride,
                        int stage_doubles, int num_stages, SweepOut out, const __grid_constant__ SweepPeers peers) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int ROWS = 8;
    constexpr int RS = SweepSmem<NT>::kRed;
    constexpr int RED = kSweepWarps * ROWS * RS;
    constexpr int COLS = 8 * NT;
    constexpr int NCOLS = 9 * (NT - 1);  // NT = 3, 4, 5 column tiles <-> 2, 3, 4 masks
    constexpr int OUTPUTS = ROWS * NCOLS;
    double* stages = reinterpret_cast<double*>(smem_raw);
    const int slack = kSweepWarps * 8 * KP;
    double* red = stages + (size_t)num_stages * stage_doubles + slack;
    double* tab_ref = red + 2 * RED;                                  // [slack] wrapped reference positions
    double* tab_a0 = tab_ref + slack;                                 // [OUTPUTS] constant term per output
    double** tab_out = reinterpret_cast<double**>(tab_a0 + OUTPUTS);  // [OUTPUTS] row-0 address per output
    uint64_t* bars = reinterpret_cast<uint64_t*>(tab_out + OUTPUTS);
    const uint32_t full0 = smem_u32(bars);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t num_tiles = (num_frames + ROWS - 1) / ROWS;
    const uint32_t row_bytes = (uint32_t)K * 8u;

    if (threadIdx.x == 0) {
        for (int s = 0; s < num_stages; s++) mbar_init(full0 + 8 * s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async;" ::: "memory");
        for (int s = 0; s < num_stages; s++) {
            const int64_t tile = blockIdx.x + (int64_t)s * gridDim.x;
            if (tile < num_tiles) {
                const int64_t frame0 = tile * ROWS;
                const int rows = (int)min((int64_t)ROWS, num_frames - frame0);
                mbar_arrive_expect_tx(full0 + 8 * s, row_bytes * rows);
                const uint32_t dst0 = smem_u32(stages + (size_t)s * stage_doubles);
                for (int r = 0; r < rows; r++)
                    tma_bulk_g2s(dst0 + (uint32_t)(r * row_stride) * 8u, in + (frame0 + r) * (int64_t)K, row_bytes,
                                 full0 + 8 * s);
            }
        }
    }
    for (int e = threadIdx.x; e < slack; e += blockDim.x) {
        tab_ref[e] = (WRAP && e < K) ? __ldg(ref + e) : 0.0;
        stages[(size_t)num_stages * stage_doubles + e] = 0.0;  // fragment loads of the last row run into this tail
    }
    for (int idx = threadIdx.x; idx < OUTPUTS; idx += blockDim.x) {
        const int f = idx / NCOLS, c = idx - f * NCOLS;
        const int mask = c / 9, q = c - 9 * mask;
        tab_a0[idx] = out.a0[c];
        tab_out[idx] = out.alpha[mask] + f * 9 + q;
    }
    __syncthreads();

    const int g = lane >> 2, t = lane & 3;
    const int kbase = warp * 8 * KP + 2 * t;
    double b[NT][KP][2];
    uint32_t validmask = 0;
#pragma unroll
    for (int p = 0; p < KP; p++) {
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int e = kbase + 8 * p + h;
            if (e < K) validmask |= 1u << (2 * p + h);
#pragma unroll
            for (int n = 0; n < NT; n++) b[n][p][h] = __ldg(stacked + (int64_t)e * COLS + 8 * n + g);
        }
    }
    const double* my_ref = tab_ref + kbase;
    const int rowoff = g * row_stride + kbase;
    double* myred = red + ((size_t)warp * ROWS + g) * RS + 2 * t;

    // sums the partials of tile `tile` (iteration i) and stores the finished rows
    auto reduce_tile = [&](int64_t tile, int64_t i) {
        const double* rbuf = red + (size_t)(i & 1) * RED;
        const int valid = (int)min((int64_t)ROWS, num_frames - tile * ROWS) * NCOLS;
#pragma unroll
        for (int u = 0; u < (OUTPUTS + kSweepWarps * 32 - 1) / (kSweepWarps * 32); u++) {
            const int idx = threadIdx.x + u * kSweepWarps * 32;
            if (idx < valid) {
                const int f = idx / NCOLS, c = idx - f * NCOLS;
                const double* r = rbuf + (size_t)f * RS + c;
                double sum = 0;
#pragma unroll
                for (int w = 0; w < kSweepWarps; w++) sum += r[(size_t)w * ROWS * RS];
                const double value = sum + tab_a0[idx];
                tab_out[idx][tile * (int64_t)(ROWS * 9)] = value;
                if (ROUTED) {
                    const AlphaPeers& P = peers.mask[c / 9];
                    const int64_t frame = tile * ROWS + f;
                    const uint32_t owners = alpha_peer_mask(P, frame, 1);
                    const int64_t off = alpha_peer_offset(P, frame) + (c - 9 * (c / 9));
                    for (int p = 0; p < P.count; p++)
                        if (((owners >> p) & 1u) && P.ptr[p]) P.ptr[p][off] = value;
                }
            }
        }
    };

    int64_t i = 0;
    int64_t prev_tile = -1;
    for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, i++) {
        const int s = (int)(i % num_stages);
        // the previous tile's reduction does not depend on this tile: issued first so that its loads,
        // adds and stores overlap the wait for the tile and the head of the DMMA stream
        if (prev_tile >= 0) reduce_tile(prev_tile, i - 1);
        mbar_wait(full0 + 8 * s, (uint32_t)(i / num_stages) & 1);
        const double* base = stages + (size_t)s * stage_doubles + rowoff;
        double c0[NT], c1[NT];
#pragma unroll
        for (int n = 0; n < NT; n++) c0[n] = c1[n] = 0.0;
#pragma unroll
        for (int p = 0; p < KP; p++) {
            const double2 v = *reinterpret_cast<const double2*>(base + 8 * p);
            double a_lo = v.x, a_hi = v.y;
            if (WRAP) {
                const double2 rf = *reinterpret_cast<const double2*>(my_ref + 8 * p);
                bool far_lo, far_hi;
                const double w_lo = wrap_disp_sel(a_lo, rf.x, far_lo);
                const double w_hi = wrap_disp_sel(a_hi, rf.y, far_hi);
                if (__any_sync(0xffffffffu, far_lo || far_hi)) {  // positions outside [0,1): general formula
                    a_lo = wrap_disp(a_lo, rf.x);
                    a_hi = wrap_disp(a_hi, rf.y);
                } else {
                    a_lo = w_lo;
                    a_hi = w_hi;
                }
            }
            if (MASKED) {  // K is not a multiple of the warps' slices: elements past K belong to other rows
                a_lo = (validmask >> (2 * p)) & 1u ? a_lo : 0.0;
                a_hi = (validmask >> (2 * p + 1)) & 1u ? a_hi : 0.0;
            }
#pragma unroll
            for (int n = 0; n < NT; n++) dmma884(c0[n], c1[n], a_lo, b[n][p][0]);
#pragma unroll
            for (int n = 0; n < NT; n++) dmma884(c0[n], c1[n], a_hi, b[n][p][1]);
        }
        double* slot = myred + (size_t)(i & 1) * RED;
#pragma unroll
        for (int n = 0; n < NT; n++) *reinterpret_cast<double2*>(slot + 8 * n) = make_double2(c0[n], c1[n]);
        __syncthreads();  // partials visible; every warp is done reading stage s
        {
            const int64_t next = tile + (int64_t)num_stages * gridDim.x;
            if (next < num_tiles && lane == 0) {
                const int64_t frame0 = next * ROWS;
                const int rows = (int)min((int64_t)ROWS, num_frames - frame0);
                if (warp == 0) mbar_arrive_expect_tx(full0 + 8 * s, row_bytes * rows);
                const uint32_t dst0 = smem_u32(stages + (size_t)s * stage_doubles);
                for (int r = warp; r < rows; r += kSweepWarps)
                    tma_bulk_g2s(dst0 + (uint32_t)(r * row_stride) * 8u, in + (frame0 + r) * (int64_t)K, row_bytes,
                                 full0 + 8 * s);
            }
        }
        prev_tile = tile;
    }
    if (prev_tile >= 0) reduce_tile(prev_tile, i - 1);
}

struct SweepLayout {
    int row_stride;
    int stage_doubles;
    int stages;
    size_t bytes;
};

static SweepLayout sweep_layout(int K, int kp, int nt) {
    SweepLayout L;
    L.row_stride = K + (8 - K % 16 + 16) % 16;
    L.stage_doubles = 8 * L.row_stride;
    const int slack = kSweepWarps * 8 * kp;
    const size_t fixed = (size_t)slack * 8 + (size_t)2 * kSweepWarps * 8 * (8 * nt + 4) * 8 + (size_t)slack * 8 +
                         (size_t)2 * 8 * 9 * (nt - 1) * 8 + 8 * 8 + 64;
    int stages = 4;
    while (stages > 1 && fixed + (size_t)stages * L.stage_doubles * 8 > 227 * 1024) stages--;
    L.stages = stages;
    L.bytes = fixed + (size_t)stages * L.stage_doubles * 8;
    return L;
}

template <int KP, int NT, bool WRAP>
static int launch_sweep_cfg(const rn_model* m, const double* d_in, int64_t frames, const double* d_stacked,
                            const SweepOut& out, const SweepPeers* peers, cudaStream_t stream) {
    const int K = (int)m->dim;
    const SweepLayout L = sweep_layout(K, KP, NT);
    if (L.bytes > 227 * 1024) return 1;
    const bool masked = (K != kSweepWarps * 8 * KP);
    auto kern = peers ? (masked ? affine_sweep_kernel<KP, NT, WRAP, true, true> : affine_sweep_kernel<KP, NT, WRAP, false, true>)
                      : (masked ? affine_sweep_kernel<KP, NT, WRAP, true, false> : affine_sweep_kernel<KP, NT, WRAP, false, false>);
    RN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.bytes));
    const int64_t tiles = (frames + 7) / 8;
    const int grid = (int)std::min<int64_t>(tiles, (int64_t)m->sm_count);
    SweepPeers routed;
    if (peers) routed = *peers;
    else
        for (int r = 0; r < kSweepMaxMasks; r++) routed.mask[r] = no_peers();
    kern<<<grid, kSweepWarps * 32, L.bytes, stream>>>(d_in, WRAP ? m->d_ref_wrapped : m->d_zero_ref, d_stacked, frames, K,
                                                      L.row_stride, L.stage_doubles, L.stages, out, routed);
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    return RN_OK;
}

template <int KP, bool WRAP>
static int launch_sweep_nt(int nt, const rn_model* m, const double* d_in, int64_t frames, const double* d_stacked,
                           const SweepOut& out, const SweepPeers* peers, cudaStream_t stream) {
    switch (nt) {
        case 3: return launch_sweep_cfg<KP, 3, WRAP>(m, d_in, frames, d_stacked, out, peers, stream);
        case 4: return launch_sweep_cfg<KP, 4, WRAP>(m, d_in, frames, d_stacked, out, peers, stream);
        case 5: return launch_sweep_cfg<KP, 5, WRAP>(m, d_in, frames, d_stacked, out, peers, stream);
        default: return 1;
    }
}

static int launch_sweep(int nt, const rn_model* m, const double* d_in, int64_t frames, const double* d_stacked,
                        const SweepOut& out, const SweepPeers* peers, cudaStream_t stream) {
    switch (m->affine_kp) {
#define RN_SWEEP_CASE(KP) \
    case KP: return launch_sweep_nt<KP, true>(nt, m, d_in, frames, d_stacked, out, peers, stream);
        RN_SWEEP_CASE(1)
        RN_SWEEP_CASE(2)
        RN_SWEEP_CASE(3)
        RN_SWEEP_CASE(4)
        RN_SWEEP_CASE(5)
        RN_SWEEP_CASE(6)
        RN_SWEEP_CASE(7)
        RN_SWEEP_CASE(8)
        RN_SWEEP_CASE(9)
#undef RN_SWEEP_CASE
        default: return 1;
    }
}

static std::atomic<bool> g_sweep_fused{true};  // A/B switches (include/ramannoodle_b200_debug.h)
static std::atomic<int> g_sweep_min_run{3};

// models that the fused kernel can take together: purely affine, TMA-eligible, same structure
static bool sweep_compatible(const rn_model* a, const rn_model* b) {
    return a->device == b->device && a->dim == b->dim && a->g_rows == b->g_rows && a->affine_kp == b->affine_kp &&
           a->ref_hash == b->ref_hash;
}
static bool sweep_eligible(const rn_model* m, const double* d_in) {
    return m->num_dense == 0 && m->num_dofs > 0 && m->affine_kp >= 1 && m->affine_kp <= 9 && m->dim % 2 == 0 &&
           reinterpret_cast<uintptr_t>(d_in) % 16 == 0;
}

// Evaluates every model of `models` (masked copies of one model: same reference structure) on the
// same positions: d_alpha_outputs[g] (num_frames*9) receives model g's series.  Replaces G calls of
// InterpolationModel.calc_polarizabilities (pmodel/_interpolation.py:191-252) on get_masked_model
// copies (:697-708).  `routed` (null, or one entry per model): the final rows of model g also go to the
// ranks routed[g] names; the affine parts of mixed models are written locally first and only the
// finished sums are stored to the peers.
int sweep_eval(const rn_model* const* models, int num_models, const double* d_positions, int64_t num_frames,
               double* const* d_alpha_outputs, cudaStream_t s, const AlphaPeers* routed) {
    RN_CHECK_ARG(models != nullptr && num_models >= 1, "at least one model is required");
    RN_CHECK_ARG(d_alpha_outputs != nullptr, "output pointers are required");
    for (int g = 0; g < num_models; g++)
        RN_CHECK_ARG(models[g] != nullptr && d_alpha_outputs[g] != nullptr, "null model or output pointer");
    RN_CHECK_ARG(num_frames >= 0, "num_frames must be non-negative");
    if (num_frames == 0) return RN_OK;
    RN_CHECK_ARG(d_positions != nullptr, "null positions pointer");
    DeviceGuard guard(models[0]->device);
    if (!guard.ok) {
        set_error("cudaSetDevice(%d) failed", models[0]->device);
        return RN_ERR_CUDA;
    }
    int g = 0;
    while (g < num_models) {
        // longest run of fusable models starting at g (at most kSweepMaxMasks)
        int run = 1;
        if (g_sweep_fused && sweep_eligible(models[g], d_positions)) {
            while (g + run < num_models && run < kSweepMaxMasks && sweep_eligible(models[g + run], d_positions) &&
                   sweep_compatible(models[g], models[g + run]))
                run++;
        }
        // measured on B200 (tools/run_sweep.py, LLZO, 1M frames): two masks fused take 1.59 ms against
        // 1.51 ms for two single-model passes, three 1.87 vs 2.27 ms, four 2.27 vs 3.06 ms
        if (run >= g_sweep_min_run) {
            const rn_model* m = models[g];
            const int columns = 9 * run;
            const int nt = (columns + 7) / 8;
            SweepTables tabs;
            SweepOut out;
            SweepPeers peers;
            for (int c = 0; c < 8 * kSweepMaxTiles; c++) out.a0[c] = 0.0;
            for (int r = 0; r < kSweepMaxMasks; r++) {
                const rn_model* mr = models[g + std::min(r, run - 1)];
                tabs.g[r] = mr->d_g_frac;
                out.alpha[r] = d_alpha_outputs[g + std::min(r, run - 1)];
                peers.mask[r] = (routed && r < run) ? routed[g + r] : no_peers();
                if (r < run)
                    for (int q = 0; q < 9; q++) out.a0[9 * r + q] = mr->alpha0[q];
            }
            out.columns = columns;
            double* d_stacked = nullptr;
            const int64_t rows = m->g_rows;
            {
                // stream-ordered scratch for the stacked table: keep freed blocks in the device's default
                // pool across synchronisations (the default threshold of 0 returns them to the driver,
                // and every chunk of a host sweep would pay a fresh physical allocation)
                static bool pool_ready[64] = {false};
                if (m->device < 64 && !pool_ready[m->device]) {
                    cudaMemPool_t pool = nullptr;
                    if (cudaDeviceGetDefaultMemPool(&pool, m->device) == cudaSuccess) {
                        uint64_t keep = 64ull << 20;
                        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
                    }
                    cudaGetLastError();
                    pool_ready[m->device] = true;
                }
            }
            RN_CUDA(cudaMallocAsync((void**)&d_stacked, sizeof(double) * rows * 8 * nt, s));
            sweep_stack_kernel<<<(unsigned)std::min<int64_t>((rows * 8 * nt + 255) / 256, 1024), 256, 0, s>>>(
                tabs, rows, columns, 8 * nt, d_stacked);
            RN_LAUNCHED();
            int rc = launch_sweep(nt, m, d_positions, num_frames, d_stacked, out, routed ? &peers : nullptr, s);
            cudaError_t free_rc = cudaFreeAsync(d_stacked, s);
            if (rc != RN_OK && rc != 1) return rc;
            RN_CUDA(free_rc);
            if (rc == RN_OK) {
                g += run;
                continue;
            }
        }
        // spline models: masked copies of one model share the projection onto the basis (rn_dense_sweep.cu)
        if (g_sweep_fused && dense_sweep_eligible(models[g]) && reinterpret_cast<uintptr_t>(d_positions) % 8 == 0) {
            int drun = 1;
            while (g + drun < num_models && drun < 4 && dense_sweep_eligible(models[g + drun]) &&
                   dense_sweep_compatible(models[g], models[g + drun]))
                drun++;
            if (drun == 3) drun = 2;  // kernels exist for 2 and 4 masks
            if (drun >= 2) {
                const bool has_affine = models[g]->num_linear > 0;
                int rc = RN_OK;
                for (int r = 0; r < drun && rc == RN_OK && has_affine; r++)
                    rc = launch_affine(models[g + r], d_positions, true, num_frames, d_alpha_outputs[g + r], s);
                if (rc != RN_OK) return rc;
                rc = launch_dense_sweep(models + g, drun, d_positions, has_affine, num_frames, d_alpha_outputs + g, s,
                                        routed ? routed + g : nullptr);
                if (rc != RN_OK && rc != 1) return rc;
                if (rc == RN_OK) {
                    g += drun;
                    continue;
                }
            }
        }
        int rc = routed ? eval_with_peers(models[g], d_positions, num_frames, d_alpha_outputs[g], s, routed[g])
                        : rn_calc_polarizabilities(models[g], d_positions, num_frames, d_alpha_outputs[g], s);
        if (rc != RN_OK) return rc;
        g++;
    }
    return RN_OK;
}

int make_sweep_peers(int num_models, double* const* peer_series, int world, int64_t first_frame, int64_t period,
                     int64_t width, AlphaPeers* routed) {
    RN_CHECK_ARG(num_models >= 1 && num_models <= kMaxSweepModels, "1..64 models are required");
    RN_CHECK_ARG(peer_series != nullptr, "peer series pointers are required");
    for (int g = 0; g < num_models; g++) {
        const int rc = make_routed_peers(peer_series + (int64_t)g * world, world, first_frame, period, width, routed + g);
        if (rc != RN_OK) return rc;
    }
    return RN_OK;
}

}  // namespace rn

using namespace rn;

extern "C" int rn_calc_polarizabilities_sweep(const rn_model* const* models, int num_models, const double* d_positions,
                                              int64_t num_frames, double* const* d_alpha_outputs, void* stream) {
    return sweep_eval(models, num_models, d_positions, num_frames, d_alpha_outputs, static_cast<cudaStream_t>(stream),
                      nullptr);
}

extern "C" int rn_calc_polarizabilities_sweep_routed(const rn_model* const* models, int num_models,
                                                     const double* d_positions, int64_t num_frames,
                                                     double* const* d_alpha_outputs, double* const* peer_series,
                                                     int world, int64_t first_frame, int64_t period, int64_t width,
                                                     void* stream) {
    AlphaPeers routed[kMaxSweepModels];
    const int rc = make_sweep_peers(num_models, peer_series, world, first_frame, period, width, routed);
    if (rc != RN_OK) return rc;
    return sweep_eval(models, num_models, d_positions, num_frames, d_alpha_outputs, static_cast<cudaStream_t>(stream),
                      routed);
}

// test hook: 0 = always evaluate the models one after the other
extern "C" void rn_debug_set_sweep_fused(int on) { rn::g_sweep_fused.store(on != 0, std::memory_order_relaxed); }
// test hook: shortest run of models that is fused (2..4; default 3)
extern "C" void rn_debug_set_sweep_min_run(int run) { rn::g_sweep_min_run.store(run < 2 ? 2 : (run > 4 ? 4 : run), std::memory_order_relaxed); }
