// Trajectory analyses on the spectrum plan's transform (sm_100a): the vibrational density of states (rn_vdos), the
// velocity spectra projected on vectors (rn_projected_vdos) and the mean squared displacement (rn_msd).
#include <algorithm>
#include <cmath>

#include "rn_spectrum_plan.cuh"

namespace rn {

using fft::cmul;

// ---- vibrational density of states (rn_vdos) -------------------------------------------------------
// The VDOS of a group is sum_{atoms i} w_i sum_c calc_signal_spectrum(v_ic) with v the minimum-image velocity
// (d @ lattice) / dt.  A slot holds two memberships a, b of one group: its six real signals sqrt(w) v_c of a
// and of b packed as z_c = (x_a + i x_b)_c are the three sequences of one window of a batched plan, so the
// identity of combine_md_kernel gives the slot's term (P[k] + P[M-k]) / (4 L^2) + E/2 unchanged.

struct VdosSlot {
    int atom[2];      // -1: the zero signal that pads a group of odd size
    double sqrtw[2];  // sqrt(weight) of each membership
};

// frames first .. first + avail - 1 of the slot's two atoms into rows (6 per frame, `frames` rows); atom -1 and
// frames past avail read as zero.  The stride is blockDim.x: with the constant block size the MSD pack compiles to
// slower code (measured on a B200: +4 % MSD time).
__device__ __forceinline__ void stage_slot_frames(const double* pos, int64_t num_atoms, const VdosSlot& slot,
                                                  int64_t first, int64_t avail, double* rows, int frames) {
    const int64_t frame_stride = 3 * num_atoms;
    for (int e = threadIdx.x; e < frames * 6; e += blockDim.x) {
        const int f = e / 6, j = e - 6 * (e / 6);
        const int atom = j < 3 ? slot.atom[0] : slot.atom[1];
        rows[e] = (f < avail && atom >= 0) ? __ldg(pos + (first + f) * frame_stride + 3 * atom + (j < 3 ? j : j - 3))
                                           : 0.0;
    }
}

struct VdosPackParams {
    const double* pos;   // (S,N,3) fractional, wrapped
    int64_t num_atoms;
    int64_t M, Lh;
    const VdosSlot* slots;  // the chunk's slots: blockIdx.y numbers them
    double lattice[9];      // rows are lattice vectors
    double inv_dt;
    double2* dst;           // (3 nb, Lh) work buffer
    double* epart;          // (nb, gridDim.x + 1) partials, then their sum
    unsigned int* ticket;   // nb tickets
};

// frames n .. n+256 of the slot's two atoms staged in shared memory; per difference n: the minimum image
// wrap_disp(x[n+1], x[n]) of each component, times the lattice and sqrt(w)/dt, chirp pre-multiply; the
// slot's energy is summed with its own partials and ticket, as the windowed pack does.
__global__ void __launch_bounds__(kPackThreads) pack_velocity_kernel(const __grid_constant__ VdosPackParams P) {
    __shared__ double rows[(kPackThreads + 1) * 6];
    __shared__ double red[kPackThreads / 32];
    const VdosSlot slot = P.slots[blockIdx.y];
    double2* dst = P.dst + (int64_t)blockIdx.y * 3 * P.Lh;
    const int64_t first = (int64_t)blockIdx.x * kPackThreads;
    const int64_t avail = min((int64_t)kPackThreads + 1, P.M + 1 - first);  // frames first .. first+avail-1
    stage_slot_frames(P.pos, P.num_atoms, slot, first, avail, rows, kPackThreads + 1);
    __syncthreads();
    const int64_t n = first + threadIdx.x;
    double energy = 0.0;
    if (n < P.M) {
        const double* r0 = rows + threadIdx.x * 6;
        const double* r1 = r0 + 6;
        double2 z[3];
#pragma unroll
        for (int m = 0; m < 2; m++) {
            const double d0 = wrap_disp(r1[3 * m], r0[3 * m]);
            const double d1 = wrap_disp(r1[3 * m + 1], r0[3 * m + 1]);
            const double d2 = wrap_disp(r1[3 * m + 2], r0[3 * m + 2]);
            const double s = slot.sqrtw[m] * P.inv_dt;
#pragma unroll
            for (int c = 0; c < 3; c++) {
                const double v = (d0 * P.lattice[c] + d1 * P.lattice[3 + c] + d2 * P.lattice[6 + c]) * s;
                if (m == 0) z[c].x = v;
                else z[c].y = v;
            }
        }
        energy = (z[0].x * z[0].x + z[0].y * z[0].y) + (z[1].x * z[1].x + z[1].y * z[1].y) +
                 (z[2].x * z[2].x + z[2].y * z[2].y);
        const double2 c = chirp(n, P.M);
#pragma unroll
        for (int s = 0; s < 3; s++) dst[(int64_t)s * P.Lh + n] = cmul(z[s], c);
    }
    const double total = block_sum(energy, red);
    publish_energy(total, P.epart + (int64_t)blockIdx.y * (gridDim.x + 1), P.ticket + blockIdx.y, red);
}

// Rows g_lo .. g_lo + num_groups - 1 of int_out (G, points), for the slots first .. first + nb - 1 of this chunk:
// row g is the sum, over its slots in slot order, of (P[k] + P[M-k]) scale + E/2.  A group's first slot writes
// the row; slots of later chunks read it and keep adding one at a time, so the sequence of additions is the
// same whatever the chunking.  power: (3 nb, M); group_slots: (G+1,) slot offsets of the groups.
__global__ void __launch_bounds__(256) combine_groups_kernel(const double* __restrict__ power,
                                                             const double* __restrict__ epart, int64_t epart_stride,
                                                             const int64_t* __restrict__ group_slots, int64_t first,
                                                             int64_t nb, int64_t g_lo, int64_t num_groups, int64_t M,
                                                             double scale, int64_t points, double dt,
                                                             double* __restrict__ wn_out, double* __restrict__ int_out) {
    for (int64_t g = g_lo + blockIdx.y; g < g_lo + num_groups; g += gridDim.y) {
        const int64_t begin = group_slots[g];
        const int64_t s0 = max(begin, first), s1 = min(group_slots[g + 1], first + nb);
        double* row = int_out + g * points;
        for (int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; o < points;
             o += (int64_t)gridDim.x * blockDim.x) {
            const int64_t k = o + 1;
            double acc = begin < first ? row[o] : 0.0;
#pragma unroll 1
            for (int64_t slot = s0; slot < s1; slot++) {
                const double* pw = power + (slot - first) * 3 * M;
                double sum = 0.0;
#pragma unroll
                for (int s = 0; s < 3; s++) sum += pw[(int64_t)s * M + k] + pw[(int64_t)s * M + (M - k)];
                const double term = __fma_rn(sum, scale, 0.5 * epart[(slot - first) * epart_stride]);
                acc = slot == begin ? term : __dadd_rn(acc, term);
            }
            row[o] = acc;
        }
    }
    if (wn_out && blockIdx.y == 0) write_wavenumbers(wn_out, points, M, dt);
}

// ---- projected VDOS (rn_projected_vdos) ---------------------------------------------------------------
// Row k is calc_signal_spectrum(q_k) of the mode velocity q_k[n] = sum_{i,c} vectors[k,i,c] v[n,i,c].  With the
// lattice and 1/dt folded into the projection matrix B[(i,a), k] = sum_c lattice[a,c] vectors[k,i,c] / dt,
// q_k[n] = sum_{(i,a)} wrap(x[n+1] - x[n])_(i,a) B[(i,a), k]: a (frames x 3N) x (3N x modes) product on the FP64
// tensor pipe whose left factor is formed from the positions as they stream in.  Modes 2j and 2j+1 of a chunk
// travel as sequence j = q_2j + i q_2j+1 of the work buffer; the real signals are separated after the transform.

constexpr int kPvFT = 128;     // differences per frame tile: 8 MMA warps x 16
constexpr int kPvNT = 64;      // modes per mode tile (blockIdx.x)
constexpr int kPvKC = 16;      // coordinates per pipeline chunk
constexpr int kPvRS = 20;      // padded smem row stride (doubles): conflict-free fragment loads
constexpr int kPvStages = 4;   // ring slots; the copies run two chunks ahead
constexpr int kPvThreads = 384;  // 8 MMA warps, then 4 producer warps
constexpr size_t kPvSmemBytes = (size_t)kPvStages * ((kPvFT + 1) + kPvNT) * kPvRS * sizeof(double) +
                                2 * kPvStages * sizeof(uint64_t);

struct ProjParams {
    const double* pos;     // (S,N,3) fractional, wrapped
    int64_t cols;          // 3N
    int64_t M, Lh;
    const double* bt;      // the chunk's rows of the transposed projection matrix: (modes, rpad), zero padded
    int rpad;              // 3N rounded up to kPvKC
    int nseq;              // 3 nb sequences of the chunk's work buffer
    int64_t tiles;         // frame tiles: ceil(M / kPvFT)
    double2* dst;          // (3 nb, Lh) work buffer
    double* epart;         // (gridDim.x kPvNT, tiles) energy of every mode in every frame tile
    double* energy;        // (gridDim.x kPvNT) their sums
    unsigned int* ticket;  // zero between launches
};

__device__ __forceinline__ void mbar_arrive_cta(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// CTA (x, y): mode tile x of the chunk, a contiguous range of frame tiles.  Producers copy frames
// n0 .. n0 + kPvFT (one halo frame) and kPvKC coordinates per ring slot with cp.async, replace them in place by
// the minimum-image steps wrap_disp(x[n+1], x[n]) (the function pack_velocity_kernel uses) and release the slot;
// the MMA warps contract it with the slot's kPvNT x kPvKC block of B.  Epilogue per frame tile: chirp
// pre-multiply, store of the packed pairs, and the tile's energy of every mode (a fixed tree, no value atomics);
// the CTA that finishes last sums every mode's tiles in tile order, so the energies do not depend on the grid.
template <bool ALIGN16>
__global__ void __launch_bounds__(kPvThreads, 1) project_velocity_kernel(const __grid_constant__ ProjParams P) {
    extern __shared__ __align__(16) unsigned char pv_smem[];  // 16: the module's other kernels keep their layout
    double* As = reinterpret_cast<double*>(pv_smem);                 // [stages][kPvFT + 1][kPvRS]
    double* Bs = As + (size_t)kPvStages * (kPvFT + 1) * kPvRS;      // [stages][kPvNT][kPvRS]
    uint64_t* bars = reinterpret_cast<uint64_t*>(Bs + (size_t)kPvStages * kPvNT * kPvRS);
    __shared__ double red[8][kPvNT];
    __shared__ bool last;
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + kPvStages);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int chunks = P.rpad / kPvKC;
    const int64_t tile_begin = P.tiles * blockIdx.y / gridDim.y, tile_end = P.tiles * (blockIdx.y + 1) / gridDim.y;
    const int64_t total = (tile_end - tile_begin) * chunks;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kPvStages; s++) {
            mbar_init(full0 + 8 * s, 128);  // every producer thread arrives after its steps
            mbar_init(empty0 + 8 * s, 8);   // one arrival per MMA warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp >= 8) {
        // =========================== producers (128 threads) ===========================
        const int ptid = threadIdx.x - 256;
        constexpr int SEGS = ALIGN16 ? kPvKC / 2 : kPvKC, ELEMS = ALIGN16 ? 2 : 1;
        constexpr int A_ITEMS = ((kPvFT + 1) * SEGS + 127) / 128;
        const int w_col = ptid & 15, w_row0 = (ptid >> 4) * 16;  // the 16 steps this thread forms
        const double* bt_src = P.bt + (int64_t)blockIdx.x * kPvNT * P.rpad;
        uint32_t is_st = 0, is_round = 0, wr_st = 0;
        int64_t is_tile = tile_begin;
        int is_kc = 0;
        auto issue = [&]() {
            if (is_tile < tile_end) {
                const uint32_t st = is_st;
                if (is_round > 0) mbar_wait(empty0 + 8 * st, (is_round - 1) & 1);  // consumed one round earlier
                const int64_t tile = is_tile;
                const int kc = is_kc;
                const uint32_t a_dst = smem_u32(As + (size_t)st * (kPvFT + 1) * kPvRS);
#pragma unroll
                for (int i = 0; i < A_ITEMS; i++) {
                    const int e = ptid + 128 * i;
                    const int row = e / SEGS, seg = e % SEGS;
                    if (row <= kPvFT) {
                        const int64_t frame = tile * kPvFT + row;
                        const int64_t col = (int64_t)kc * kPvKC + seg * ELEMS;
                        const bool ok = frame <= P.M && col < P.cols;  // zero fill past the last frame / coordinate
                        const double* src = ok ? P.pos + frame * P.cols + col : P.pos;
                        const uint32_t d = a_dst + (uint32_t)(row * kPvRS + seg * ELEMS) * 8u;
                        if (ALIGN16) cp_async_16(d, src, ok ? 16 : 0);
                        else cp_async_8(d, src, ok ? 8 : 0);
                    }
                }
                const uint32_t b_dst = smem_u32(Bs + (size_t)st * kPvNT * kPvRS);
#pragma unroll
                for (int i = 0; i < (kPvNT * 8) / 128; i++) {
                    const int e = ptid + 128 * i;
                    const int row = e >> 3, seg = e & 7;
                    cp_async_16(b_dst + (uint32_t)(row * kPvRS + seg * 2) * 8u,
                                bt_src + (int64_t)row * P.rpad + kc * kPvKC + seg * 2, 16);
                }
                if (++is_kc == chunks) {
                    is_kc = 0;
                    ++is_tile;
                }
                if (++is_st == (uint32_t)kPvStages) {
                    is_st = 0;
                    ++is_round;
                }
            }
            cp_async_commit();
        };
        issue();
        issue();
        for (int64_t c = 0; c < total; c++) {
            issue();             // item c+2
            cp_async_wait<2>();  // this thread's copies of item c have landed
            asm volatile("bar.sync 1, 128;" ::: "memory");  // ... and every producer's
            double* a = As + (size_t)wr_st * (kPvFT + 1) * kPvRS + w_col;
            const double halo = a[(w_row0 + 16) * kPvRS];  // the next thread's first frame, before it is replaced
            asm volatile("bar.sync 1, 128;" ::: "memory");
            double prev = a[w_row0 * kPvRS];
#pragma unroll
            for (int r = 0; r < 16; r++) {
                const double next = r < 15 ? a[(w_row0 + r + 1) * kPvRS] : halo;
                a[(w_row0 + r) * kPvRS] = wrap_disp(next, prev);
                prev = next;
            }
            mbar_arrive_cta(full0 + 8 * wr_st);  // release: this thread's steps are visible to the MMA warps
            if (++wr_st == (uint32_t)kPvStages) wr_st = 0;
        }
        cp_async_wait<0>();
        return;
    }

    // =============================== MMA warps (256 threads) ===============================
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp;  // differences 16 wm .. 16 wm + 15 of a tile
    const int seq0 = blockIdx.x * (kPvNT / 2);
    uint32_t co_st = 0, co_round = 0;
    for (int64_t tile = tile_begin; tile < tile_end; tile++) {
        double acc[2][8][2];
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
            for (int nt = 0; nt < 8; nt++) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
        for (int kc = 0; kc < chunks; kc++) {
            const uint32_t st = co_st;
            mbar_wait(full0 + 8 * st, co_round & 1);
            const double* a_src = As + (size_t)st * (kPvFT + 1) * kPvRS + (wm * 16 + g) * kPvRS + t;
            const double* b_src = Bs + (size_t)st * kPvNT * kPvRS + g * kPvRS + t;
#pragma unroll
            for (int s = 0; s < kPvKC / 4; s++) {
                double af[2], bf[8];
#pragma unroll
                for (int mt = 0; mt < 2; mt++) af[mt] = a_src[mt * 8 * kPvRS + 4 * s];
#pragma unroll
                for (int nt = 0; nt < 8; nt++) bf[nt] = b_src[nt * 8 * kPvRS + 4 * s];
#pragma unroll
                for (int nt = 0; nt < 8; nt++)
#pragma unroll
                    for (int mt = 0; mt < 2; mt++) dmma884(acc[mt][nt][0], acc[mt][nt][1], af[mt], bf[nt]);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive_cta(empty0 + 8 * st);  // slot may be refilled
            if (++co_st == (uint32_t)kPvStages) {
                co_st = 0;
                ++co_round;
            }
        }
        // lane (g, t) holds q of difference 8 mt + g for modes 8 nt + 2t and 8 nt + 2t + 1: one packed value
        double e[8][2];
#pragma unroll
        for (int nt = 0; nt < 8; nt++) e[nt][0] = e[nt][1] = 0.0;
#pragma unroll
        for (int mt = 0; mt < 2; mt++) {
            const int64_t n = tile * kPvFT + wm * 16 + mt * 8 + g;
            if (n < P.M) {
                const double2 c = chirp(n, P.M);
                double2* out = P.dst + (int64_t)(seq0 + t) * P.Lh + n;  // sequence seq0 + 4 nt + t
#pragma unroll
                for (int nt = 0; nt < 8; nt++) {
                    const double2 z = make_double2(acc[mt][nt][0], acc[mt][nt][1]);
                    e[nt][0] += z.x * z.x;
                    e[nt][1] += z.y * z.y;
                    if (seq0 + nt * 4 + t < P.nseq) *out = cmul(z, c);
                    out += 4 * P.Lh;
                }
            }
        }
#pragma unroll
        for (int nt = 0; nt < 8; nt++)
#pragma unroll
            for (int c = 0; c < 2; c++)
#pragma unroll
                for (int off = 4; off < 32; off <<= 1) e[nt][c] += __shfl_xor_sync(0xffffffffu, e[nt][c], off);
        if (g == 0)
#pragma unroll
            for (int nt = 0; nt < 8; nt++) {
                red[wm][nt * 8 + 2 * t] = e[nt][0];
                red[wm][nt * 8 + 2 * t + 1] = e[nt][1];
            }
        asm volatile("bar.sync 2, 256;" ::: "memory");
        if (threadIdx.x < kPvNT) {
            double sum = 0.0;
#pragma unroll
            for (int w = 0; w < 8; w++) sum += red[w][threadIdx.x];
            P.epart[((int64_t)blockIdx.x * kPvNT + threadIdx.x) * P.tiles + tile] = sum;
        }
        asm volatile("bar.sync 2, 256;" ::: "memory");  // `red` is reused
    }
    __threadfence();
    asm volatile("bar.sync 2, 256;" ::: "memory");
    if (threadIdx.x == 0) last = atomicAdd(P.ticket, 1u) == gridDim.x * gridDim.y - 1;
    asm volatile("bar.sync 2, 256;" ::: "memory");
    if (!last) return;
    __threadfence();
    for (int64_t m = warp; m < (int64_t)gridDim.x * kPvNT; m += 8) {
        double v = 0.0;
        for (int64_t b = lane; b < P.tiles; b += 32) v += __ldcg(P.epart + m * P.tiles + b);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        if (lane == 0) P.energy[m] = v;
    }
    if (threadIdx.x == 0) *P.ticket = 0;
}

// Rows first_mode + 2j and first_mode + 2j + 1 (those < num_modes) of int_out (num_modes, points) from sequence j
// of the transform outputs y (natural order; the spectrum is Z[m] = chirp(m) y[m] / L).  The two real signals of
// z = a + i b separate as A = (Z[k] + conj Z[M-k]) / 2 and B = (Z[k] - conj Z[M-k]) / (2i), formed before they
// are squared, and each row is (|X|^2 + E) / 2 as in combine_signal_kernel with scale = 1 / (8 L^2) for the
// unhalved sums.  A mode of zero energy is the zero signal: its row is exactly zero, free of its partner's
// rounding.
__global__ void __launch_bounds__(256) combine_modes_kernel(const double2* __restrict__ y, int64_t Lh, int nseq,
                                                            const double* __restrict__ energy, int64_t first_mode,
                                                            int64_t num_modes, int64_t M, double scale,
                                                            int64_t points, double dt, double* __restrict__ wn_out,
                                                            double* __restrict__ int_out) {
    for (int64_t j = blockIdx.y; j < nseq; j += gridDim.y) {
        const int64_t a = first_mode + 2 * j;
        if (a >= num_modes) break;  // sequences past the last mode carry padding only
        const bool has_b = a + 1 < num_modes;
        const double ea = energy[2 * j], eb = energy[2 * j + 1];
        const double2* yj = y + j * Lh;
        for (int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; o < points;
             o += (int64_t)gridDim.x * blockDim.x) {
            const int64_t k = o + 1;
            const double2 z1 = cmul(yj[k], chirp(k, M)), z2 = cmul(yj[M - k], chirp(M - k, M));
            const double ax = z1.x + z2.x, ay = z1.y - z2.y;
            int_out[a * points + o] = ea == 0.0 ? 0.0 : __fma_rn(ax * ax + ay * ay, scale, 0.5 * ea);
            if (has_b) {
                const double bx = z1.y + z2.y, by = z1.x - z2.x;
                int_out[(a + 1) * points + o] = eb == 0.0 ? 0.0 : __fma_rn(bx * bx + by * by, scale, 0.5 * eb);
            }
        }
    }
    if (wn_out && blockIdx.y == 0) write_wavenumbers(wn_out, points, M, dt);
}

// ---- mean squared displacement (rn_msd) -------------------------------------------------------------
// With the unwrapped path r(n) = (x(n) - x(0) - K(n)) @ lattice, K(n) = sum_{j<n} k_j the integer image shifts of
// the minimum-image steps (k_j = ceil(x[j+1] - x[j] - 0.5), so that the step is wrap_disp(x[j+1], x[j])), and
// D(n) = |r(n)|^2, expanding the square gives
//   sum_{n<S-m} |r(n+m) - r(n)|^2 = sum_{n<S-m} D(n) + sum_{n>=m} D(n) - 2 C(m),
// C the linear autocorrelation of r.  A slot (the VDOS slot layout, sqrt(w) = 1) carries the six coordinate paths
// of its two atoms as z_c = r_a,c + i r_b,c, c = x, y, z: the autocorrelation tile pass turns them into
// C_a(m) + C_b(m) = Re(y_0 + y_1 + y_2)[m] / L, and D_a + D_b is one row.  The frames of a slot run in blocks of
// kPackThreads; K and the prefix sums of D combine per-block totals, scanned over the blocks by the block of the
// slot that finishes last, with in-block scans of a fixed order: every value is bit-reproducible (the K are exact
// integers in any order).

struct MsdParams {
    const double* pos;      // (S,N,3) fractional
    int64_t num_atoms;
    int64_t S, Lh;
    int64_t nb;             // slots in the chunk: blockIdx.x = frame block * nb + slot
    int64_t fblocks;        // frame blocks of a slot
    const VdosSlot* slots;  // the chunk's slots
    double lattice[9];      // rows are lattice vectors
    double* counts;         // (nb, fblocks, 6) image shifts of each block's steps, then their inclusive scan
    double2* dst;           // (3 nb, Lh) work buffer: r(n), n < S
    double* dloc;           // (nb, 3 S) power rows: D summed over the frames of its block up to n (inclusive)
    double* dsum;           // (nb, fblocks + 1) block sums of D, then their inclusive scan
    unsigned int* ticket;   // nb tickets, zero between launches
};

// inclusive scan of NV values over the block in a fixed order (bit-reproducible); sm holds NV doubles per warp
template <int NV>
__device__ __forceinline__ void block_scan(double (&v)[NV], double* sm) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1)
#pragma unroll
        for (int c = 0; c < NV; c++) {
            const double u = __shfl_up_sync(0xffffffffu, v[c], off);
            if (lane >= off) v[c] += u;
        }
    if (lane == 31)
#pragma unroll
        for (int c = 0; c < NV; c++) sm[warp * NV + c] = v[c];
    __syncthreads();
    double before[NV];
#pragma unroll
    for (int c = 0; c < NV; c++) before[c] = 0.0;
    for (int w = 0; w < warp; w++)
#pragma unroll
        for (int c = 0; c < NV; c++) before[c] += sm[w * NV + c];
#pragma unroll
    for (int c = 0; c < NV; c++) v[c] += before[c];
    __syncthreads();  // sm is reused
}

// The last thread publishes its block's totals (NV values) at vals + NV * fb of the slot's row of `count` blocks;
// the slot's block that finishes last replaces the row by its inclusive scan and re-arms the ticket.
template <int NV>
__device__ __forceinline__ void publish_and_scan(const double (&total)[NV], double* vals, int64_t fb, int64_t count,
                                                 unsigned int* ticket, double* sm) {
    __shared__ bool last;
    if (threadIdx.x == blockDim.x - 1) {
#pragma unroll
        for (int c = 0; c < NV; c++) vals[fb * NV + c] = total[c];
        __threadfence();
        last = atomicAdd(ticket, 1u) == (unsigned int)(count - 1);
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    double carry[NV];
#pragma unroll
    for (int c = 0; c < NV; c++) carry[c] = 0.0;
    for (int64_t base = 0; base < count; base += blockDim.x) {
        const int64_t i = base + threadIdx.x;
        double v[NV];
#pragma unroll
        for (int c = 0; c < NV; c++) v[c] = i < count ? __ldcg(vals + i * NV + c) : 0.0;
        block_scan<NV>(v, sm);
#pragma unroll
        for (int c = 0; c < NV; c++) {
            v[c] = carry[c] + v[c];
            if (i < count) vals[i * NV + c] = v[c];
        }
        if (threadIdx.x == blockDim.x - 1)
#pragma unroll
            for (int c = 0; c < NV; c++) sm[c] = v[c];
        __syncthreads();
#pragma unroll
        for (int c = 0; c < NV; c++) carry[c] = sm[c];
        __syncthreads();
    }
    if (threadIdx.x == 0) *ticket = 0;
}

// Count pass: the image shifts of the steps n -> n + 1 of a frame block (its frames and the next block's first),
// summed per block, then scanned over the slot's blocks.
__global__ void __launch_bounds__(kPackThreads) msd_count_kernel(const __grid_constant__ MsdParams P) {
    __shared__ double rows[(kPackThreads + 1) * 6];
    __shared__ double sm[6 * (kPackThreads / 32)];
    const int64_t j = blockIdx.x % P.nb, fb = blockIdx.x / P.nb;
    const int64_t first = fb * kPackThreads;
    const int64_t avail = min((int64_t)kPackThreads + 1, P.S - first);
    stage_slot_frames(P.pos, P.num_atoms, P.slots[j], first, avail, rows, kPackThreads + 1);
    __syncthreads();
    double k[6];
#pragma unroll
    for (int e = 0; e < 6; e++)
        k[e] = threadIdx.x + 1 < avail ? ceil((rows[(threadIdx.x + 1) * 6 + e] - rows[threadIdx.x * 6 + e]) - 0.5) : 0.0;
    block_scan<6>(k, sm);
    publish_and_scan<6>(k, P.counts + j * P.fblocks * 6, fb, P.fblocks, P.ticket + j, sm);
}

// Unwrap + pack: r(n) of the slot's two atoms from the block's base shifts and an in-block scan of the step shifts,
// stored as the three sequences z_c (no chirp: a plain zero-padded correlation), and the in-block prefix sums of D.
__global__ void __launch_bounds__(kPackThreads) msd_pack_kernel(const __grid_constant__ MsdParams P) {
    __shared__ double rows[kPackThreads * 6];
    __shared__ double origin[6];
    __shared__ double sm[6 * (kPackThreads / 32)];
    const int64_t j = blockIdx.x % P.nb, fb = blockIdx.x / P.nb;
    const VdosSlot slot = P.slots[j];
    const int64_t first = fb * kPackThreads;
    const int64_t avail = min((int64_t)kPackThreads, P.S - first);
    stage_slot_frames(P.pos, P.num_atoms, slot, first, avail, rows, kPackThreads);
    if (threadIdx.x < 6) {
        const int atom = slot.atom[threadIdx.x / 3];
        origin[threadIdx.x] = atom >= 0 ? __ldg(P.pos + 3 * atom + threadIdx.x % 3) : 0.0;
    }
    __syncthreads();
    const int t = threadIdx.x;
    double k[6];
#pragma unroll
    for (int e = 0; e < 6; e++) k[e] = (t >= 1 && t < avail) ? ceil((rows[t * 6 + e] - rows[(t - 1) * 6 + e]) - 0.5) : 0.0;
    block_scan<6>(k, sm);  // K(n) - K(first)
    double d[1] = {0.0};
    const int64_t n = first + t;
    if (t < avail) {
        const double* base = fb > 0 ? P.counts + (j * P.fblocks + fb - 1) * 6 : nullptr;  // K(first)
        double2 z[3];
#pragma unroll
        for (int m = 0; m < 2; m++) {
            double u[3];
#pragma unroll
            for (int e = 0; e < 3; e++) {
                const double shift = base ? __ldcg(base + 3 * m + e) + k[3 * m + e] : k[3 * m + e];
                u[e] = (rows[t * 6 + 3 * m + e] - origin[3 * m + e]) - shift;
            }
#pragma unroll
            for (int c = 0; c < 3; c++) {
                const double r = u[0] * P.lattice[c] + u[1] * P.lattice[3 + c] + u[2] * P.lattice[6 + c];
                if (m == 0) z[c].x = r;
                else z[c].y = r;
            }
        }
        d[0] = (z[0].x * z[0].x + z[1].x * z[1].x + z[2].x * z[2].x) + (z[0].y * z[0].y + z[1].y * z[1].y + z[2].y * z[2].y);
        double2* dst = P.dst + j * 3 * P.Lh;
#pragma unroll
        for (int c = 0; c < 3; c++) dst[(int64_t)c * P.Lh + n] = z[c];
    }
    block_scan<1>(d, sm);
    if (t < avail) P.dloc[j * 3 * P.S + n] = d[0];
    publish_and_scan<1>(d, P.dsum + j * (P.fblocks + 1), fb, P.fblocks, P.ticket + j, sm);
}

// sum_{n<k} D(n) of a slot: the scanned totals of the blocks before n's block plus the in-block prefix
__device__ __forceinline__ double d_prefix(const double* dloc, const double* dsum, int64_t k) {
    if (k == 0) return 0.0;
    const int64_t n = k - 1, b = n / kPackThreads;
    return b > 0 ? dsum[b - 1] + dloc[n] : dloc[n];
}

// Rows g_lo .. g_lo + num_groups - 1 of out (G, S), for the slots first .. first + nb - 1 of this chunk: row g at lag m
// is the sum, over its slots in slot order, of A(m) - 2 C(m) with A(m) = sum_{n<S-m} D(n) + sum_{n>=m} D(n).  A
// group's first slot writes the row and later slots add to it one at a time, as combine_groups_kernel does.
__global__ void __launch_bounds__(256) msd_combine_kernel(const double2* __restrict__ y, int64_t Lh,
                                                          const double* __restrict__ dloc,
                                                          const double* __restrict__ dsum, int64_t dsum_stride,
                                                          const int64_t* __restrict__ group_slots, int64_t first,
                                                          int64_t nb, int64_t g_lo, int64_t num_groups, int64_t S,
                                                          double inv_l, double* __restrict__ out) {
    for (int64_t g = g_lo + blockIdx.y; g < g_lo + num_groups; g += gridDim.y) {
        const int64_t begin = group_slots[g];
        const int64_t s0 = max(begin, first), s1 = min(group_slots[g + 1], first + nb);
        double* row = out + g * S;
        for (int64_t m = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; m < S; m += (int64_t)gridDim.x * blockDim.x) {
            double acc = begin < first ? row[m] : 0.0;
#pragma unroll 1
            for (int64_t slot = s0; slot < s1; slot++) {
                const int64_t j = slot - first;
                const double2* yj = y + j * 3 * Lh;
                const double c = (yj[m].x + yj[Lh + m].x) + yj[2 * Lh + m].x;
                const double* dl = dloc + j * 3 * S;
                const double* ds = dsum + j * dsum_stride;
                const double a = d_prefix(dl, ds, S - m) + (d_prefix(dl, ds, S) - d_prefix(dl, ds, m));
                const double term = __fma_rn(-2.0 * inv_l, c, a);
                acc = slot == begin ? term : __dadd_rn(acc, term);
            }
            row[m] = acc;
        }
    }
}

// MSD_g(m) = row_g(m) / ((S - m) |g|); lag 0 is exactly 0
__global__ void __launch_bounds__(256) msd_finish_kernel(const int64_t* __restrict__ group_offsets, int64_t num_groups,
                                                         int64_t S, double* __restrict__ out) {
    for (int64_t g = blockIdx.y; g < num_groups; g += gridDim.y) {
        const double size = (double)(group_offsets[g + 1] - group_offsets[g]);
        double* row = out + g * S;
        for (int64_t m = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; m < S; m += (int64_t)gridDim.x * blockDim.x)
            row[m] = m == 0 ? 0.0 : row[m] / ((double)(S - m) * size);
    }
}

}  // namespace rn

using namespace rn;

// The slots of G atom groups (CSR: group g is h_atoms[h_group_offsets[g] .. h_group_offsets[g+1]-1], checked here):
// two memberships of a group per slot, in group order; a group of odd size pads its last slot with atom -1, the
// zero signal.  group_slots (G+1) receives the slot offsets of the groups.
static int make_slots(const int64_t* h_group_offsets, const int64_t* h_atoms, int64_t num_groups, int64_t num_atoms,
                      const double* h_weights, std::vector<int64_t>& group_slots, std::vector<VdosSlot>& slots) {
    RN_CHECK_ARG(h_group_offsets[0] == 0, "group offsets must start at 0");
    group_slots.assign((size_t)num_groups + 1, 0);
    for (int64_t g = 0; g < num_groups; g++) {
        const int64_t size = h_group_offsets[g + 1] - h_group_offsets[g];
        RN_CHECK_ARG(size >= 1, "group %lld is empty", (long long)g);
        group_slots[(size_t)g + 1] = group_slots[(size_t)g] + (size + 1) / 2;
    }
    slots.assign((size_t)group_slots[(size_t)num_groups], VdosSlot{});
    for (int64_t g = 0; g < num_groups; g++) {
        for (int64_t m = h_group_offsets[g]; m < h_group_offsets[g + 1]; m++) {
            const int64_t atom = h_atoms[m];
            RN_CHECK_ARG(atom >= 0 && atom < num_atoms, "atom index %lld of group %lld out of range [0, %lld)",
                         (long long)atom, (long long)g, (long long)num_atoms);
            const int64_t half = m - h_group_offsets[g];
            VdosSlot& slot = slots[(size_t)(group_slots[(size_t)g] + half / 2)];
            slot.atom[half & 1] = (int)atom;
            slot.sqrtw[half & 1] = h_weights ? std::sqrt(h_weights[atom]) : 1.0;
            if ((half & 1) == 0) {  // the partner, unless the group has another atom
                slot.atom[1] = -1;
                slot.sqrtw[1] = 0.0;
            }
        }
    }
    return RN_OK;
}

// Uploads the slot table, the groups' slot offsets and (h_group_offsets != nullptr) their atom offsets, in that
// order, to the plan's scratch buffer, which keeps extra_bytes after them.
static int upload_slots(rn_spectrum_plan* plan, const std::vector<VdosSlot>& slots,
                        const std::vector<int64_t>& group_slots, const int64_t* h_group_offsets, int64_t extra_bytes,
                        cudaStream_t s, char** table_out) {
    const int64_t table_bytes = (int64_t)sizeof(VdosSlot) * (int64_t)slots.size();
    const int64_t group_bytes = (int64_t)sizeof(int64_t) * (int64_t)group_slots.size();
    const int64_t need = table_bytes + group_bytes * (h_group_offsets ? 2 : 1) + extra_bytes;
    void* scratch = nullptr;
    const int rc = plan_scratch(plan, need, s, "VDOS slot tables", &scratch);
    if (rc != RN_OK) return rc;
    char* table = static_cast<char*>(scratch);
    // pageable sources: the copies return once the data is staged, so the vectors may go out of scope
    RN_CUDA(cudaMemcpyAsync(table, slots.data(), (size_t)table_bytes, cudaMemcpyHostToDevice, s));
    RN_CUDA(cudaMemcpyAsync(table + table_bytes, group_slots.data(), (size_t)group_bytes, cudaMemcpyHostToDevice, s));
    if (h_group_offsets)
        RN_CUDA(cudaMemcpyAsync(table + table_bytes + group_bytes, h_group_offsets, (size_t)group_bytes,
                                cudaMemcpyHostToDevice, s));
    *table_out = table;
    return RN_OK;
}

// The number of groups with slots among first .. first + nb - 1, from *g_lo on; *g_lo enters as the first group of
// the previous chunk (0 for the first).
static int64_t chunk_groups(const std::vector<int64_t>& group_slots, int64_t first, int64_t nb, int64_t* g_lo) {
    while (group_slots[(size_t)*g_lo + 1] <= first) ++*g_lo;
    int64_t g_hi = *g_lo;  // last group with a slot in the chunk
    while (group_slots[(size_t)g_hi + 1] < first + nb) g_hi++;
    return g_hi - *g_lo + 1;
}

// The slots of all groups, in group order, run in chunks of the plan's batch: per chunk one velocity pack, the
// convolution of its 3 nb sequences with OUT_POWER and one combine that adds the chunk's slots to the rows of
// the groups they belong to.
extern "C" int rn_vdos(rn_spectrum_plan* plan, const double* d_positions, int64_t num_atoms, const double* h_lattice,
                       const double* h_weights, const int64_t* h_group_offsets, const int64_t* h_atoms,
                       int64_t num_groups, double timestep_fs, double* d_wavenumbers, double* d_intensities,
                       void* stream) {
    RN_CHECK_ARG(plan != nullptr, "plan is null");
    RN_CHECK_ARG(plan->world == 1, "rn_vdos needs a single-GPU plan (rn_spectrum_plan_create_batched)");
    RN_CHECK_ARG(d_positions && h_lattice && h_group_offsets && h_atoms, "null pointer");
    RN_CHECK_ARG(num_atoms >= 1 && num_atoms <= INT32_MAX, "invalid num_atoms %lld", (long long)num_atoms);
    RN_CHECK_ARG(num_groups >= 1, "num_groups must be at least 1 (got %lld)", (long long)num_groups);
    RN_CHECK_ARG(timestep_fs > 0 && std::isfinite(timestep_fs), "timestep must be positive");
    for (int i = 0; i < 9; i++) RN_CHECK_ARG(std::isfinite(h_lattice[i]), "lattice entry %d is not finite", i);
    if (h_weights)
        for (int64_t i = 0; i < num_atoms; i++)
            RN_CHECK_ARG(std::isfinite(h_weights[i]) && h_weights[i] >= 0, "invalid weight %g of atom %lld",
                         h_weights[i], (long long)i);
    std::vector<int64_t> group_slots;
    std::vector<VdosSlot> slots;
    int rc = make_slots(h_group_offsets, h_atoms, num_groups, num_atoms, h_weights, group_slots, slots);
    if (rc != RN_OK) return rc;
    const int64_t num_slots = group_slots[(size_t)num_groups];
    const int64_t points = rn_spectrum_num_points(plan->S);
    if (points == 0) return RN_OK;
    RN_CHECK_ARG(d_wavenumbers && d_intensities, "null output pointer");
    DeviceGuard guard(plan->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    char* table = nullptr;
    rc = upload_slots(plan, slots, group_slots, nullptr, 0, s, &table);
    if (rc != RN_OK) return rc;
    const VdosSlot* d_slots = reinterpret_cast<const VdosSlot*>(table);
    const int64_t* d_group_slots = reinterpret_cast<const int64_t*>(table + sizeof(VdosSlot) * num_slots);

    const int64_t M = plan->M;
    const double scale = 0.25 / ((double)plan->L * (double)plan->L);
    VdosPackParams pp;
    pp.pos = d_positions;
    pp.num_atoms = num_atoms;
    pp.M = M;
    pp.Lh = plan->Lh;
    for (int i = 0; i < 9; i++) pp.lattice[i] = h_lattice[i];
    pp.inv_dt = 1.0 / timestep_fs;
    pp.dst = plan->d_work;
    pp.epart = plan->d_epart;
    pp.ticket = plan->d_ticket;
    int64_t g_lo = 0;  // first group with a slot in the chunk
    for (int64_t first = 0; first < num_slots; first += plan->batch) {
        const int64_t nb = std::min(plan->batch, num_slots - first);
        const int64_t groups = chunk_groups(group_slots, first, nb, &g_lo);
        pp.slots = d_slots + first;
        pack_velocity_kernel<<<dim3(plan->pack_blocks, (unsigned)nb), kPackThreads, 0, s>>>(pp);
        RN_LAUNCHED();
        rc = run_convolution(plan, plan->d_work, (int)(3 * nb), M, power_out(plan), nullptr, s);
        if (rc != RN_OK) return rc;
        combine_groups_kernel<<<dim3(grid_for(points, plan->sm_count), (unsigned)std::min<int64_t>(groups, 65535)), 256,
                                0, s>>>(plan->d_power, plan->d_epart + plan->pack_blocks, plan->pack_blocks + 1,
                                        d_group_slots, first, nb, g_lo, groups, M, scale, points, timestep_fs,
                                        first == 0 ? d_wavenumbers : nullptr, d_intensities);
        RN_LAUNCHED();
        RN_CUDA(cudaGetLastError());
    }
    return RN_OK;
}

// The MSD runs on the VDOS slots (two memberships of a group per slot, unit weights) in chunks of the plan's batch:
// per chunk the count pass, the unwrap + pack, the autocorrelation of its 3 nb sequences (the transform passes of
// one measure, the tile pass squaring instead of filtering) and one combine that adds the chunk's slots to their
// group rows; one finishing launch divides the rows.
extern "C" int rn_msd(rn_spectrum_plan* plan, const double* d_positions, int64_t num_atoms, const double* h_lattice,
                      const int64_t* h_group_offsets, const int64_t* h_atoms, int64_t num_groups, double* d_msd,
                      void* stream) {
    RN_CHECK_ARG(plan != nullptr, "plan is null");
    RN_CHECK_ARG(plan->world == 1, "rn_msd needs a single-GPU plan (rn_spectrum_plan_create_batched)");
    RN_CHECK_ARG(d_positions && h_lattice && h_group_offsets && h_atoms && d_msd, "null pointer");
    RN_CHECK_ARG(num_atoms >= 1 && num_atoms <= INT32_MAX, "invalid num_atoms %lld", (long long)num_atoms);
    RN_CHECK_ARG(num_groups >= 1, "num_groups must be at least 1 (got %lld)", (long long)num_groups);
    for (int i = 0; i < 9; i++) RN_CHECK_ARG(std::isfinite(h_lattice[i]), "lattice entry %d is not finite", i);
    std::vector<int64_t> group_slots;
    std::vector<VdosSlot> slots;
    int rc = make_slots(h_group_offsets, h_atoms, num_groups, num_atoms, nullptr, group_slots, slots);
    if (rc != RN_OK) return rc;
    const int64_t num_slots = group_slots[(size_t)num_groups];
    DeviceGuard guard(plan->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int64_t S = plan->M, fblocks = plan->pack_blocks;
    const int64_t chunk = std::min(plan->batch, (int64_t)INT32_MAX / fblocks);  // the passes' blocks on gridDim.x
    char* table = nullptr;
    rc = upload_slots(plan, slots, group_slots, h_group_offsets, (int64_t)sizeof(double) * 6 * fblocks * chunk, s,
                      &table);
    if (rc != RN_OK) return rc;
    const int64_t group_bytes = (int64_t)sizeof(int64_t) * (num_groups + 1);
    const VdosSlot* d_slots = reinterpret_cast<const VdosSlot*>(table);
    const int64_t* d_group_slots = reinterpret_cast<const int64_t*>(table + sizeof(VdosSlot) * num_slots);
    const int64_t* d_group_offsets = reinterpret_cast<const int64_t*>(table + sizeof(VdosSlot) * num_slots + group_bytes);

    MsdParams pp;
    pp.pos = d_positions;
    pp.num_atoms = num_atoms;
    pp.S = S;
    pp.Lh = plan->Lh;
    pp.fblocks = fblocks;
    for (int i = 0; i < 9; i++) pp.lattice[i] = h_lattice[i];
    pp.counts = reinterpret_cast<double*>(table + sizeof(VdosSlot) * num_slots + 2 * group_bytes);
    pp.dst = plan->d_work;
    pp.dloc = plan->d_power;
    pp.dsum = plan->d_epart;
    pp.ticket = plan->d_ticket;
    const double inv_l = 1.0 / (double)plan->L;
    int64_t g_lo = 0;  // first group with a slot in the chunk
    for (int64_t first = 0; first < num_slots; first += chunk) {
        const int64_t nb = std::min(chunk, num_slots - first);
        const int64_t groups = chunk_groups(group_slots, first, nb, &g_lo);
        pp.slots = d_slots + first;
        pp.nb = nb;
        // slot fastest: the blocks of neighbouring slots read the same frames side by side
        const unsigned blocks = (unsigned)(nb * fblocks);
        msd_count_kernel<<<blocks, kPackThreads, 0, s>>>(pp);
        RN_LAUNCHED();
        msd_pack_kernel<<<blocks, kPackThreads, 0, s>>>(pp);
        RN_LAUNCHED();
        rc = run_convolution(plan, plan->d_work, (int)(3 * nb), S, plain_out(), nullptr, s, 0, true);
        if (rc != RN_OK) return rc;
        msd_combine_kernel<<<dim3(grid_for(S, plan->sm_count), (unsigned)std::min<int64_t>(groups, 65535)), 256, 0,
                             s>>>(plan->d_work, plan->Lh, plan->d_power, plan->d_epart, plan->pack_blocks + 1,
                                  d_group_slots, first, nb, g_lo, groups, S, inv_l, d_msd);
        RN_LAUNCHED();
        RN_CUDA(cudaGetLastError());
    }
    msd_finish_kernel<<<dim3(grid_for(S, plan->sm_count), (unsigned)std::min<int64_t>(num_groups, 65535)), 256, 0, s>>>(
        d_group_offsets, num_groups, S, d_msd);
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    return RN_OK;
}

// The modes, padded to windows of six, run in chunks of the plan's batch: per chunk one projection (the
// trajectory streamed once per 64 modes of the chunk), the convolution of its 3 nb sequences with OUT_PLAIN and
// one combine that separates the packed pairs into their rows.
extern "C" int rn_projected_vdos(rn_spectrum_plan* plan, const double* d_positions, int64_t num_atoms,
                                 const double* h_lattice, const double* h_vectors, int64_t num_vectors,
                                 double timestep_fs, double* d_wavenumbers, double* d_intensities, void* stream) {
    RN_CHECK_ARG(plan != nullptr, "plan is null");
    RN_CHECK_ARG(plan->world == 1, "rn_projected_vdos needs a single-GPU plan (rn_spectrum_plan_create_batched)");
    RN_CHECK_ARG(d_positions && h_lattice && h_vectors, "null pointer");
    RN_CHECK_ARG(num_atoms >= 1 && num_atoms <= INT32_MAX / 3, "invalid num_atoms %lld", (long long)num_atoms);
    RN_CHECK_ARG(num_vectors >= 1 && num_vectors <= INT32_MAX / 3, "invalid num_vectors %lld",
                 (long long)num_vectors);
    RN_CHECK_ARG(timestep_fs > 0 && std::isfinite(timestep_fs), "timestep must be positive");
    for (int i = 0; i < 9; i++) RN_CHECK_ARG(std::isfinite(h_lattice[i]), "lattice entry %d is not finite", i);
    const int64_t cols = 3 * num_atoms;
    for (int64_t e = 0; e < num_vectors * cols; e++)
        RN_CHECK_ARG(std::isfinite(h_vectors[e]), "entry %lld of vectors is not finite", (long long)e);
    const int64_t points = rn_spectrum_num_points(plan->S);
    if (points == 0) return RN_OK;
    RN_CHECK_ARG(d_wavenumbers && d_intensities, "null output pointer");
    DeviceGuard guard(plan->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int64_t M = plan->M;
    const int64_t rpad = (cols + kPvKC - 1) / kPvKC * kPvKC;
    const int64_t windows = (num_vectors + 5) / 6;  // six modes per window of the plan
    const int64_t rows = 6 * windows + kPvNT;       // a chunk's last mode tile reads up to 63 rows past its modes
    const int64_t tiles = (M + kPvFT - 1) / kPvFT;
    const int64_t mtiles_max = (6 * std::min(plan->batch, windows) + kPvNT - 1) / kPvNT;
    const int64_t matrix = rows * rpad, parts = mtiles_max * kPvNT * tiles;
    void* scratch = nullptr;
    int rc = plan_scratch(plan, (int64_t)sizeof(double) * (matrix + parts + mtiles_max * kPvNT), s,
                          "projection matrix and energy partials", &scratch);
    if (rc != RN_OK) return rc;
    double* d_proj = static_cast<double*>(scratch);
    // B^T[k][3i + a] = sum_c lattice[a][c] vectors[k][i][c] / dt; padding rows (modes >= K) and columns are zero
    std::vector<double> bt((size_t)matrix, 0.0);
    for (int64_t k = 0; k < num_vectors; k++)
        for (int64_t i = 0; i < num_atoms; i++) {
            const double* v = h_vectors + (k * num_atoms + i) * 3;
            for (int a = 0; a < 3; a++)
                bt[(size_t)(k * rpad + 3 * i + a)] =
                    (h_lattice[3 * a] * v[0] + h_lattice[3 * a + 1] * v[1] + h_lattice[3 * a + 2] * v[2]) / timestep_fs;
        }
    // pageable source: the copy returns once the data is staged, so the vector may go out of scope
    RN_CUDA(cudaMemcpyAsync(d_proj, bt.data(), sizeof(double) * (size_t)matrix, cudaMemcpyHostToDevice, s));

    const bool align16 = reinterpret_cast<uintptr_t>(d_positions) % 16 == 0 && cols % 2 == 0;
    const auto kernel = align16 ? project_velocity_kernel<true> : project_velocity_kernel<false>;
    RN_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPvSmemBytes));
    ProjParams pp;
    pp.pos = d_positions;
    pp.cols = cols;
    pp.M = M;
    pp.Lh = plan->Lh;
    pp.rpad = (int)rpad;
    pp.tiles = tiles;
    pp.dst = plan->d_work;
    pp.epart = d_proj + matrix;
    pp.energy = pp.epart + parts;
    pp.ticket = plan->d_ticket;
    const double scale = 0.125 / ((double)plan->L * (double)plan->L);
    for (int64_t first = 0; first < windows; first += plan->batch) {
        const int64_t nb = std::min(plan->batch, windows - first);
        const int64_t mtiles = (6 * nb + kPvNT - 1) / kPvNT;
        pp.bt = d_proj + 6 * first * rpad;
        pp.nseq = (int)(3 * nb);
        // mode tiles of one frame range run side by side, so the second reads the frames from L2
        const int64_t ranges = std::max<int64_t>(1, std::min<int64_t>(tiles, plan->sm_count / mtiles));
        kernel<<<dim3((unsigned)mtiles, (unsigned)ranges), kPvThreads, kPvSmemBytes, s>>>(pp);
        RN_LAUNCHED();
        rc = run_convolution(plan, plan->d_work, (int)(3 * nb), M, plain_out(), nullptr, s);
        if (rc != RN_OK) return rc;
        combine_modes_kernel<<<dim3(grid_for(points, plan->sm_count), (unsigned)std::min<int64_t>(3 * nb, 65535)), 256,
                               0, s>>>(plan->d_work, plan->Lh, (int)(3 * nb), pp.energy, 6 * first, num_vectors, M,
                                       scale, points, timestep_fs, first == 0 ? d_wavenumbers : nullptr,
                                       d_intensities);
        RN_LAUNCHED();
        RN_CUDA(cudaGetLastError());
    }
    return RN_OK;
}
