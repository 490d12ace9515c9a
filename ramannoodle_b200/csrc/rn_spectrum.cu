// MD Raman spectrum (sm_100a): MDRamanSpectrum.measure (ramannoodle/spectrum/_raman.py:241-309) and
// calc_signal_spectrum (ramannoodle/spectrum/utils.py:76-124).
//
// The reference forms the linear autocorrelation of each signal x (length M = S-1) with
// scipy.signal.correlate and takes the real part of its length-M FFT.  With the exact identity
//   Re FFT_M(ac+)[k] = (|FFT_M(x)[k]|^2 + sum_n x_n^2) / 2                      (SURVEY.md §7 step 7)
// only FFT_M(x) is needed, for arbitrary M: Bluestein's chirp-z algorithm on the in-place
// power-of-two convolution core of rn_fft.cuh.
//
// Orientational average without unpacking.  45 a^2 + 7 g^2 (_raman.py:286-297) is
//   I[k] = 1/2 sum_s w_s (|X_s[k]|^2 + E_s),  weights 5 (trace), 3.5 (xx-yy, yy-zz, zz-xx), 21 (xy, yz, xz).
// Since |X_a|^2 + |X_b|^2 + |X_a + X_b|^2 = 3/2 |X_a + X_b|^2 + 1/2 |X_a - X_b|^2, six real signals scaled
// by the square roots of their weights carry everything:
//   sqrt5 (xx+yy+zz), sqrt5.25 (xx-zz), sqrt1.75 (xx-2yy+zz), sqrt21 xy, sqrt21 yz, sqrt21 xz.
// Packed pairwise into three complex sequences z_p, |Z_p[k]|^2 + |Z_p[M-k]|^2 = 2 (|X_1[k]|^2 + |X_2[k]|^2)
// for ANY pair of real signals, hence
//   I[k] = (P[k] + P[M-k]) / 4 + E / 2,   P[m] = sum_p |Z_p[m]|^2,   E = sum_p sum_n |z_p[n]|^2:
// no separation of the packed signals, no chirp post-multiply (|c| = 1), and the pairing of bins k and
// M-k is a sum of two reals.  The same holds bin by bin when the transform is shared by several GPUs.
//
// Multi-GPU (G = 2, 4 or 8 ranks share ONE length-L transform, L = G Lh): decimation in frequency at
// rank level.  Rank p packs the difference signals n = q Lh + n' of its block of n' (rows pushed to it by
// the evaluation kernels), takes the G-point DFT over q, multiplies by W_L^{r n'} and stores the result
// for residue r into rank r's work buffer over NVLink; rank r runs the local length-Lh convolution with
// its decimated filter; the inverse's last pass stores z_r[m'] to the rank that owns m', which finishes
// y[q Lh + m'] = sum_r W_G^{-qr} W_L^{-r m'} z_r[m'] and writes P to every rank.
#include <algorithm>
#include <cmath>
#include <cstdlib>

#include "rn_device.cuh"
#include "rn_fft.cuh"

struct rn_spectrum_plan {
    int device = 0;
    int sm_count = 0;
    int64_t S = 0, M = 0, L = 0;
    int log2l = 0;
    int world = 1;          // ranks sharing the transform (power of two)
    int rank = 0;           // this plan's rank; >= world: a spectator that only combines
    int64_t Lh = 0;         // local transform length L / world (>= 4096)
    int log2lh = 0;
    int nlev = 0;           // strided levels of the local transform
    int lev_log2r[2] = {0, 0};
    int split = 0;          // two-level twiddle split: m = hi << split | lo
    double2* d_whi = nullptr;   // L >> split   exp(-2 pi i (a << split) / L)
    double2* d_wlo = nullptr;   // 1 << split   exp(-2 pi i b / L)
    double2* d_wsub = nullptr;  // 4096         exp(-2 pi i m / 4096)
    double2* d_H = nullptr;     // Lh   filter spectrum of this rank's residue, in the transform's own order
    double2* d_work = nullptr;  // 3 Lh work buffer (single-GPU entries; plan creation)
    double* d_power = nullptr;  // 3 M  |y_p[m]|^2 (single-GPU entries)
    double* d_epart = nullptr;  // energy partial of every pack block, then their sum
    unsigned int* d_ticket = nullptr;
    int pack_blocks = 0;
    int64_t batch = 1;      // windows the work, power, partial and ticket buffers hold (single-GPU plans)
    double* d_cross = nullptr;  // cross spectra: energy partials of every series pair, then their sums
    int64_t cross_doubles = 0;
    void* d_vdos = nullptr;     // VDOS: slot table, then the slot offsets of the groups
    int64_t vdos_bytes = 0;
};

namespace rn {

using fft::cmul;
using fft::kE;
using fft::kLog2E;
using fft::kNT;
using fft::Twiddles;

constexpr int kPackThreads = 256;
constexpr double kSqrt5 = 2.2360679774997896964;
constexpr double kSqrt5_25 = 2.2912878474779200033;
constexpr double kSqrt1_75 = 1.3228756555322952953;
constexpr double kSqrt21 = 4.5825756949558400066;

// exp(-i*pi*n^2/M) (forward chirp); n^2 mod 2M is formed exactly in 64-bit integers
__device__ __forceinline__ double2 chirp(int64_t n, int64_t M) {
    const uint64_t m = ((uint64_t)n * (uint64_t)n) % (uint64_t)(2 * M);
    double s, c;
    sincospi((double)m / (double)M, &s, &c);
    return make_double2(c, -s);
}

static Twiddles plan_twiddles(const rn_spectrum_plan* p) {
    Twiddles t;
    t.hi = p->d_whi;
    t.lo = p->d_wlo;
    t.sub = p->d_wsub;
    t.split = p->split;
    return t;
}

// ---- pack: series -> chirp-multiplied packed sequences (+ rank-level DFT) ------------------------
struct PackParams {
    const double* src;   // (S,3,3) series (MD) or (M,) real signal
    int64_t M;
    int64_t Lh;
    int64_t begin, end;  // this rank's block of n'
    double2* dst[8];     // work buffers of ranks 0..G-1 (nseq, Lh); G == 1: the local one
    int aligned16;         // src is 16-byte aligned (vector loads)
    int seq_sel;           // -1: pack all three sequences; 0..2: only this one (0 also sums the energies)
    double* epart;         // [blocks] partials, then their sum
    unsigned int* ticket;  // zero between launches
    double* share[8];      // shared transform: the sum also goes to slot `share_slot` of these spectrum buffers
    int num_share;
    int share_slot;
    int zero_slot;         // >= 0: this slot is cleared (the other phase's share when the pack is not split)
    int log2_stripe;       // >= 0: this launch packs one half of every block of 2^(log2_stripe+1) n' ...
    int phase;             // ... the first (0) or the second (1)
    Twiddles tw;
    int64_t win_stride;    // windowed pack: doubles between the series of windows blockIdx.y and blockIdx.y + 1
};

// block reduction of one double (fixed tree: bit-reproducible), result valid in thread 0
__device__ __forceinline__ double block_sum(double v, double* sm) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    if (lane == 0) sm[warp] = v;
    __syncthreads();
    double total = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) total += sm[w];
    return total;
}

// Every pack block leaves its energy partial in epart[block]; the block that finishes last sums all
// partials in index order (bit-reproducible whichever block that is) into epart[gridDim.x] and re-arms
// the ticket counter.
__device__ __forceinline__ void publish_energy(double block_total, double* epart, unsigned int* ticket, double* red,
                                               const PackParams* share = nullptr) {
    __shared__ bool last;
    if (threadIdx.x == 0) {
        epart[blockIdx.x] = block_total;
        __threadfence();
        last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    double v = 0.0;
    for (unsigned int b = threadIdx.x; b < gridDim.x; b += blockDim.x) v += __ldcg(epart + b);
    __syncthreads();  // `red` is reused
    const double total = block_sum(v, red);
    if (threadIdx.x == 0) {
        epart[gridDim.x] = total;
        *ticket = 0;
        if (share)  // this rank's share of the series energy, to every rank that forms intensities
            for (int d = 0; d < share->num_share; d++) {
                share->share[d][share->share_slot] = total;
                if (share->zero_slot >= 0) share->share[d][share->zero_slot] = 0.0;
            }
    }
}

// MD series: np.diff (_raman.py:282), the six weighted signals, chirp pre-multiply; with G > 1 the
// G-point DFT over the blocks q (inputs q >= G/2 are zero: M <= L/2) and the twiddle W_L^{r n'}.
// WIN (G == 1): blockIdx.y numbers a window of a batch; window w reads the series at src + w win_stride,
// packs into its own 3 Lh of dst[0] and sums its energy with its own partials and ticket, exactly as a
// single-window launch does.
template <int G, bool WIN = false>
__global__ void __launch_bounds__(kPackThreads) pack_alpha_kernel(const __grid_constant__ PackParams P) {
    static_assert(!WIN || G == 1, "windows are packed for single-GPU transforms only");
    constexpr int GH = G > 1 ? G / 2 : 1;
    __shared__ __align__(16) double rows[(kPackThreads + 1) * 9 + 1];
    __shared__ double red[kPackThreads / 32];
    const double* src = P.src;
    double2* dst0 = P.dst[0];
    double* epart = P.epart;
    unsigned int* ticket = P.ticket;
    bool aligned16 = P.aligned16;
    if constexpr (WIN) {
        src += (int64_t)blockIdx.y * P.win_stride;
        dst0 += (int64_t)blockIdx.y * 3 * P.Lh;
        epart += (int64_t)blockIdx.y * (gridDim.x + 1);
        ticket += blockIdx.y;
        aligned16 = reinterpret_cast<uintptr_t>(src) % 16 == 0;  // 72 hop bytes: odd hops alternate
    }
    int64_t n0 = P.begin + (int64_t)blockIdx.x * kPackThreads;
    if (P.log2_stripe >= 0) {  // stripes are multiples of the block size: a block stays inside one stripe
        const int64_t idx = (int64_t)blockIdx.x * kPackThreads, stripe = (int64_t)1 << P.log2_stripe;
        n0 = P.begin + ((idx >> P.log2_stripe) << (P.log2_stripe + 1)) + (idx & (stripe - 1)) + P.phase * stripe;
    }
    const int64_t n1 = n0 + threadIdx.x;  // n'
    double2 a[GH][3];
    double energy = 0.0;
#pragma unroll
    for (int q = 0; q < GH; q++) {
        const int64_t first = (int64_t)q * P.Lh + n0;  // first difference index of this block
        const int64_t avail = min((int64_t)kPackThreads + 1, P.M + 1 - first);  // series rows first .. first+avail-1
        __syncthreads();
        const int64_t valid = avail > 0 ? avail * 9 : 0;  // doubles of the series this block may read
        if (aligned16) {
            // independent 16-byte loads, all in flight before the first store (first * 72 bytes is a multiple of 16:
            // block starts are even)
            constexpr int kVec = ((kPackThreads + 1) * 9 + 1) / 2;
            constexpr int kPer = (kVec + kPackThreads - 1) / kPackThreads;
            const double2* src2 = reinterpret_cast<const double2*>(src + first * 9);
            double2 staged[kPer];
#pragma unroll
            for (int i = 0; i < kPer; i++) {
                const int e = threadIdx.x + i * kPackThreads;
                staged[i] = make_double2(0.0, 0.0);
                if (2 * e + 1 < valid) staged[i] = __ldg(src2 + e);
                else if (2 * e < valid) staged[i].x = __ldg(src + first * 9 + 2 * e);
            }
#pragma unroll
            for (int i = 0; i < kPer; i++) {
                const int e = threadIdx.x + i * kPackThreads;
                if (e < kVec) {
                    rows[2 * e] = staged[i].x;
                    if (2 * e + 1 < (kPackThreads + 1) * 9) rows[2 * e + 1] = staged[i].y;
                }
            }
        } else {
            for (int e = threadIdx.x; e < (kPackThreads + 1) * 9; e += kPackThreads)
                rows[e] = (e < valid) ? __ldg(src + first * 9 + e) : 0.0;
        }
        __syncthreads();
        const int64_t n = first + threadIdx.x;
#pragma unroll
        for (int s = 0; s < 3; s++) a[q][s] = make_double2(0.0, 0.0);
        if (n < P.M && n1 < P.end) {
            const double* r = rows + threadIdx.x * 9;
            const double xx = r[9] - r[0], yy = r[13] - r[4], zz = r[17] - r[8];
            const double xy = r[10] - r[1], yz = r[14] - r[5], xz = r[11] - r[2];
            const double2 z0 = make_double2(kSqrt5 * (xx + yy + zz), kSqrt5_25 * (xx - zz));
            const double2 z1 = make_double2(kSqrt1_75 * (xx - 2.0 * yy + zz), kSqrt21 * xy);
            const double2 z2 = make_double2(kSqrt21 * yz, kSqrt21 * xz);
            energy += (z0.x * z0.x + z0.y * z0.y) + (z1.x * z1.x + z1.y * z1.y) + (z2.x * z2.x + z2.y * z2.y);
            const double2 c = chirp(n, P.M);
            a[q][0] = cmul(z0, c);
            a[q][1] = cmul(z1, c);
            a[q][2] = cmul(z2, c);
        }
    }
    if (n1 < P.end) {
        if constexpr (G == 1) {
            if (n1 < P.M) {
#pragma unroll
                for (int s = 0; s < 3; s++) dst0[(int64_t)s * P.Lh + n1] = a[0][s];
            }
        } else {
            const double2 w1 = fft::tw_global(P.tw, (uint32_t)n1);  // W_L^{n'}
#pragma unroll
            for (int s = 0; s < 3; s++) {
                if (P.seq_sel >= 0 && s != P.seq_sel) continue;
                double2 x[G];
#pragma unroll
                for (int q = 0; q < G; q++) x[q] = q < GH ? a[q < GH ? q : 0][s] : make_double2(0.0, 0.0);
                fft::Dft<G, -1>::run(x);
                fft::apply_powers<G>(x, w1);
#pragma unroll
                for (int r = 0; r < G; r++) P.dst[r][(int64_t)s * P.Lh + n1] = x[r];
            }
        }
    }
    if (P.seq_sel <= 0) {  // uniform over the grid
        const double total = block_sum(energy, red);
        publish_energy(total, epart, ticket, red, G > 1 ? &P : nullptr);
    }
}

// one real signal (calc_signal_spectrum): z = x, chirp pre-multiply
__global__ void __launch_bounds__(kPackThreads) pack_signal_kernel(const __grid_constant__ PackParams P) {
    __shared__ double red[kPackThreads / 32];
    const int64_t n = (int64_t)blockIdx.x * kPackThreads + threadIdx.x;
    double energy = 0.0;
    if (n < P.M) {
        const double x = __ldg(P.src + n);
        energy = x * x;
        const double2 c = chirp(n, P.M);
        P.dst[0][n] = make_double2(x * c.x, x * c.y);
    }
    const double total = block_sum(energy, red);
    publish_energy(total, P.epart, P.ticket, red);
}

// ---- filter: h_r[n'] = W_L^{r n'} sum_q h[q Lh + n'] W_G^{qr},  h[m] = exp(+i pi m^2 / M) for |m| < M
// stored circularly in a length-L array ----------------------------------------------------------
__global__ void __launch_bounds__(256) filter_fill_kernel(double2* __restrict__ out, int64_t M, int64_t L, int64_t Lh,
                                                          int world, int rank, const __grid_constant__ Twiddles tw) {
    for (int64_t n1 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n1 < Lh; n1 += (int64_t)gridDim.x * blockDim.x) {
        double2 acc = make_double2(0.0, 0.0);
        for (int q = 0; q < world; q++) {
            const int64_t idx = (int64_t)q * Lh + n1;
            int64_t m = -1;
            if (idx < M) m = idx;
            else if (L - idx < M) m = L - idx;
            if (m < 0) continue;
            const double2 c = chirp(m, M);
            double2 h = make_double2(c.x, -c.y);
            if (world > 1) h = cmul(h, fft::tw_global(tw, (uint32_t)(((int64_t)((q * rank) % world)) * Lh)));
            acc.x += h.x;
            acc.y += h.y;
        }
        if (world > 1) acc = cmul(acc, fft::tw_global(tw, (uint32_t)((int64_t)rank * n1)));
        out[n1] = acc;
    }
}

struct SpectrumParams {
    double timestep;
    int laser;
    double laser_wavenumber;
    int bose_einstein;
    double kt;  // BOLTZMANN_CONSTANT * temperature
};

// wavenumbers: scipy.fftpack.fftfreq(M, dt)[k] * 33.35640951981521 * 1e3 with fftfreq = k * (1/(M*dt))
__device__ __forceinline__ double wavenumber_of(int64_t k, int64_t M, double dt) {
    const double val = 1.0 / ((double)M * dt);
    return ((double)k * val) * 33.35640951981521 * 1e3;
}

// laser / Bose-Einstein corrections of one point (_raman.py:13-69,303-307)
__device__ __forceinline__ double corrected(double inten, double wn, const SpectrumParams& prm) {
    if (prm.laser) {
        const double r = (wn - prm.laser_wavenumber) / 10000.0;
        const double r2 = r * r;
        inten *= (r2 * r2) / wn;
    }
    if (prm.bose_einstein) {
        const double en = wn * 29979245800.0 * 4.1357e-15;
        inten *= 1.0 / (1.0 - exp(-en / prm.kt));
    }
    return inten;
}

// ---- final stage of a shared transform: y[q Lh + m'] from the G residues for a mirror pair of m', the
// pair's finished intensities I[k] = (P[k] + P[M-k]) / (4 L^2) + E/2 (corrections included) to every rank
constexpr int kSpecHeader = 16;  // spectrum buffer: energy shares (rank + 8 * pack phase), then the intensities

struct FinalParams {
    const double2* recv;  // (3, G, w + 128) slices z_r[m'] of the residues this rank owns (fft::mirror_owner)
    int64_t M, Lh, c;     // c = M mod Lh
    int log2w, log2lh;
    int rank;
    double* dest[8];      // spectrum buffers of the destination ranks
    int num_dest;
    const double* shares;  // this rank's spectrum buffer (energy shares written by the pack kernels)
    int64_t points;
    double scale;
    SpectrumParams prm;
    double* wn_out;       // local wavenumbers (points) or nullptr
    Twiddles tw;
};

template <int G>
__global__ void __launch_bounds__(256) final_dist_kernel(const __grid_constant__ FinalParams P) {
    constexpr int GH = G / 2;
    const int64_t w = (int64_t)1 << P.log2w;
    const int64_t half = w >> 1;
    const int64_t local = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // pair number within this rank's slice
    const int64_t a = ((int64_t)P.rank << P.log2w) + 2 * local + (P.c & 1);  // doubled distance from c/2
    const bool valid = local < half || (local == half && P.rank == G - 1 && a == P.Lh);
    if (valid) {
        double energy = 0.0;
#pragma unroll
        for (int r = 0; r < G; r++) energy += P.shares[r] + P.shares[8 + r];
        const double econst = 0.5 * energy;
        const bool self_paired = (a == 0 || a == P.Lh);
        const int64_t stride = 2 * fft::mirror_half_slots(P.log2w);
        int64_t m1[2], near_origin, far_top;
        m1[0] = ((a + P.c) >> 1) & (P.Lh - 1);
        m1[1] = ((2 * P.Lh + P.c - a) >> 1) & (P.Lh - 1);
        fft::mirror_arcs(P.rank, P.c, P.log2lh, P.log2w, &near_origin, &far_top);
        double power[2][GH];
#pragma unroll
        for (int side = 0; side < 2; side++) {
#pragma unroll
            for (int q = 0; q < GH; q++) power[side][q] = 0.0;
            if (side == 1 && self_paired) {
#pragma unroll
                for (int q = 0; q < GH; q++) power[1][q] = power[0][q];
                continue;
            }
            double2 w1 = fft::tw_global(P.tw, (uint32_t)m1[side]);
            w1.y = -w1.y;
            const int64_t slot = side ? fft::mirror_half_slots(P.log2w) + ((far_top - m1[1]) & (P.Lh - 1))
                                      : ((m1[0] - near_origin) & (P.Lh - 1));
#pragma unroll
            for (int s = 0; s < 3; s++) {
                double2 z[G];
#pragma unroll
                for (int r = 0; r < G; r++) z[r] = P.recv[(int64_t)(s * G + r) * stride + slot];
                fft::apply_powers<G>(z, w1);
                fft::Dft<G, +1>::run(z);
#pragma unroll
                for (int q = 0; q < GH; q++) power[side][q] += z[q].x * z[q].x + z[q].y * z[q].y;
            }
        }
#pragma unroll
        for (int q = 0; q < GH; q++) {
            const int64_t m = (int64_t)q * P.Lh + m1[0];
            if (m < 1 || m >= P.M) continue;
            const int64_t m2 = P.M - m;  // its residue is m1[1]
            const int q2 = (int)(m2 >> P.log2lh);
            double partner = 0.0;
#pragma unroll
            for (int j = 0; j < GH; j++)
                if (j == q2) partner = power[1][j];
            const int64_t k = m < m2 ? m : m2;
            if (k > P.points) continue;  // the middle bin of an even M is not part of the spectrum
            const double first = m < m2 ? power[0][q] : partner, second = m < m2 ? partner : power[0][q];
            double inten = (first + second) * P.scale + econst;  // (P[k] + P[M-k]) in that order
            inten = corrected(inten, wavenumber_of(k, P.M, P.prm.timestep), P.prm);
            for (int d = 0; d < P.num_dest; d++) P.dest[d][kSpecHeader + k - 1] = inten;
        }
    }
    if (P.wn_out)  // the wavenumbers do not travel: every rank writes its own while the stores above drain
        for (int64_t o = local; o < P.points; o += (int64_t)gridDim.x * blockDim.x)
            P.wn_out[o] = wavenumber_of(o + 1, P.M, P.prm.timestep);
}

// after the last barrier: the finished intensities out of the spectrum buffer (and, for ranks that did not run
// the final stage, the wavenumbers)
__global__ void __launch_bounds__(256) finish_dist_kernel(const double* __restrict__ spec, int64_t points, int64_t M,
                                                          double timestep, double* __restrict__ wn_out,
                                                          double* __restrict__ int_out) {
    for (int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; o < points; o += (int64_t)gridDim.x * blockDim.x) {
        int_out[o] = spec[kSpecHeader + o];
        if (wn_out) wn_out[o] = wavenumber_of(o + 1, M, timestep);
    }
}

// I[k] = (P[k] + P[M-k]) / (4 L^2) + E/2 for k = 1 .. ceil(M/2)-1 (bin 0 dropped, _raman.py:299-301),
// wavenumbers, laser / Bose-Einstein corrections (_raman.py:13-69,303-307).  power: (nseq, M);
// epart: nparts energy partials summed in a fixed order by every block.
// WIN: blockIdx.y numbers a window of a batch; window w reads sequences nseq w .. nseq w + nseq - 1 of power,
// the partials at epart + w epart_stride, writes row w of int_out (points per row) and, for w = 0 only and
// if wn_out is given, the wavenumbers.
template <bool WIN = false>
__global__ void __launch_bounds__(256) combine_md_kernel(const double* __restrict__ power, int nseq,
                                                         const double* __restrict__ epart, int nparts, int64_t M,
                                                         double scale, int64_t points, SpectrumParams prm,
                                                         double* __restrict__ wn_out, double* __restrict__ int_out,
                                                         int64_t epart_stride = 0) {
    __shared__ double red[8];
    __shared__ double s_energy;
    if constexpr (WIN) {
        power += (int64_t)blockIdx.y * nseq * M;
        epart += (int64_t)blockIdx.y * epart_stride;
        int_out += (int64_t)blockIdx.y * points;
        if (blockIdx.y != 0) wn_out = nullptr;
    }
    double v = 0.0;
    for (int b = threadIdx.x; b < nparts; b += blockDim.x) v += epart[b];
    const double total = block_sum(v, red);
    if (threadIdx.x == 0) s_energy = total;
    __syncthreads();
    const double econst = 0.5 * s_energy;
    for (int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; o < points; o += (int64_t)gridDim.x * blockDim.x) {
        const int64_t k = o + 1;
        double sum = 0.0;
        for (int s = 0; s < nseq; s++) sum += power[(int64_t)s * M + k] + power[(int64_t)s * M + (M - k)];
        const double wn = wavenumber_of(k, M, prm.timestep);
        if (!WIN || wn_out) wn_out[o] = wn;
        int_out[o] = corrected(sum * scale + econst, wn, prm);
    }
}

// calc_signal_spectrum for one real signal: I[k] = (|X[k]|^2 + E)/2, k = 0 .. ceil(M/2)-1
__global__ void __launch_bounds__(256) combine_signal_kernel(const double* __restrict__ power,
                                                             const double* __restrict__ epart, int nparts, int64_t M,
                                                             double scale, int64_t points, double dt,
                                                             double* __restrict__ wn_out, double* __restrict__ int_out) {
    __shared__ double red[8];
    __shared__ double s_energy;
    double v = 0.0;
    for (int b = threadIdx.x; b < nparts; b += blockDim.x) v += epart[b];
    const double total = block_sum(v, red);
    if (threadIdx.x == 0) s_energy = total;
    __syncthreads();
    const double econst = 0.5 * s_energy;
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < points; k += (int64_t)gridDim.x * blockDim.x) {
        int_out[k] = power[k] * scale + econst;
        wn_out[k] = wavenumber_of(k, M, dt);
    }
}

// ---- cross spectra of G series (rn_md_cross_spectra) ----------------------------------------------
// The orientational average is a sum of squares, so it polarizes into a symmetric bilinear form: with the
// six weighted signals of the pack and X the length-M DFT,
//   I_gh[k] = 1/2 sum_p (Re(X_gp[k] conj X_hp[k]) + E_gh),   E_gh = sum_p sum_n x_gp[n] x_hp[n],
// and for packed Z = A + iB,  Re(Z_g Z_h*)[k] + Re(Z_g Z_h*)[M-k] = 2 Re(A_g A_h* + B_g B_h*)[k].  The chirp
// post-factor has modulus 1 and is the same for every sequence at bin m, so the products of the transform
// outputs y are those of the spectra: I_gh[k] = C[k] / (4 L^2) + E_gh / 2 with
//   C[k] = sum_s Re(y_gs[k] conj y_hs[k]) + Re(y_gs[M-k] conj y_hs[M-k]).

constexpr int kCrossTile = 4;  // series whose signals a thread of cross_energy_kernel holds at once

// pair (g, h), g < h, in row-major order of the strict upper triangle
__device__ __forceinline__ int64_t upper_pair(int64_t g, int64_t h, int64_t G) {
    return g * (2 * G - g - 1) / 2 + (h - g - 1);
}

// the six weighted difference signals of frame n (rows r0 = n, r1 = n + 1), the formulas of pack_alpha_kernel
__device__ __forceinline__ void md_signals(const double* __restrict__ r0, double z[6]) {
    const double* r1 = r0 + 9;
    const double xx = __ldg(r1 + 0) - __ldg(r0 + 0), yy = __ldg(r1 + 4) - __ldg(r0 + 4);
    const double zz = __ldg(r1 + 8) - __ldg(r0 + 8), xy = __ldg(r1 + 1) - __ldg(r0 + 1);
    const double yz = __ldg(r1 + 5) - __ldg(r0 + 5), xz = __ldg(r1 + 2) - __ldg(r0 + 2);
    z[0] = kSqrt5 * (xx + yy + zz);
    z[1] = kSqrt5_25 * (xx - zz);
    z[2] = kSqrt1_75 * (xx - 2.0 * yy + zz);
    z[3] = kSqrt21 * xy;
    z[4] = kSqrt21 * yz;
    z[5] = kSqrt21 * xz;
}

// E_gh for every pair g < h of the G series at src + g stride (one frame per thread).  Block b leaves the
// partial of pair p in part[p gridDim.x + b]; the block that finishes last sums every pair's partials in
// block order (bit-reproducible whichever block that is) into energy[p] and re-arms the ticket.  The diagonal
// energies are the pack's.
__global__ void __launch_bounds__(256) cross_energy_kernel(const double* __restrict__ src, int64_t stride, int G,
                                                           int64_t M, double* __restrict__ part,
                                                           double* __restrict__ energy, unsigned int* ticket) {
    __shared__ double red[kCrossTile][8];
    __shared__ bool last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (int g0 = 0; g0 < G - 1; g0 += kCrossTile) {
        double zg[kCrossTile][6];
#pragma unroll
        for (int r = 0; r < kCrossTile; r++) {
#pragma unroll
            for (int i = 0; i < 6; i++) zg[r][i] = 0.0;
            if (n < M && g0 + r < G) md_signals(src + (int64_t)(g0 + r) * stride + n * 9, zg[r]);
        }
        for (int h = g0 + 1; h < G; h++) {
            double zh[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
            if (n < M) md_signals(src + (int64_t)h * stride + n * 9, zh);
#pragma unroll
            for (int r = 0; r < kCrossTile; r++) {
                double v = (zg[r][0] * zh[0] + zg[r][1] * zh[1]) + (zg[r][2] * zh[2] + zg[r][3] * zh[3]) +
                           (zg[r][4] * zh[4] + zg[r][5] * zh[5]);
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
                if (lane == 0) red[r][warp] = v;
            }
            __syncthreads();
            if (threadIdx.x < kCrossTile && g0 + (int)threadIdx.x < h) {
                const int r = threadIdx.x;
                double total = 0.0;
                for (int w = 0; w < (int)(blockDim.x >> 5); w++) total += red[r][w];
                part[upper_pair(g0 + r, h, G) * gridDim.x + blockIdx.x] = total;
                __threadfence();
            }
            __syncthreads();  // `red` is reused
        }
    }
    if (threadIdx.x == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    const int64_t pairs = (int64_t)G * (G - 1) / 2;
    for (int64_t p = warp; p < pairs; p += blockDim.x >> 5) {
        double v = 0.0;
        for (unsigned int b = lane; b < gridDim.x; b += 32) v += __ldcg(part + p * gridDim.x + b);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        if (lane == 0) energy[p] = v;
    }
    if (threadIdx.x == 0) *ticket = 0;
}

// Re(a conj b) in the form store_out gives |v|^2 (v.x*v.x + v.y*v.y), so that a == b reproduces the power
__device__ __forceinline__ double re_dot(double2 a, double2 b) { return a.x * b.x + a.y * b.y; }

// I_gh[k], k = 1 .. points, for every pair g <= h, into rows (g, h) and (h, g) of int_out (G, G, points).
// y: the 3 G transform outputs (natural order, sequence 3g + s of series g at y + (3g + s) Lh).  Row g of the
// grid (strided by gridDim.y) holds its own y at bins k and M-k and pairs it with every h >= g.  The sums
// over s and the final scale run in the order of combine_md_kernel and the diagonal energy is the pack's, so
// row (g, g) is bit-identical to rn_md_spectrum of series g.
__global__ void __launch_bounds__(256) cross_combine_kernel(const double2* __restrict__ y, int64_t Lh, int G,
                                                            const double* __restrict__ epart, int64_t epart_stride,
                                                            const double* __restrict__ energy, int64_t M,
                                                            double scale, int64_t points, SpectrumParams prm,
                                                            double* __restrict__ wn_out, double* __restrict__ int_out) {
    for (int64_t g = blockIdx.y; g < G; g += gridDim.y) {
        const double2* yg = y + 3 * g * Lh;
        for (int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; o < points;
             o += (int64_t)gridDim.x * blockDim.x) {
            const int64_t k = o + 1;
            double2 a[3][2];
#pragma unroll
            for (int s = 0; s < 3; s++) {
                a[s][0] = yg[s * Lh + k];
                a[s][1] = yg[s * Lh + (M - k)];
            }
            const double wn = wavenumber_of(k, M, prm.timestep);
            if (g == 0) wn_out[o] = wn;
            for (int64_t h = g; h < G; h++) {
                const double2* yh = y + 3 * h * Lh;
                double sum = 0.0;
#pragma unroll
                for (int s = 0; s < 3; s++)  // __dadd_rn: no product may fuse into these sums
                    sum = __dadd_rn(sum, __dadd_rn(re_dot(a[s][0], yh[s * Lh + k]), re_dot(a[s][1], yh[s * Lh + (M - k)])));
                const double e = h == g ? epart[g * epart_stride] : energy[upper_pair(g, h, G)];
                const double econst = 0.5 * e;
                const double inten = corrected(sum * scale + econst, wn, prm);
                int_out[(g * G + h) * points + o] = inten;
                if (h != g) int_out[(h * G + g) * points + o] = inten;
            }
        }
    }
}

// ---- vibrational density of states (rn_vdos) -------------------------------------------------------
// The VDOS of a group is sum_{atoms i} w_i sum_c calc_signal_spectrum(v_ic) with v the minimum-image velocity
// (d @ lattice) / dt.  A slot holds two memberships a, b of one group: its six real signals sqrt(w) v_c of a
// and of b packed as z_c = (x_a + i x_b)_c are the three sequences of one window of a batched plan, so the
// identity of combine_md_kernel gives the slot's term (P[k] + P[M-k]) / (4 L^2) + E/2 unchanged.

struct VdosSlot {
    int atom[2];      // -1: the zero signal that pads a group of odd size
    double sqrtw[2];  // sqrt(weight) of each membership
};

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
    const int64_t frame_stride = 3 * P.num_atoms;
    for (int e = threadIdx.x; e < (kPackThreads + 1) * 6; e += kPackThreads) {
        const int f = e / 6, j = e - 6 * (e / 6);
        const int atom = j < 3 ? slot.atom[0] : slot.atom[1];
        rows[e] = (f < avail && atom >= 0) ? __ldg(P.pos + (first + f) * frame_stride + 3 * atom + (j < 3 ? j : j - 3))
                                           : 0.0;
    }
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
    if (wn_out && blockIdx.y == 0)
        for (int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; o < points;
             o += (int64_t)gridDim.x * blockDim.x)
            wn_out[o] = wavenumber_of(o + 1, M, dt);
}

static int grid_for(int64_t n, int sms) {
    return (int)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)sms * 16));
}

// ---- host side of the convolution core ------------------------------------------------------------
static int ensure_smem_attr(int device) {
    static std::atomic<bool> done[64];  // the attribute is per function and per device
    if (device >= 0 && device < 64 && done[device].load(std::memory_order_acquire)) return RN_OK;
#define RN_FFT_SMEM(kern) \
    RN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fft::kTileSmemBytes))
    RN_FFT_SMEM((fft::tile_kernel<false, false>));
    RN_FFT_SMEM((fft::tile_kernel<false, true>));
    RN_FFT_SMEM((fft::tile_kernel<true, false>));
    RN_FFT_SMEM((fft::level_kernel<-1, false>));
    RN_FFT_SMEM((fft::level_kernel<-1, true>));
    RN_FFT_SMEM((fft::level_kernel<+1, false>));
    RN_FFT_SMEM((fft::level_kernel<+1, true>));
#undef RN_FFT_SMEM
    if (device >= 0 && device < 64) done[device].store(true, std::memory_order_release);
    return RN_OK;
}

// kernel variant: bit 0 = lean level kernels, bit 1 = lean tile kernel (RN_FFT_LEAN, read once; tuning)
static int fft_lean() {
    static const int value = [] {
        // measured on B200 (S = 1e6): 0.252 ms with the unrolled variants (2 CTAs/SM, 126 registers),
        // 0.232 ms with the lean ones (3 CTAs/SM, 80 registers)
        const char* env = getenv("RN_FFT_LEAN");
        return env ? atoi(env) : 3;
    }();
    return value;
}

static fft::OutSpec plain_out() {
    fft::OutSpec o;
    o.mode = fft::OUT_PLAIN;
    o.power = nullptr;
    o.M = 0;
    for (int i = 0; i < 8; i++) o.peers.ptr[i] = nullptr;
    o.peers.log2w = 0;
    o.peers.rank = 0;
    o.peers.world = 1;
    return o;
}

template <int SGN>
static int launch_level(const rn_spectrum_plan* p, double2* X, int nseq, int seq_base, int lev, int64_t limit,
                        const fft::OutSpec& out, cudaStream_t stream) {
    fft::LevelParams P;
    P.X = X;
    P.seq_base = seq_base;
    P.seq_stride = p->Lh;
    int log2lsub = p->log2lh;
    for (int i = 0; i < lev; i++) log2lsub -= p->lev_log2r[i];
    P.log2lsub = log2lsub;
    P.log2r = p->lev_log2r[lev];
    P.nsub = (int)(p->Lh >> log2lsub);
    P.tw_shift = p->log2l - log2lsub;
    P.limit = limit;
    P.out = out;
    P.tw = plan_twiddles(p);
    const int64_t grid = (int64_t)nseq * (p->Lh >> kLog2E);
    if (fft_lean() & 1) fft::level_kernel<SGN, true><<<(unsigned)grid, kNT, fft::kTileSmemBytes, stream>>>(P);
    else fft::level_kernel<SGN, false><<<(unsigned)grid, kNT, fft::kTileSmemBytes, stream>>>(P);
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    return RN_OK;
}

// forward levels, tile pass (with the filter), inverse levels: X (nseq, Lh) in place.  `limit`: input
// elements at or beyond it are zero (never read); `out`: where the inverse transform's result goes.
// hout != nullptr: forward transform only, written to hout (plan creation: the filter spectrum).
static int run_convolution(const rn_spectrum_plan* p, double2* X, int nseq, int64_t limit, const fft::OutSpec& out,
                           double2* hout, cudaStream_t stream, int seq_base = 0) {
    int rc = ensure_smem_attr(p->device);
    if (rc != RN_OK) return rc;
    const fft::OutSpec plain = plain_out();
    for (int lev = 0; lev < p->nlev; lev++) {
        rc = launch_level<-1>(p, X, nseq, seq_base, lev, lev == 0 ? limit : p->Lh, plain, stream);
        if (rc != RN_OK) return rc;
    }
    fft::TileParams T;
    T.X = X;
    T.seq_stride = p->Lh;
    T.tiles_per_seq = (int)(p->Lh >> kLog2E);
    T.H = p->d_H;
    T.Hout = hout;
    T.limit = p->nlev == 0 ? limit : p->Lh;
    T.seq_base = seq_base;
    T.out = p->nlev == 0 ? out : plain;
    T.tw = plan_twiddles(p);
    const unsigned grid = (unsigned)((int64_t)nseq * T.tiles_per_seq);
    if (hout) fft::tile_kernel<true, false><<<grid, kNT, fft::kTileSmemBytes, stream>>>(T);
    else if (fft_lean() & 2) fft::tile_kernel<false, true><<<grid, kNT, fft::kTileSmemBytes, stream>>>(T);
    else fft::tile_kernel<false, false><<<grid, kNT, fft::kTileSmemBytes, stream>>>(T);
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    if (hout) return RN_OK;
    for (int lev = p->nlev - 1; lev >= 0; lev--) {
        rc = launch_level<+1>(p, X, nseq, seq_base, lev, p->Lh, lev == 0 ? out : plain, stream);
        if (rc != RN_OK) return rc;
    }
    return RN_OK;
}

static void destroy_plan(rn_spectrum_plan* p) {
    if (!p) return;
    cudaFree(p->d_whi);
    cudaFree(p->d_wlo);
    cudaFree(p->d_wsub);
    cudaFree(p->d_H);
    cudaFree(p->d_work);
    cudaFree(p->d_power);
    cudaFree(p->d_epart);
    cudaFree(p->d_ticket);
    cudaFree(p->d_cross);
    cudaFree(p->d_vdos);
    delete p;
}

// exp(-2 pi i num/den) in 80-bit arithmetic
static double2 unit_root(int64_t num, int64_t den) {
    const long double two_pi = 6.283185307179586476925286766559005768L;
    const long double ang = two_pi * (long double)num / (long double)den;
    return make_double2((double)cosl(ang), (double)-sinl(ang));
}

// largest batch of windows: gridDim.y of the windowed pack and combine
constexpr int64_t kMaxBatch = 65535;

static int create_plan(int64_t num_frames, int device, int world, int rank, rn_spectrum_plan** out,
                       int64_t batch = 1) {
    RN_CHECK_ARG(out != nullptr, "out is null");
    *out = nullptr;
    RN_CHECK_ARG(num_frames >= 2, "a spectrum needs at least 2 frames (got %lld)", (long long)num_frames);
    RN_CHECK_ARG(world >= 1 && world <= 8 && rank >= 0 && rank < world, "invalid rank %d of %d", rank, world);
    RN_CHECK_ARG(batch >= 1 && batch <= kMaxBatch && (batch == 1 || world == 1),
                 "invalid batch %lld (1 .. %lld windows, single-GPU plans only)", (long long)batch,
                 (long long)kMaxBatch);
    int count = 0;
    RN_CUDA(cudaGetDeviceCount(&count));
    RN_CHECK_ARG(device >= 0 && device < count, "device %d out of range (%d devices)", device, count);
    DeviceGuard guard(device);
    if (!guard.ok) {
        set_error("cudaSetDevice(%d) failed", device);
        return RN_ERR_CUDA;
    }
    cudaDeviceProp prop;
    RN_CUDA(cudaGetDeviceProperties(&prop, device));
    // the transform is shared by the largest power-of-two number of ranks; the others are spectators
    int group = 1;
    while (group * 2 <= world) group *= 2;
    const int64_t M = num_frames - 1;
    int log2l = kLog2E;
    while (((int64_t)1 << log2l) < std::max<int64_t>(2 * M - 1, (int64_t)kE * group)) log2l++;
    RN_CHECK_ARG(log2l <= 30, "series too long for one spectrum plan (%lld frames)", (long long)num_frames);
    // the level and tile passes launch 3 batch L / 4096 blocks along gridDim.x
    RN_CHECK_ARG(3 * batch * (((int64_t)1 << log2l) >> kLog2E) <= (int64_t)INT32_MAX,
                 "batch %lld too large for windows of %lld frames", (long long)batch, (long long)num_frames);
    rn_spectrum_plan* p = new rn_spectrum_plan();
    p->batch = batch;
    p->device = device;
    p->sm_count = prop.multiProcessorCount;
    p->S = num_frames;
    p->M = M;
    p->log2l = log2l;
    p->L = (int64_t)1 << log2l;
    p->world = group;
    p->rank = rank;
    p->Lh = p->L / group;
    p->log2lh = log2l;
    for (int g = group; g > 1; g >>= 1) p->log2lh--;
    const int q = p->log2lh - kLog2E;
    if (q == 0) {
        p->nlev = 0;
    } else if (q <= 10) {
        p->nlev = 1;
        p->lev_log2r[0] = q;
    } else {
        p->nlev = 2;
        p->lev_log2r[0] = (q + 1) / 2;
        p->lev_log2r[1] = q - p->lev_log2r[0];
    }
    const int64_t owned = rank < group ? (group > 1 ? p->Lh / group : M) : 0;  // n' this rank packs
    p->pack_blocks = (int)((owned + kPackThreads - 1) / kPackThreads);
    if (rank >= group) {  // spectator: combines what the group sends, owns nothing else
        *out = p;
        return RN_OK;
    }
    p->split = log2l / 2;
    const int64_t n_hi = p->L >> p->split, n_lo = (int64_t)1 << p->split;
    cudaError_t err = cudaSuccess;
    auto alloc = [&](void** ptr, size_t bytes) {
        if (err == cudaSuccess) err = cudaMalloc(ptr, bytes);
    };
    alloc((void**)&p->d_whi, sizeof(double2) * n_hi);
    alloc((void**)&p->d_wlo, sizeof(double2) * n_lo);
    alloc((void**)&p->d_wsub, sizeof(double2) * kE);
    alloc((void**)&p->d_H, sizeof(double2) * p->Lh);
    // partials and tickets: two pack phases (shared transforms) or one set per window
    const int64_t psets = std::max<int64_t>(2, batch);
    alloc((void**)&p->d_work, sizeof(double2) * (group > 1 ? 1 : 3 * batch) * p->Lh);
    if (group == 1) alloc((void**)&p->d_power, sizeof(double) * 3 * batch * M);
    alloc((void**)&p->d_epart, sizeof(double) * psets * (p->pack_blocks + 1));
    alloc((void**)&p->d_ticket, psets * sizeof(unsigned int));
    if (err != cudaSuccess) {
        set_error("cudaMalloc failed while creating a spectrum plan for %lld frames: %s", (long long)num_frames,
                  cudaGetErrorString(err));
        destroy_plan(p);
        cudaGetLastError();
        return RN_ERR_OUT_OF_MEMORY;
    }
    cudaMemset(p->d_ticket, 0, psets * sizeof(unsigned int));
    std::vector<double2> whi((size_t)n_hi), wlo((size_t)n_lo), wsub((size_t)kE);
    for (int64_t a = 0; a < n_hi; a++) whi[(size_t)a] = unit_root(a << p->split, p->L);
    for (int64_t b = 0; b < n_lo; b++) wlo[(size_t)b] = unit_root(b, p->L);
    for (int m = 0; m < kE; m++) wsub[(size_t)m] = unit_root(m, kE);
    cudaError_t e1 = cudaMemcpy(p->d_whi, whi.data(), sizeof(double2) * n_hi, cudaMemcpyHostToDevice);
    if (e1 == cudaSuccess) e1 = cudaMemcpy(p->d_wlo, wlo.data(), sizeof(double2) * n_lo, cudaMemcpyHostToDevice);
    if (e1 == cudaSuccess) e1 = cudaMemcpy(p->d_wsub, wsub.data(), sizeof(double2) * kE, cudaMemcpyHostToDevice);
    if (e1 != cudaSuccess) {
        set_error("twiddle table upload failed: %s", cudaGetErrorString(e1));
        destroy_plan(p);
        return RN_ERR_CUDA;
    }
    // filter spectrum of this rank's residue, left in the order the forward transform produces
    filter_fill_kernel<<<grid_for(p->Lh, p->sm_count), 256>>>(p->d_work, M, p->L, p->Lh, group, rank, plan_twiddles(p));
    RN_LAUNCHED();
    int rc = run_convolution(p, p->d_work, 1, p->Lh, plain_out(), p->d_H, nullptr);
    if (rc == RN_OK) {
        cudaError_t e2 = cudaStreamSynchronize(nullptr);
        if (e2 != cudaSuccess) {
            set_error("spectrum plan initialisation failed: %s", cudaGetErrorString(e2));
            rc = RN_ERR_CUDA;
        }
    }
    if (rc != RN_OK) {
        destroy_plan(p);
        return rc;
    }
    if (group > 1) {  // shared transforms run in the caller's (peer-visible) buffers
        cudaFree(p->d_work);
        p->d_work = nullptr;
    }
    *out = p;
    return RN_OK;
}

static SpectrumParams spectrum_params(double timestep_fs, int laser, double laser_wavelength_nm, int be,
                                      double temperature_K) {
    SpectrumParams prm;
    prm.timestep = timestep_fs;
    prm.laser = laser ? 1 : 0;
    prm.laser_wavenumber = laser ? 10000000.0 / laser_wavelength_nm : 0.0;
    prm.bose_einstein = be ? 1 : 0;
    prm.kt = 8.617333262e-5 * temperature_K;  // constants.py:249
    return prm;
}

// pack of one whole (S,3,3) series on a single-GPU plan into its first work buffer
static PackParams md_pack_params(const rn_spectrum_plan* plan, const double* d_alpha) {
    PackParams pp;
    pp.src = d_alpha;
    pp.M = plan->M;
    pp.Lh = plan->Lh;
    pp.begin = 0;
    pp.end = plan->M;
    for (int i = 0; i < 8; i++) pp.dst[i] = nullptr;
    pp.dst[0] = plan->d_work;
    pp.aligned16 = (reinterpret_cast<uintptr_t>(pp.src) % 16 == 0) ? 1 : 0;
    pp.seq_sel = -1;
    pp.num_share = 0;
    pp.share_slot = 0;
    pp.zero_slot = -1;
    pp.log2_stripe = -1;
    pp.phase = 0;
    for (int i = 0; i < 8; i++) pp.share[i] = nullptr;
    pp.epart = plan->d_epart;
    pp.ticket = plan->d_ticket;
    pp.tw = plan_twiddles(plan);
    pp.win_stride = 0;
    return pp;
}

}  // namespace rn

using namespace rn;

extern "C" int64_t rn_spectrum_num_points(int64_t num_frames) {
    const int64_t M = num_frames - 1;
    if (M < 1) return 0;
    return (M + 1) / 2 - 1;
}

extern "C" int rn_spectrum_plan_create(int64_t num_frames, int device, rn_spectrum_plan** out) {
    return create_plan(num_frames, device, 1, 0, out);
}

extern "C" int rn_spectrum_plan_create_batched(int64_t window_frames, int64_t batch, int device,
                                               rn_spectrum_plan** out) {
    return create_plan(window_frames, device, 1, 0, out, batch);
}

extern "C" int rn_spectrum_plan_create_dist(int64_t num_frames, int device, int world, int rank,
                                            rn_spectrum_plan** out) {
    return create_plan(num_frames, device, world, rank, out);
}

extern "C" int rn_spectrum_plan_destroy(rn_spectrum_plan* plan) {
    if (!plan) return RN_OK;
    DeviceGuard guard(plan->device);
    destroy_plan(plan);
    return RN_OK;
}

extern "C" int rn_spectrum_plan_info(const rn_spectrum_plan* plan, int64_t info[8]) {
    RN_CHECK_ARG(plan != nullptr && info != nullptr, "null pointer");
    info[0] = plan->log2l;
    info[1] = plan->world;
    info[2] = plan->log2lh;
    info[3] = plan->nlev;
    info[4] = plan->lev_log2r[0];
    info[5] = plan->lev_log2r[1];
    info[6] = plan->world > 1 ? plan->Lh / plan->world : plan->Lh;  // block of n' / m' one rank owns
    info[7] = plan->M;
    return RN_OK;
}

extern "C" int rn_md_spectrum(rn_spectrum_plan* plan, const double* d_alpha, double timestep_fs, int laser_correction,
                              double laser_wavelength_nm, int bose_einstein_correction, double temperature_K,
                              double* d_wavenumbers, double* d_intensities, void* stream) {
    RN_CHECK_ARG(plan != nullptr, "plan is null");
    RN_CHECK_ARG(plan->world == 1, "rn_md_spectrum needs a single-GPU plan (rn_spectrum_plan_create)");
    RN_CHECK_ARG(d_alpha != nullptr, "d_alpha is null");
    RN_CHECK_ARG(timestep_fs > 0, "timestep must be positive");
    if (laser_correction) RN_CHECK_ARG(laser_wavelength_nm > 0, "invalid laser_wavelength");
    if (bose_einstein_correction) RN_CHECK_ARG(temperature_K > 0, "invalid temperature: %g <= 0", temperature_K);
    const int64_t points = rn_spectrum_num_points(plan->S);
    if (points == 0) return RN_OK;
    RN_CHECK_ARG(d_wavenumbers && d_intensities, "null output pointer");
    DeviceGuard guard(plan->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int64_t M = plan->M;

    const PackParams pp = md_pack_params(plan, d_alpha);
    pack_alpha_kernel<1><<<plan->pack_blocks, kPackThreads, 0, s>>>(pp);
    RN_LAUNCHED();
    fft::OutSpec out = plain_out();
    out.mode = fft::OUT_POWER;
    out.power = plan->d_power;
    out.M = M;
    int rc = run_convolution(plan, plan->d_work, 3, M, out, nullptr, s);
    if (rc != RN_OK) return rc;
    const SpectrumParams prm = spectrum_params(timestep_fs, laser_correction, laser_wavelength_nm,
                                               bose_einstein_correction, temperature_K);
    const double scale = 0.25 / ((double)plan->L * (double)plan->L);
    combine_md_kernel<<<grid_for(points, plan->sm_count), 256, 0, s>>>(plan->d_power, 3, plan->d_epart + plan->pack_blocks, 1,
                                                                      M, scale, points, prm, d_wavenumbers, d_intensities);
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    return RN_OK;
}

// Every window of a batch runs the arithmetic of rn_md_spectrum on its slice in the same order: the pack
// reads it at its own offset and sums its energy with its own partials, the convolution treats the 3 nb
// sequences independently, the combine reads its own three rows of power and its own energy.
extern "C" int rn_md_spectrum_windows(rn_spectrum_plan* plan, const double* d_alpha, int64_t num_frames,
                                      int64_t hop_frames, double timestep_fs, int laser_correction,
                                      double laser_wavelength_nm, int bose_einstein_correction, double temperature_K,
                                      double* d_wavenumbers, double* d_intensities, void* stream) {
    RN_CHECK_ARG(plan != nullptr, "plan is null");
    RN_CHECK_ARG(plan->world == 1, "rn_md_spectrum_windows needs a single-GPU plan (rn_spectrum_plan_create_batched)");
    RN_CHECK_ARG(d_alpha != nullptr, "d_alpha is null");
    RN_CHECK_ARG(num_frames >= plan->S, "a window of %lld frames does not fit a series of %lld frames",
                 (long long)plan->S, (long long)num_frames);
    RN_CHECK_ARG(hop_frames >= 1, "hop_frames must be at least 1 (got %lld)", (long long)hop_frames);
    RN_CHECK_ARG(timestep_fs > 0, "timestep must be positive");
    if (laser_correction) RN_CHECK_ARG(laser_wavelength_nm > 0, "invalid laser_wavelength");
    if (bose_einstein_correction) RN_CHECK_ARG(temperature_K > 0, "invalid temperature: %g <= 0", temperature_K);
    const int64_t points = rn_spectrum_num_points(plan->S);
    if (points == 0) return RN_OK;
    RN_CHECK_ARG(d_wavenumbers && d_intensities, "null output pointer");
    DeviceGuard guard(plan->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int64_t M = plan->M;
    const int64_t windows = 1 + (num_frames - plan->S) / hop_frames;
    const SpectrumParams prm = spectrum_params(timestep_fs, laser_correction, laser_wavelength_nm,
                                               bose_einstein_correction, temperature_K);
    const double scale = 0.25 / ((double)plan->L * (double)plan->L);
    for (int64_t first = 0; first < windows; first += plan->batch) {
        const int64_t nb = std::min(plan->batch, windows - first);
        PackParams pp = md_pack_params(plan, d_alpha + first * hop_frames * 9);
        pp.win_stride = hop_frames * 9;
        pack_alpha_kernel<1, true><<<dim3(plan->pack_blocks, (unsigned)nb), kPackThreads, 0, s>>>(pp);
        RN_LAUNCHED();
        fft::OutSpec out = plain_out();
        out.mode = fft::OUT_POWER;
        out.power = plan->d_power;
        out.M = M;
        int rc = run_convolution(plan, plan->d_work, (int)(3 * nb), M, out, nullptr, s);
        if (rc != RN_OK) return rc;
        combine_md_kernel<true><<<dim3(grid_for(points, plan->sm_count), (unsigned)nb), 256, 0, s>>>(
            plan->d_power, 3, plan->d_epart + plan->pack_blocks, 1, M, scale, points, prm,
            first == 0 ? d_wavenumbers : nullptr, d_intensities + first * points, plan->pack_blocks + 1);
        RN_LAUNCHED();
        RN_CUDA(cudaGetLastError());
    }
    return RN_OK;
}

// The G series are the windows of hop S over the (G,S,3,3) array: the windowed pack leaves the chirped signals
// of series g in sequences 3g .. 3g+2 and its energy in its own partials, the convolution keeps every output
// y (OUT_PLAIN), and the two cross kernels form every pair from them.
extern "C" int rn_md_cross_spectra(rn_spectrum_plan* plan, const double* d_alpha, int64_t num_series,
                                   double timestep_fs, int laser_correction, double laser_wavelength_nm,
                                   int bose_einstein_correction, double temperature_K, double* d_wavenumbers,
                                   double* d_intensities, void* stream) {
    RN_CHECK_ARG(plan != nullptr, "plan is null");
    RN_CHECK_ARG(plan->world == 1, "rn_md_cross_spectra needs a single-GPU plan (rn_spectrum_plan_create_batched)");
    RN_CHECK_ARG(d_alpha != nullptr, "d_alpha is null");
    RN_CHECK_ARG(num_series >= 1 && num_series <= plan->batch,
                 "num_series must be 1 .. %lld (the plan's batch), got %lld", (long long)plan->batch,
                 (long long)num_series);
    RN_CHECK_ARG(timestep_fs > 0, "timestep must be positive");
    if (laser_correction) RN_CHECK_ARG(laser_wavelength_nm > 0, "invalid laser_wavelength");
    if (bose_einstein_correction) RN_CHECK_ARG(temperature_K > 0, "invalid temperature: %g <= 0", temperature_K);
    const int64_t points = rn_spectrum_num_points(plan->S);
    if (points == 0) return RN_OK;
    RN_CHECK_ARG(d_wavenumbers && d_intensities, "null output pointer");
    DeviceGuard guard(plan->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int64_t M = plan->M;
    const int G = (int)num_series;
    const int64_t energy_blocks = (M + 255) / 256;
    const int64_t pairs = (int64_t)G * (G - 1) / 2;
    const int64_t need = pairs * (energy_blocks + 1);
    if (need > plan->cross_doubles) {  // kept with the plan; calls on one plan are ordered on one stream
        RN_CUDA(cudaStreamSynchronize(s));
        cudaFree(plan->d_cross);
        plan->d_cross = nullptr;
        plan->cross_doubles = 0;
        if (cudaMalloc((void**)&plan->d_cross, sizeof(double) * need) != cudaSuccess) {
            cudaGetLastError();
            set_error("cudaMalloc of %lld bytes of cross-energy partials failed", (long long)(sizeof(double) * need));
            return RN_ERR_OUT_OF_MEMORY;
        }
        plan->cross_doubles = need;
    }
    PackParams pp = md_pack_params(plan, d_alpha);
    pp.win_stride = plan->S * 9;
    pack_alpha_kernel<1, true><<<dim3(plan->pack_blocks, (unsigned)G), kPackThreads, 0, s>>>(pp);
    RN_LAUNCHED();
    int rc = run_convolution(plan, plan->d_work, 3 * G, M, plain_out(), nullptr, s);
    if (rc != RN_OK) return rc;
    double* energy = plan->d_cross + pairs * energy_blocks;
    if (G > 1) {
        cross_energy_kernel<<<(unsigned)energy_blocks, 256, 0, s>>>(d_alpha, plan->S * 9, G, M, plan->d_cross, energy,
                                                                    plan->d_ticket);
        RN_LAUNCHED();
    }
    const SpectrumParams prm = spectrum_params(timestep_fs, laser_correction, laser_wavelength_nm,
                                               bose_einstein_correction, temperature_K);
    const double scale = 0.25 / ((double)plan->L * (double)plan->L);
    cross_combine_kernel<<<dim3(grid_for(points, plan->sm_count), (unsigned)std::min(G, 65535)), 256, 0, s>>>(
        plan->d_work, plan->Lh, G, plan->d_epart + plan->pack_blocks, plan->pack_blocks + 1, energy, M, scale, points,
        prm, d_wavenumbers, d_intensities);
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    return RN_OK;
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
    RN_CHECK_ARG(h_group_offsets[0] == 0, "group offsets must start at 0");
    std::vector<int64_t> group_slots((size_t)num_groups + 1, 0);
    for (int64_t g = 0; g < num_groups; g++) {
        const int64_t size = h_group_offsets[g + 1] - h_group_offsets[g];
        RN_CHECK_ARG(size >= 1, "group %lld is empty", (long long)g);
        group_slots[(size_t)g + 1] = group_slots[(size_t)g] + (size + 1) / 2;
    }
    const int64_t num_slots = group_slots[(size_t)num_groups];
    std::vector<VdosSlot> slots((size_t)num_slots);
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
    const int64_t points = rn_spectrum_num_points(plan->S);
    if (points == 0) return RN_OK;
    RN_CHECK_ARG(d_wavenumbers && d_intensities, "null output pointer");
    DeviceGuard guard(plan->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int64_t table_bytes = (int64_t)sizeof(VdosSlot) * num_slots;
    const int64_t need = table_bytes + (int64_t)sizeof(int64_t) * (num_groups + 1);
    if (need > plan->vdos_bytes) {  // kept with the plan; calls on one plan are ordered on one stream
        RN_CUDA(cudaStreamSynchronize(s));
        cudaFree(plan->d_vdos);
        plan->d_vdos = nullptr;
        plan->vdos_bytes = 0;
        if (cudaMalloc(&plan->d_vdos, (size_t)need) != cudaSuccess) {
            cudaGetLastError();
            set_error("cudaMalloc of %lld bytes of VDOS slot tables failed", (long long)need);
            return RN_ERR_OUT_OF_MEMORY;
        }
        plan->vdos_bytes = need;
    }
    char* table = static_cast<char*>(plan->d_vdos);
    // pageable sources: the copies return once the data is staged, so the vectors may go out of scope
    RN_CUDA(cudaMemcpyAsync(table, slots.data(), (size_t)table_bytes, cudaMemcpyHostToDevice, s));
    RN_CUDA(cudaMemcpyAsync(table + table_bytes, group_slots.data(), sizeof(int64_t) * (num_groups + 1),
                            cudaMemcpyHostToDevice, s));
    const VdosSlot* d_slots = reinterpret_cast<const VdosSlot*>(table);
    const int64_t* d_group_slots = reinterpret_cast<const int64_t*>(table + table_bytes);

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
        while (group_slots[(size_t)g_lo + 1] <= first) g_lo++;
        int64_t g_hi = g_lo;  // last group with a slot in the chunk
        while (group_slots[(size_t)g_hi + 1] < first + nb) g_hi++;
        pp.slots = d_slots + first;
        pack_velocity_kernel<<<dim3(plan->pack_blocks, (unsigned)nb), kPackThreads, 0, s>>>(pp);
        RN_LAUNCHED();
        fft::OutSpec out = plain_out();
        out.mode = fft::OUT_POWER;
        out.power = plan->d_power;
        out.M = M;
        int rc = run_convolution(plan, plan->d_work, (int)(3 * nb), M, out, nullptr, s);
        if (rc != RN_OK) return rc;
        const int64_t groups = g_hi - g_lo + 1;
        combine_groups_kernel<<<dim3(grid_for(points, plan->sm_count), (unsigned)std::min<int64_t>(groups, 65535)), 256,
                                0, s>>>(plan->d_power, plan->d_epart + plan->pack_blocks, plan->pack_blocks + 1,
                                        d_group_slots, first, nb, g_lo, groups, M, scale, points, timestep_fs,
                                        first == 0 ? d_wavenumbers : nullptr, d_intensities);
        RN_LAUNCHED();
        RN_CUDA(cudaGetLastError());
    }
    return RN_OK;
}

extern "C" int rn_signal_spectrum(rn_spectrum_plan* plan, const double* d_signal, double sampling_rate,
                                  double* d_wavenumbers, double* d_intensities, void* stream) {
    RN_CHECK_ARG(plan != nullptr, "plan is null");
    RN_CHECK_ARG(plan->world == 1, "rn_signal_spectrum needs a single-GPU plan");
    RN_CHECK_ARG(d_signal && d_wavenumbers && d_intensities, "null device pointer");
    RN_CHECK_ARG(sampling_rate > 0, "sampling_rate must be positive");
    DeviceGuard guard(plan->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int64_t M = plan->M;
    const int64_t points = (M + 1) / 2;
    PackParams pp;
    pp.src = d_signal;
    pp.M = M;
    pp.Lh = plan->Lh;
    pp.begin = 0;
    pp.end = M;
    for (int i = 0; i < 8; i++) pp.dst[i] = nullptr;
    pp.dst[0] = plan->d_work;
    pp.aligned16 = (reinterpret_cast<uintptr_t>(pp.src) % 16 == 0) ? 1 : 0;
    pp.seq_sel = -1;
    pp.num_share = 0;
    pp.share_slot = 0;
    pp.zero_slot = -1;
    pp.log2_stripe = -1;
    pp.phase = 0;
    for (int i = 0; i < 8; i++) pp.share[i] = nullptr;
    pp.epart = plan->d_epart;
    pp.ticket = plan->d_ticket;
    pp.tw = plan_twiddles(plan);
    pack_signal_kernel<<<plan->pack_blocks, kPackThreads, 0, s>>>(pp);
    RN_LAUNCHED();
    fft::OutSpec out = plain_out();
    out.mode = fft::OUT_POWER;
    out.power = plan->d_power;
    out.M = M;
    int rc = run_convolution(plan, plan->d_work, 1, M, out, nullptr, s);
    if (rc != RN_OK) return rc;
    const double scale = 0.5 / ((double)plan->L * (double)plan->L);
    combine_signal_kernel<<<grid_for(points, plan->sm_count), 256, 0, s>>>(plan->d_power, plan->d_epart + plan->pack_blocks, 1,
                                                                          M, scale, points, sampling_rate, d_wavenumbers,
                                                                          d_intensities);
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    return RN_OK;
}

// ---- one transform shared by the ranks of a process group -----------------------------------------

extern "C" int rn_spectrum_dist_sizes(const rn_spectrum_plan* plan, int64_t* work_bytes, int64_t* recv_bytes,
                                      int64_t* spectrum_bytes) {
    RN_CHECK_ARG(plan && work_bytes && recv_bytes && spectrum_bytes, "null pointer");
    *work_bytes = (int64_t)sizeof(double2) * 3 * plan->Lh;
    // 3 sequences x G residues x (Lh / G + 128) slots for the m' this rank owns (fft::mirror_owner)
    *recv_bytes = (int64_t)sizeof(double2) * 3 * (plan->Lh + 128 * plan->world);
    *spectrum_bytes = (int64_t)sizeof(double) * (kSpecHeader + rn_spectrum_num_points(plan->S));
    return RN_OK;
}

extern "C" int rn_spectrum_dist_route(const rn_spectrum_plan* plan, int64_t* period, int64_t* width) {
    RN_CHECK_ARG(plan && period && width, "null pointer");
    *period = plan->Lh;
    *width = plan->Lh / plan->world;
    return RN_OK;
}

template <int G>
static int launch_pack_dist(const rn_spectrum_plan* plan, const PackParams& pp, int blocks, cudaStream_t s) {
    pack_alpha_kernel<G><<<blocks, kPackThreads, 0, s>>>(pp);
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    (void)plan;
    return RN_OK;
}

// stripe of the pipelined schedule: half of the block of n' one rank packs (0: the block is too small)
static int64_t dist_stripe(const rn_spectrum_plan* plan) {
    const int64_t w = plan->Lh / plan->world;
    return (plan->world > 1 && w >= 4096) ? w / 2 : 0;
}

extern "C" int rn_spectrum_dist_stripe(const rn_spectrum_plan* plan, int64_t* stripe) {
    RN_CHECK_ARG(plan && stripe, "null pointer");
    *stripe = dist_stripe(plan);
    return RN_OK;
}

extern "C" int rn_spectrum_dist_pack(rn_spectrum_plan* plan, const double* d_series, double* const* peer_work,
                                     double* const* dest_spectrum, int num_dest, int seq, int phase, void* stream) {
    RN_CHECK_ARG(plan && d_series && peer_work && dest_spectrum, "null pointer");
    RN_CHECK_ARG(seq >= -1 && seq <= 2, "seq must be -1 (all) or 0..2");
    RN_CHECK_ARG(phase >= -1 && phase <= 1, "phase must be -1 (whole block), 0 or 1");
    RN_CHECK_ARG(phase < 0 || (seq < 0 && dist_stripe(plan) > 0), "a split pack handles all sequences of a large enough block");
    RN_CHECK_ARG(num_dest >= 1 && num_dest <= 8, "between 1 and 8 destinations");
    if (plan->rank >= plan->world) return RN_OK;  // spectator
    RN_CHECK_ARG(plan->world > 1, "rn_spectrum_dist_pack needs a plan from rn_spectrum_plan_create_dist with world > 1");
    DeviceGuard guard(plan->device);
    PackParams pp;
    pp.src = d_series;
    pp.M = plan->M;
    pp.Lh = plan->Lh;
    const int64_t w = plan->Lh / plan->world;
    pp.begin = (int64_t)plan->rank * w;
    pp.end = pp.begin + w;
    for (int i = 0; i < 8; i++) pp.dst[i] = nullptr;
    for (int r = 0; r < plan->world; r++) {
        RN_CHECK_ARG(peer_work[r] != nullptr, "null work buffer pointer for rank %d", r);
        pp.dst[r] = reinterpret_cast<double2*>(peer_work[r]);
    }
    pp.aligned16 = (reinterpret_cast<uintptr_t>(pp.src) % 16 == 0) ? 1 : 0;
    // the two phases of a split pack may run concurrently: each has its own partials and ticket
    const int second = phase == 1 ? 1 : 0;
    pp.epart = plan->d_epart + second * (plan->pack_blocks + 1);
    pp.ticket = plan->d_ticket + second;
    pp.tw = plan_twiddles(plan);
    pp.seq_sel = seq;
    for (int i = 0; i < 8; i++) pp.share[i] = nullptr;
    for (int d = 0; d < num_dest; d++) {
        RN_CHECK_ARG(dest_spectrum[d] != nullptr, "null spectrum buffer pointer %d", d);
        pp.share[d] = dest_spectrum[d];
    }
    pp.num_share = num_dest;
    pp.share_slot = plan->rank + 8 * second;
    pp.zero_slot = phase < 0 ? plan->rank + 8 : -1;
    pp.log2_stripe = -1;
    pp.phase = second;
    int blocks = plan->pack_blocks;
    if (phase >= 0) {
        const int64_t stripe = dist_stripe(plan);
        while (((int64_t)1 << (pp.log2_stripe + 1)) <= stripe) pp.log2_stripe++;
        blocks = (int)(stripe / kPackThreads);
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (plan->world == 2) return launch_pack_dist<2>(plan, pp, blocks, s);
    if (plan->world == 4) return launch_pack_dist<4>(plan, pp, blocks, s);
    return launch_pack_dist<8>(plan, pp, blocks, s);
}

extern "C" int rn_spectrum_dist_transform(rn_spectrum_plan* plan, double* d_work, double* const* peer_recv,
                                          int seq, void* stream) {
    RN_CHECK_ARG(plan && d_work && peer_recv, "null pointer");
    RN_CHECK_ARG(seq >= -1 && seq <= 2, "seq must be -1 (all) or 0..2");
    if (plan->rank >= plan->world) return RN_OK;
    RN_CHECK_ARG(plan->world > 1, "rn_spectrum_dist_transform needs a shared plan (world > 1)");
    DeviceGuard guard(plan->device);
    fft::OutSpec out = plain_out();
    out.mode = fft::OUT_PEERS;
    out.peers.world = plan->world;
    out.peers.rank = plan->rank;
    int log2w = plan->log2lh;
    for (int g = plan->world; g > 1; g >>= 1) log2w--;
    out.peers.log2w = log2w;
    out.peers.log2lh = plan->log2lh;
    out.peers.c = plan->M & (plan->Lh - 1);
    for (int r = 0; r < plan->world; r++) {
        RN_CHECK_ARG(peer_recv[r] != nullptr, "null receive buffer pointer for rank %d", r);
        out.peers.ptr[r] = reinterpret_cast<double2*>(peer_recv[r]);
    }
    double2* work = reinterpret_cast<double2*>(d_work);
    if (seq < 0) return run_convolution(plan, work, 3, plan->Lh, out, nullptr, static_cast<cudaStream_t>(stream));
    return run_convolution(plan, work + (int64_t)seq * plan->Lh, 1, plan->Lh, out, nullptr,
                           static_cast<cudaStream_t>(stream), seq);
}

template <int G>
static int launch_final_dist(const rn_spectrum_plan* plan, const FinalParams& fp, cudaStream_t s) {
    const int64_t pairs = ((int64_t)1 << (fp.log2w - 1)) + 1;
    final_dist_kernel<G><<<(unsigned)((pairs + 255) / 256), 256, 0, s>>>(fp);
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    (void)plan;
    return RN_OK;
}

extern "C" int rn_spectrum_dist_final(rn_spectrum_plan* plan, const double* d_recv, const double* d_spectrum,
                                      double* const* dest_spectrum, int num_dest, double timestep_fs,
                                      int laser_correction, double laser_wavelength_nm, int bose_einstein_correction,
                                      double temperature_K, double* d_wavenumbers, void* stream) {
    RN_CHECK_ARG(plan && dest_spectrum, "null pointer");
    RN_CHECK_ARG(timestep_fs > 0, "timestep must be positive");
    if (laser_correction) RN_CHECK_ARG(laser_wavelength_nm > 0, "invalid laser_wavelength");
    if (bose_einstein_correction) RN_CHECK_ARG(temperature_K > 0, "invalid temperature: %g <= 0", temperature_K);
    if (plan->rank >= plan->world) return RN_OK;
    RN_CHECK_ARG(plan->world > 1 && d_recv && d_spectrum,
                 "rn_spectrum_dist_final needs a shared plan, its receive buffer and its spectrum buffer");
    RN_CHECK_ARG(num_dest >= 1 && num_dest <= 8, "between 1 and 8 destinations");
    DeviceGuard guard(plan->device);
    FinalParams fp;
    fp.recv = reinterpret_cast<const double2*>(d_recv);
    fp.M = plan->M;
    fp.Lh = plan->Lh;
    fp.c = plan->M & (plan->Lh - 1);
    int log2w = plan->log2lh;
    for (int g = plan->world; g > 1; g >>= 1) log2w--;
    fp.log2w = log2w;
    fp.log2lh = plan->log2lh;
    fp.rank = plan->rank;
    for (int i = 0; i < 8; i++) fp.dest[i] = nullptr;
    for (int d = 0; d < num_dest; d++) {
        RN_CHECK_ARG(dest_spectrum[d] != nullptr, "null destination pointer %d", d);
        fp.dest[d] = dest_spectrum[d];
    }
    fp.num_dest = num_dest;
    fp.shares = d_spectrum;
    fp.points = rn_spectrum_num_points(plan->S);
    fp.scale = 0.25 / ((double)plan->L * (double)plan->L);
    fp.prm = spectrum_params(timestep_fs, laser_correction, laser_wavelength_nm, bose_einstein_correction,
                             temperature_K);
    fp.wn_out = d_wavenumbers;
    fp.tw = plan_twiddles(plan);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (plan->world == 2) return launch_final_dist<2>(plan, fp, s);
    if (plan->world == 4) return launch_final_dist<4>(plan, fp, s);
    return launch_final_dist<8>(plan, fp, s);
}

extern "C" int rn_spectrum_dist_finish(const rn_spectrum_plan* plan, const double* d_spectrum, double timestep_fs,
                                       double* d_wavenumbers, double* d_intensities, void* stream) {
    RN_CHECK_ARG(plan != nullptr && d_spectrum != nullptr, "null pointer");
    RN_CHECK_ARG(timestep_fs > 0, "timestep must be positive");
    const int64_t points = rn_spectrum_num_points(plan->S);
    if (points == 0) return RN_OK;
    RN_CHECK_ARG(d_intensities, "null output pointer");
    DeviceGuard guard(plan->device);
    int sms = plan->sm_count;
    if (sms <= 0) sms = 148;
    finish_dist_kernel<<<grid_for(points, sms), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        d_spectrum, points, plan->M, timestep_fs, d_wavenumbers, d_intensities);
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    return RN_OK;
}

// Test hooks (include/ramannoodle_b200_debug.h).
// forward transform of plan->Lh complex values, left in the transform's own (digit-reversed) order
extern "C" int rn_debug_fft_forward(rn_spectrum_plan* plan, const double* d_in, double* d_out, void* stream) {
    RN_CHECK_ARG(plan && d_in && d_out && plan->d_work, "null pointer");
    DeviceGuard guard(plan->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    RN_CUDA(cudaMemcpyAsync(plan->d_work, d_in, sizeof(double2) * plan->Lh, cudaMemcpyDeviceToDevice, s));
    return run_convolution(plan, plan->d_work, 1, plan->Lh, plain_out(), reinterpret_cast<double2*>(d_out), s);
}
// IFFT(FFT(in) * H) (unnormalised), H = the plan's chirp filter spectrum; natural order in and out
extern "C" int rn_debug_fft_convolve(rn_spectrum_plan* plan, const double* d_in, double* d_out, void* stream) {
    RN_CHECK_ARG(plan && d_in && d_out && plan->d_work, "null pointer");
    DeviceGuard guard(plan->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    RN_CUDA(cudaMemcpyAsync(plan->d_work, d_in, sizeof(double2) * plan->Lh, cudaMemcpyDeviceToDevice, s));
    int rc = run_convolution(plan, plan->d_work, 1, plan->Lh, plain_out(), nullptr, s);
    if (rc != RN_OK) return rc;
    RN_CUDA(cudaMemcpyAsync(d_out, plan->d_work, sizeof(double2) * plan->Lh, cudaMemcpyDeviceToDevice, s));
    return RN_OK;
}
