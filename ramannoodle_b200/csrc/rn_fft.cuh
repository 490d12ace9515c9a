// In-place power-of-two FFT convolution core of the spectrum path (sm_100a, fp64).
//
// The chirp-z (Bluestein) transform behind MDRamanSpectrum.measure / calc_signal_spectrum
// (ramannoodle/spectrum/_raman.py:241-309, spectrum/utils.py:76-124) is a cyclic convolution
//   y = IFFT_L( FFT_L(a) * H ),   L = 2^p.
// A convolution does not care in which order the frequency bins are stored, so the forward
// transform runs as an in-place decimation-in-frequency (DIF) FFT whose output is left in
// digit-reversed order, H is stored in that same order (it is produced by the same code), and
// the inverse runs as the exact mirror (decimation in time, DIT), again in place.  No transposes,
// no ping-pong buffer, and the last forward stages, the filter multiply and the first inverse
// stages of a 4096-element contiguous tile happen in ONE kernel:
//
//   level kernel (fwd)   strided radix-R DIF pass over the sub-arrays, R <= 1024 : 1 round trip
//   tile kernel          4096-point DIF, * H, 4096-point DIT                        : 1 round trip
//   level kernel (inv)   the mirror of the forward level pass                      : 1 round trip
//
// i.e. 3 memory round trips per sequence for L = 2^21 where a Stockham autosort FFT pair needs 6.
// Every CTA owns a 4096-element tile (64 KB of shared memory, 256 threads x 16 elements); stages
// are radix 8 (one radix-2/4 stage completes R when log2 R is not a multiple of 3).  In-place
// stages read and write the same shared-memory positions from the same thread, so one
// __syncthreads per stage suffices; an XOR swizzle of the 16-byte unit index keeps every stage's
// LDS.128/STS.128 pattern bank-conflict free.
#pragma once

#include "rn_common.cuh"

namespace rn {
namespace fft {

constexpr int kLog2E = 12;
constexpr int kE = 1 << kLog2E;  // complex elements per CTA tile
constexpr int kNT = 256;         // threads per CTA (16 elements each)
constexpr int kPerThread = kE / kNT;
constexpr size_t kTileSmemBytes = (size_t)kE * sizeof(double2);

enum { OUT_PLAIN = 0, OUT_POWER = 1, OUT_PEERS = 2 };

__device__ __forceinline__ double2 cmul(double2 a, double2 b) {
    return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
__device__ __forceinline__ double2 cadd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 csub(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ double2 conj(double2 a) { return make_double2(a.x, -a.y); }

// multiply by sgn*i
template <int SGN>
__device__ __forceinline__ double2 mul_i(double2 a) {
    return SGN > 0 ? make_double2(-a.y, a.x) : make_double2(a.y, -a.x);
}

// y[k] = sum_q x[q] exp(SGN 2 pi i q k / RADIX), natural order in and out
template <int RADIX, int SGN>
struct Dft;

template <int SGN>
struct Dft<2, SGN> {
    static __device__ __forceinline__ void run(double2* v) {
        const double2 a = v[0];
        v[0] = cadd(a, v[1]);
        v[1] = csub(a, v[1]);
    }
};

template <int SGN>
struct Dft<4, SGN> {
    static __device__ __forceinline__ void run(double2* v) {
        const double2 s02 = cadd(v[0], v[2]), d02 = csub(v[0], v[2]);
        const double2 s13 = cadd(v[1], v[3]), d13 = mul_i<SGN>(csub(v[1], v[3]));
        v[0] = cadd(s02, s13);
        v[1] = cadd(d02, d13);
        v[2] = csub(s02, s13);
        v[3] = csub(d02, d13);
    }
};

template <int SGN>
struct Dft<8, SGN> {
    static __device__ __forceinline__ void run(double2* v) {
        double2 e[4] = {v[0], v[2], v[4], v[6]};
        double2 o[4] = {v[1], v[3], v[5], v[7]};
        Dft<4, SGN>::run(e);
        Dft<4, SGN>::run(o);
        const double h = 0.70710678118654752440;
        // W8^1 = (1 + sgn i)/sqrt2, W8^2 = sgn i, W8^3 = (-1 + sgn i)/sqrt2
        const double2 o1 = make_double2(h * (o[1].x - SGN * o[1].y), h * (SGN * o[1].x + o[1].y));
        const double2 o2 = mul_i<SGN>(o[2]);
        const double2 o3 = make_double2(h * (-o[3].x - SGN * o[3].y), h * (SGN * o[3].x - o[3].y));
        v[0] = cadd(e[0], o[0]);
        v[4] = csub(e[0], o[0]);
        v[1] = cadd(e[1], o1);
        v[5] = csub(e[1], o1);
        v[2] = cadd(e[2], o2);
        v[6] = csub(e[2], o2);
        v[3] = cadd(e[3], o3);
        v[7] = csub(e[3], o3);
    }
};

template <int RADIX>
struct Log2;
template <>
struct Log2<2> {
    static constexpr int value = 1;
};
template <>
struct Log2<4> {
    static constexpr int value = 2;
};
template <>
struct Log2<8> {
    static constexpr int value = 3;
};

// x[q] *= w^q, q = 1 .. RADIX-1 (powers by squaring/products: depth <= 3 multiplications)
template <int RADIX>
__device__ __forceinline__ void apply_powers(double2* x, double2 w1) {
    x[1] = cmul(x[1], w1);
    if constexpr (RADIX >= 4) {
        const double2 w2 = cmul(w1, w1);
        const double2 w3 = cmul(w2, w1);
        x[2] = cmul(x[2], w2);
        x[3] = cmul(x[3], w3);
        if constexpr (RADIX == 8) {
            const double2 w4 = cmul(w2, w2);
            x[4] = cmul(x[4], w4);
            x[5] = cmul(x[5], cmul(w4, w1));
            x[6] = cmul(x[6], cmul(w3, w3));
            x[7] = cmul(x[7], cmul(w4, w3));
        }
    }
}

// x[q] *= base * step^q, q = 0 .. RADIX-1
template <int RADIX>
__device__ __forceinline__ void apply_base_step(double2* x, double2 base, double2 step) {
    double2 w = base;
#pragma unroll
    for (int q = 0; q < RADIX; q++) {
        x[q] = cmul(x[q], w);
        if (q + 1 < RADIX) w = cmul(w, step);
    }
}

// shared-memory position of tile element `pos` (16-byte units): XOR the low three bits with the
// next three.  Eight consecutive threads then always touch eight different 16-byte columns, whether
// their positions differ in the low bits (strides >= 8 elements) or in bits 3..5 (the last stages).
__device__ __forceinline__ int swz(int pos) { return pos ^ ((pos >> 3) & 7); }

// exact (80-bit host computed, rounded once) twiddle tables: W_L^m = hi[m >> split] * lo[m & mask],
// W_4096^m = sub[m];  W_n = exp(-2 pi i / n)
struct Twiddles {
    const double2* hi;
    const double2* lo;
    const double2* sub;
    int split;
};

__device__ __forceinline__ double2 tw_global(const Twiddles& T, uint32_t m) {
    return cmul(__ldg(T.hi + (m >> T.split)), __ldg(T.lo + (m & ((1u << T.split) - 1u))));
}

// Destination of the inverse transform's output when the transform is shared by G ranks.  The spectrum
// pairs bin m with bin M - m, whose residues m' = m mod Lh are mirror images, m'' = (c - m') mod Lh with
// c = M mod Lh; ownership of m' is therefore MIRROR-SYMMETRIC, so that one rank holds both members of
// every pair and finishes the pair's intensity by itself.  With u = (2 m' - c) mod 2 Lh and
// a = min(u, 2 Lh - u) (the doubled circular distance from c/2, the same for m' and its mirror image),
// the owner is min(a / w, G - 1), w = Lh / G.  The owner's slice (seq, source rank) has two halves of
// w/2 + 64 slots: residues on the side u <= Lh ascend from a 32-aligned origin, the mirror side descends
// from a top that is 31 (mod 32) — either way a run of 32 consecutive residues that starts at a multiple of
// 32 lands in one aligned 512-byte block of the peer's buffer (unaligned runs cost the NVLink stores of the
// last pass a third of their rate).
struct PeerOut {
    double2* ptr[8];
    int log2w;
    int log2lh;
    int rank;
    int world;
    int64_t c;  // M mod Lh
};

__host__ __device__ __forceinline__ int64_t mirror_half_slots(int log2w) { return ((int64_t)1 << (log2w - 1)) + 64; }

// origin of owner o's ascending half and top of its descending half (residues)
__device__ __forceinline__ void mirror_arcs(int o, int64_t c, int log2lh, int log2w, int64_t* near_origin,
                                            int64_t* far_top) {
    const int64_t lh = (int64_t)1 << log2lh;
    const int64_t a0 = ((int64_t)o << log2w) + (c & 1);  // smallest doubled distance this owner holds
    *near_origin = (((c + a0) >> 1) & (lh - 1)) & ~(int64_t)31;
    *far_top = (((2 * lh + c - a0) >> 1) & (lh - 1)) | 31;
}

// owner of residue m1 and its slot within one (seq, source rank) slice of 2 * mirror_half_slots() slots
__device__ __forceinline__ void mirror_owner(int64_t m1, int64_t c, int log2lh, int log2w, int world, int* owner,
                                             int64_t* slot) {
    const int64_t lh = (int64_t)1 << log2lh;
    int64_t u = 2 * m1 - c;
    if (u < 0) u += 2 * lh;
    const bool far_side = u > lh;
    const int64_t a = far_side ? 2 * lh - u : u;
    const int o = min((int)(a >> log2w), world - 1);
    int64_t near_origin, far_top;
    mirror_arcs(o, c, log2lh, log2w, &near_origin, &far_top);
    *owner = o;
    *slot = far_side ? mirror_half_slots(log2w) + ((far_top - m1) & (lh - 1)) : ((m1 - near_origin) & (lh - 1));
}

struct OutSpec {
    int mode;        // OUT_PLAIN / OUT_POWER / OUT_PEERS
    double* power;   // OUT_POWER: power[seq * M + m] = |y[m]|^2, m < M
    int64_t M;
    PeerOut peers;   // OUT_PEERS
};

__device__ __forceinline__ void store_out(const OutSpec& out, double2* plain, int seq, int64_t m, double2 v) {
    if (out.mode == OUT_PLAIN) {
        *plain = v;
    } else if (out.mode == OUT_POWER) {
        if (m < out.M) out.power[(int64_t)seq * out.M + m] = v.x * v.x + v.y * v.y;
    } else {
        int owner;
        int64_t slot;
        mirror_owner(m, out.peers.c, out.peers.log2lh, out.peers.log2w, out.peers.world, &owner, &slot);
        const int64_t stride = 2 * mirror_half_slots(out.peers.log2w);
        out.peers.ptr[owner][(int64_t)(seq * out.peers.world + out.peers.rank) * stride + slot] = v;
    }
}

// One in-place stage of the tile: butterflies over positions pos0 + q * sp (q < RADIX), sp = 2^log2sp.
// The tile is a [n][b] array (b < B = 2^log2b the batch of independent transforms, fastest); the stage
// splits blocks of Ns = RADIX * sp / B points.  SGN < 0: DIF forward (twiddle W_Ns^{i k} after the
// butterfly); SGN > 0: DIT inverse, the mirror (conjugate twiddle before the butterfly).
// rd(pos, slot) / wr(pos, slot, value) move elements; slot = m * RADIX + q numbers the thread's 16 elements.
template <int SGN, int RADIX, bool LEAN, class Rd, class Wr>
__device__ __forceinline__ void fft_stage(int log2sp, int log2b, const double2* __restrict__ wsub, Rd rd, Wr wr) {
    constexpr int NB = kPerThread / RADIX;
    constexpr int LR = Log2<RADIX>::value;
    const int sp = 1 << log2sp;
    const int log2ns = log2sp - log2b + LR;
    const bool has_tw = log2sp > log2b;
    // LEAN: one butterfly in flight per thread (fewer registers, three CTAs per SM); otherwise the
    // thread's butterflies are unrolled and interleaved (two CTAs per SM)
#pragma unroll(LEAN ? 1 : NB)
    for (int m = 0; m < NB; m++) {
        const int u = (int)threadIdx.x + m * kNT;
        const int lo = u & (sp - 1);
        const int pos0 = ((u >> log2sp) << (log2sp + LR)) + lo;
        double2 x[RADIX];
#pragma unroll
        for (int q = 0; q < RADIX; q++) x[q] = rd(pos0 + (q << log2sp), m * RADIX + q);
        double2 w1 = make_double2(1.0, 0.0);
        if (has_tw) {
            w1 = __ldg(wsub + ((lo >> log2b) << (kLog2E - log2ns)));
            if (SGN > 0) w1.y = -w1.y;
        }
        if (SGN > 0 && has_tw) apply_powers<RADIX>(x, w1);
        Dft<RADIX, SGN>::run(x);
        if (SGN < 0 && has_tw) apply_powers<RADIX>(x, w1);
#pragma unroll
        for (int q = 0; q < RADIX; q++) wr(pos0 + (q << log2sp), m * RADIX + q, x[q]);
    }
}

// ---- tile kernel: 4096-point DIF, filter multiply, 4096-point DIT on contiguous tiles -----------
struct TileParams {
    double2* X;            // (nseq, seq_stride) work buffer, transformed in place
    int64_t seq_stride;
    int tiles_per_seq;
    const double2* H;      // (seq_stride) filter spectrum in the transform's digit-reversed order
    double2* Hout;         // FWD_ONLY: forward transform written here (plan creation)
    int64_t limit;         // input elements with index >= limit (within the sequence) read as zero
    int seq_base;          // number of the first sequence in X (names the slot in OUT_POWER / OUT_PEERS)
    OutSpec out;
    Twiddles tw;
};

// AUTOCORR: the filter multiply becomes x[q] -> (|x[q]|^2, 0) and H is not read, so the pass computes
// L * IFFT(|FFT(z)|^2), the circular autocorrelation of z.  For z = a + i b with a, b real and Z = A + i B,
// |Z|^2 = |A|^2 + |B|^2 - 2 Im(B conj A); A and B are Hermitian, so Im(B[k] conj A[k]) is odd in k and its
// inverse transform is purely imaginary.  With plain output, Re(y[m]) / L is therefore the autocorrelation of
// a plus that of b at lag m, linear for m < L - (length of z) when z is zero-padded.
template <bool FWD_ONLY, bool LEAN, bool AUTOCORR = false>
__global__ void __launch_bounds__(kNT, LEAN ? 3 : 2) tile_kernel(const __grid_constant__ TileParams P) {
    extern __shared__ __align__(16) unsigned char fft_smem[];
    double2* S = reinterpret_cast<double2*>(fft_smem);
    const int seq = blockIdx.x / P.tiles_per_seq;
    const int tile = blockIdx.x - seq * P.tiles_per_seq;
    const int64_t tile_base = (int64_t)tile * kE;
    double2* base = P.X + (int64_t)seq * P.seq_stride + tile_base;
    const double2* wsub = P.tw.sub;

    auto rd_s = [&](int pos, int) { return S[swz(pos)]; };
    auto wr_s = [&](int pos, int, double2 v) { S[swz(pos)] = v; };
    auto rd_g = [&](int pos, int) {
        return (tile_base + pos < P.limit) ? base[pos] : make_double2(0.0, 0.0);
    };

    fft_stage<-1, 8, LEAN>(9, 0, wsub, rd_g, wr_s);
    __syncthreads();
    fft_stage<-1, 8, LEAN>(6, 0, wsub, rd_s, wr_s);
    __syncthreads();
    fft_stage<-1, 8, LEAN>(3, 0, wsub, rd_s, wr_s);
    __syncthreads();
    // last forward stage, filter multiply and first inverse stage on the same eight registers
#pragma unroll(LEAN ? 1 : kPerThread / 8)
    for (int m = 0; m < kPerThread / 8; m++) {
        const int pos0 = ((int)threadIdx.x + m * kNT) << 3;
        double2 h[8];
        // the filter spectrum of a tile is stored [q][u] (element pos0 + q of butterfly u at q * 512 + u):
        // consecutive threads read consecutive addresses
        const int hu = (int)threadIdx.x + m * kNT;
        if (!FWD_ONLY && !AUTOCORR) {
#pragma unroll
            for (int q = 0; q < 8; q++) h[q] = __ldg(P.H + tile_base + (q << 9) + hu);
        }
        double2 x[8];
#pragma unroll
        for (int q = 0; q < 8; q++) x[q] = S[swz(pos0 + q)];
        Dft<8, -1>::run(x);
        if (FWD_ONLY) {
#pragma unroll
            for (int q = 0; q < 8; q++) P.Hout[tile_base + (q << 9) + hu] = x[q];
        } else {
#pragma unroll
            for (int q = 0; q < 8; q++)
                x[q] = AUTOCORR ? make_double2(x[q].x * x[q].x + x[q].y * x[q].y, 0.0) : cmul(x[q], h[q]);
            Dft<8, +1>::run(x);
#pragma unroll
            for (int q = 0; q < 8; q++) S[swz(pos0 + q)] = x[q];
        }
    }
    if (FWD_ONLY) return;
    __syncthreads();
    fft_stage<+1, 8, LEAN>(3, 0, wsub, rd_s, wr_s);
    __syncthreads();
    fft_stage<+1, 8, LEAN>(6, 0, wsub, rd_s, wr_s);
    __syncthreads();
    auto wr_g = [&](int pos, int, double2 v) { store_out(P.out, base + pos, P.seq_base + seq, tile_base + pos, v); };
    fft_stage<+1, 8, LEAN>(9, 0, wsub, rd_s, wr_g);
}

// ---- level kernel: strided radix-R pass (R = 2^log2r <= 1024) over sub-arrays of length Lsub ------
// Tile = R rows x B columns (B = 4096 / R consecutive elements, 16 B each): element (row, col) of tile
// `chunk` of sub-array `sub` lives at  X[seq][sub * Lsub + row * s + chunk * B + col],  s = Lsub / R.
// Forward (DIF): u[k] = DFT_R over rows, stored in place at the row whose radix-8 digits are those of
// k reversed, times W_Lsub^{k j} (j = chunk * B + col).  Inverse (DIT): the mirror.
// Stage schedule: radix-8 stages, then one radix-2^(log2r % 3) stage if log2r is not a multiple of 3.
struct LevelParams {
    double2* X;
    int64_t seq_stride;
    int log2lsub;
    int log2r;
    int nsub;
    int tw_shift;     // W_Lsub^e = W_L^(e << tw_shift)
    int64_t limit;    // forward: input elements with index >= limit (within the sequence) read as zero
    int seq_base;     // number of the first sequence in X (names the slot in OUT_POWER / OUT_PEERS)
    OutSpec out;      // inverse: where the result goes
    Twiddles tw;
};

// reverse the order of the `groups` 3-bit digits of x
__device__ __forceinline__ int rev3(int x, int groups) {
    int r = 0;
    for (int i = 0; i < groups; i++) {
        r = (r << 3) | (x & 7);
        x >>= 3;
    }
    return r;
}

template <int SGN>
struct LevelCtx {
    const LevelParams& P;
    double2* S;
    double2* base;      // element (row, col) at base[row * s + col]
    int64_t elem_base;  // index of (row 0, col 0) within the sequence
    int seq;
    int log2b, log2s;
    int a8;             // radix-8 stages
    int j0;             // chunk * B
};

// the stage that touches global memory with the level twiddle: forward = last stage (smem or global in,
// global out), inverse = first stage (global in, smem or global out).  RADIX-point butterflies over rows
// rowbase + q at column col; k = krest + q * (R / RADIX).
template <int SGN, int RADIX, bool SMEM_SIDE, bool LEAN>
__device__ __forceinline__ void level_twiddle_stage(const LevelCtx<SGN>& C) {
    constexpr int NB = kPerThread / RADIX;
    constexpr int LR = Log2<RADIX>::value;
    const LevelParams& P = C.P;
    const int B = 1 << C.log2b;
    const int groups = (P.log2r - LR) / 3;  // radix-8 digits above this stage's digit
#pragma unroll(LEAN ? 1 : (RADIX == 8 ? NB : 2))
    for (int m = 0; m < NB; m++) {
        const int u = (int)threadIdx.x + m * kNT;
        const int col = u & (B - 1);
        const int rb = u >> C.log2b;
        const int pos0 = (rb << (C.log2b + LR)) + col;  // (rowbase = rb * RADIX, col)
        const uint32_t j = (uint32_t)(C.j0 + col);
        const uint32_t krest = (uint32_t)rev3(rb, groups);
        double2 wb = tw_global(P.tw, (krest * j) << P.tw_shift);
        double2 ws = tw_global(P.tw, (j << (P.log2r - LR)) << P.tw_shift);
        if (SGN > 0) {
            wb.y = -wb.y;
            ws.y = -ws.y;
        }
        double2 x[RADIX];
        if (SGN < 0) {
#pragma unroll
            for (int q = 0; q < RADIX; q++) {
                const int pos = pos0 + (q << C.log2b);
                if (SMEM_SIDE) {
                    x[q] = C.S[swz(pos)];
                } else {
                    const int64_t off = ((int64_t)(pos >> C.log2b) << C.log2s) + (pos & (B - 1));
                    x[q] = (C.elem_base + off < P.limit) ? C.base[off] : make_double2(0.0, 0.0);
                }
            }
            Dft<RADIX, SGN>::run(x);
            apply_base_step<RADIX>(x, wb, ws);
#pragma unroll
            for (int q = 0; q < RADIX; q++) {
                const int pos = pos0 + (q << C.log2b);
                C.base[((int64_t)(pos >> C.log2b) << C.log2s) + (pos & (B - 1))] = x[q];
            }
        } else {
#pragma unroll
            for (int q = 0; q < RADIX; q++) {
                const int pos = pos0 + (q << C.log2b);
                x[q] = C.base[((int64_t)(pos >> C.log2b) << C.log2s) + (pos & (B - 1))];
            }
            apply_base_step<RADIX>(x, wb, ws);
            Dft<RADIX, SGN>::run(x);
#pragma unroll
            for (int q = 0; q < RADIX; q++) {
                const int pos = pos0 + (q << C.log2b);
                if (SMEM_SIDE) {
                    C.S[swz(pos)] = x[q];
                } else {
                    const int64_t off = ((int64_t)(pos >> C.log2b) << C.log2s) + (pos & (B - 1));
                    store_out(P.out, C.base + off, C.seq, C.elem_base + off, x[q]);
                }
            }
        }
    }
}

template <int SGN, bool LEAN>
__global__ void __launch_bounds__(kNT, LEAN ? 3 : 2) level_kernel(const __grid_constant__ LevelParams P) {
    extern __shared__ __align__(16) unsigned char fft_smem[];
    double2* S = reinterpret_cast<double2*>(fft_smem);
    const int log2b = kLog2E - P.log2r;
    const int log2s = P.log2lsub - P.log2r;
    const int log2chunks = log2s - log2b;
    const int chunk = blockIdx.x & ((1 << log2chunks) - 1);
    const int rest = blockIdx.x >> log2chunks;
    const int sub = rest % P.nsub;
    const int seq = rest / P.nsub;
    const int64_t elem_base = ((int64_t)sub << P.log2lsub) + ((int64_t)chunk << log2b);
    double2* base = P.X + (int64_t)seq * P.seq_stride + elem_base;
    const double2* wsub = P.tw.sub;
    const int a8 = P.log2r / 3, r1 = P.log2r % 3;
    const int B = 1 << log2b;
    LevelCtx<SGN> C{P, S, base, elem_base, P.seq_base + seq, log2b, log2s, a8, chunk << log2b};

    auto rd_s = [&](int pos, int) { return S[swz(pos)]; };
    auto wr_s = [&](int pos, int, double2 v) { S[swz(pos)] = v; };
    auto goff = [&](int pos) { return ((int64_t)(pos >> log2b) << log2s) + (pos & (B - 1)); };

    if (a8 + (r1 ? 1 : 0) == 1) {  // a single stage: global -> global
        if (r1 == 1) level_twiddle_stage<SGN, 2, false, LEAN>(C);
        else if (r1 == 2) level_twiddle_stage<SGN, 4, false, LEAN>(C);
        else level_twiddle_stage<SGN, 8, false, LEAN>(C);
        return;
    }
    if constexpr (SGN < 0) {
        // first stage: radix 8 straight from global memory
        auto rd_g = [&](int pos, int) {
            const int64_t off = goff(pos);
            return (elem_base + off < P.limit) ? base[off] : make_double2(0.0, 0.0);
        };
        int log2sp = kLog2E - 3;
        fft_stage<-1, 8, LEAN>(log2sp, log2b, wsub, rd_g, wr_s);
        __syncthreads();
        const int mid = (r1 ? a8 : a8 - 1) - 1;  // radix-8 stages strictly between the first and the last
        for (int i = 0; i < mid; i++) {
            log2sp -= 3;
            fft_stage<-1, 8, LEAN>(log2sp, log2b, wsub, rd_s, wr_s);
            __syncthreads();
        }
        if (r1 == 1) level_twiddle_stage<-1, 2, true, LEAN>(C);
        else if (r1 == 2) level_twiddle_stage<-1, 4, true, LEAN>(C);
        else level_twiddle_stage<-1, 8, true, LEAN>(C);
    } else {
        if (r1 == 1) level_twiddle_stage<+1, 2, true, LEAN>(C);
        else if (r1 == 2) level_twiddle_stage<+1, 4, true, LEAN>(C);
        else level_twiddle_stage<+1, 8, true, LEAN>(C);
        __syncthreads();
        const int mid = (r1 ? a8 : a8 - 1) - 1;
        int log2sp = kLog2E - 3 * (mid + 1);
        for (int i = 0; i < mid; i++) {
            fft_stage<+1, 8, LEAN>(log2sp, log2b, wsub, rd_s, wr_s);
            __syncthreads();
            log2sp += 3;
        }
        auto wr_g = [&](int pos, int, double2 v) {
            const int64_t off = goff(pos);
            store_out(P.out, base + off, P.seq_base + seq, elem_base + off, v);
        };
        fft_stage<+1, 8, LEAN>(kLog2E - 3, log2b, wsub, rd_s, wr_g);
    }
}

}  // namespace fft
}  // namespace rn
