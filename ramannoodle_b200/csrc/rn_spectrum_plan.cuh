// The spectrum plan as the trajectory analyses (rn_trajectory.cu) see it: the plan's state, the device helpers
// of its packs and combines, and the host helpers that run its transform (defined in rn_spectrum.cu).
#pragma once

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
    // per-call scratch of the entries that need more than the buffers above (cross-energy partials, slot tables,
    // projection matrix); one call uses it at a time, so it holds the largest request (plan_scratch)
    void* d_scratch = nullptr;
    int64_t scratch_bytes = 0;
};

namespace rn {

constexpr int kPackThreads = 256;

// exp(-i*pi*n^2/M) (forward chirp); n^2 mod 2M is formed exactly in 64-bit integers
__device__ __forceinline__ double2 chirp(int64_t n, int64_t M) {
    const uint64_t m = ((uint64_t)n * (uint64_t)n) % (uint64_t)(2 * M);
    double s, c;
    sincospi((double)m / (double)M, &s, &c);
    return make_double2(c, -s);
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
    fft::Twiddles tw;
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

// wavenumbers: scipy.fftpack.fftfreq(M, dt)[k] * 33.35640951981521 * 1e3 with fftfreq = k * (1/(M*dt))
__device__ __forceinline__ double wavenumber_of(int64_t k, int64_t M, double dt) {
    const double val = 1.0 / ((double)M * dt);
    return ((double)k * val) * 33.35640951981521 * 1e3;
}

// the wavenumbers of bins 1 .. points into wn_out, strided over the blocks along x
__device__ __forceinline__ void write_wavenumbers(double* wn_out, int64_t points, int64_t M, double dt) {
    for (int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; o < points; o += (int64_t)gridDim.x * blockDim.x)
        wn_out[o] = wavenumber_of(o + 1, M, dt);
}

// ---- host helpers (rn_spectrum.cu) -------------------------------------------------------------------
int grid_for(int64_t n, int sms);

// the inverse transform's result left in the work buffer
fft::OutSpec plain_out();

// the inverse transform's |y_p[m]|^2 into the plan's power buffer
fft::OutSpec power_out(const rn_spectrum_plan* plan);

// forward levels, tile pass (with the filter), inverse levels: X (nseq, Lh) in place.  `limit`: input
// elements at or beyond it are zero (never read); `out`: where the inverse transform's result goes.
// hout != nullptr: forward transform only, written to hout (plan creation: the filter spectrum).
// autocorr: |X|^2 in place of the filter multiply (tile_kernel's AUTOCORR), the circular autocorrelation of X.
int run_convolution(const rn_spectrum_plan* p, double2* X, int nseq, int64_t limit, const fft::OutSpec& out,
                    double2* hout, cudaStream_t stream, int seq_base = 0, bool autocorr = false);

// *out = the plan's scratch buffer, grown to at least `bytes` (`what` names the contents in the error message).
// Growing waits for the stream first: calls on one plan are ordered on one stream.
int plan_scratch(rn_spectrum_plan* plan, int64_t bytes, cudaStream_t stream, const char* what, void** out);

}  // namespace rn
