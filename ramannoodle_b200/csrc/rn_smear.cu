// Spectrum smearing (convolve_spectrum, ramannoodle/spectrum/utils.py:12-73).
//
// out[l] = sum_i I_i f(wn_i - o_l), f = gaussian (1/w)(1/sqrt(2 pi)) exp(-x^2/(2 w^2)) or
// lorentzian (1/pi) (w/2) / (x^2 + (w/2)^2).  The reference loops over the K inputs in Python
// (O(K L) numpy work).  Here the (input chunk) x (output tile) grid is evaluated in
// parallel; each CTA first reduces the min/max of its input chunk and output tile and skips
// the pair when every Gaussian factor would underflow to exactly 0 in fp64 (|x| > 39 w:
// exp(-760.5) == 0), which is bit-identical to evaluating it.  Partial sums per input chunk
// are combined in a fixed order (deterministic).
//
// convolve_spectra smears B rows that share the input and output grids: smear_rows_partial_kernel
// evaluates each factor f(wn_i - o_l) once and applies it to a group of kRows rows (see there).
#include <cfloat>

#include "rn_common.cuh"

namespace rn {

constexpr int kOutTile = 256;    // outputs per CTA (one per thread)
constexpr int kInChunk = 2048;   // inputs per CTA
constexpr int kRows = 8;         // rows per CTA of the batched kernel (one factor, kRows accumulators)
constexpr int kRowSub = 256;     // inputs of a row group staged in shared memory at a time

__device__ __forceinline__ double block_reduce_minmax(double v, bool is_max, double* sm) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const double o = __shfl_xor_sync(0xffffffffu, v, off);
        v = is_max ? fmax(v, o) : fmin(v, o);
    }
    if (lane == 0) sm[warp] = v;
    __syncthreads();
    double r = sm[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); w++) r = is_max ? fmax(r, sm[w]) : fmin(r, sm[w]);
    __syncthreads();
    return r;
}

template <int KIND>
__global__ void __launch_bounds__(kOutTile) smear_partial_kernel(const double* __restrict__ wn,
                                                                 const double* __restrict__ inten, int64_t K,
                                                                 const double* __restrict__ out_wn, int64_t L,
                                                                 double width, double* __restrict__ partial) {
    __shared__ double s_wn[kInChunk];
    __shared__ double s_in[kInChunk];
    __shared__ double s_red[kOutTile / 32];
    const int64_t l = (int64_t)blockIdx.x * kOutTile + threadIdx.x;
    const int64_t i0 = (int64_t)blockIdx.y * kInChunk;
    const int n_in = (int)min((int64_t)kInChunk, K - i0);
    double lo_in = DBL_MAX, hi_in = -DBL_MAX;
    bool finite = true;
    for (int i = threadIdx.x; i < n_in; i += kOutTile) {
        const double w = wn[i0 + i];
        s_wn[i] = w;
        s_in[i] = inten[i0 + i];
        lo_in = fmin(lo_in, w);
        hi_in = fmax(hi_in, w);
        finite = finite && (w - w == 0.0) && (s_in[i] - s_in[i] == 0.0);
    }
    const double o = (l < L) ? out_wn[l] : 0.0;
    double acc = 0.0;
    bool skip = false;
    if (KIND == 0) {
        // the pair can be skipped only if every factor underflows to +0 and nothing is NaN/Inf
        const double lo_o = block_reduce_minmax((l < L) ? o : DBL_MAX, false, s_red);
        const double hi_o = block_reduce_minmax((l < L) ? o : -DBL_MAX, true, s_red);
        lo_in = block_reduce_minmax(lo_in, false, s_red);
        hi_in = block_reduce_minmax(hi_in, true, s_red);
        const int all_finite = __syncthreads_and(finite && (o - o == 0.0));
        const double cut = 39.0 * width;
        skip = all_finite && (lo_in - hi_o > cut || lo_o - hi_in > cut);
    } else {
        __syncthreads();
    }
    if (!skip && l < L) {
        if (KIND == 0) {
            const double norm = (1 / width) * (1 / sqrt(2 * 3.141592653589793));
            const double denom = 2 * (width * width);
            for (int i = 0; i < n_in; i++) {
                const double dx = s_wn[i] - o;
                acc += (norm * exp(-(dx * dx) / denom)) * s_in[i];
            }
        } else {
            const double hw = 0.5 * width;
            const double hw2 = hw * hw;
            const double inv_pi = 1 / 3.141592653589793;
            for (int i = 0; i < n_in; i++) {
                const double dx = s_wn[i] - o;
                acc += (inv_pi * (hw / (dx * dx + hw2))) * s_in[i];
            }
        }
    }
    if (l < L) partial[(int64_t)blockIdx.y * L + l] = acc;
}

// convolve_spectrum of B rows on one grid.  A CTA owns the (input chunk, output tile) pair of the
// single-row kernel and groups of kRows rows (blockIdx.z, looped past gridDim.z).  Thread l evaluates
// f(wn_i - o_l) once per i, with the single-row kernel's expression, and adds f * I[r][i] to the
// accumulator of every row r of the group in the same i order, so that each row's partial is that of
// smear_partial_kernel on the row bit for bit.  The chunk's wavenumbers are staged once; the group's
// intensities stream through shared memory kRowSub inputs at a time (all of the chunk would be
// kRows x 16 KB), stored [i][r] so that a thread reads the kRows values of one i with 16-byte broadcast loads.
// The Gaussian skip is the single-row predicate with the finiteness taken over every row of the group:
// a row with a NaN or Inf turns skipping off for its group, and for the other rows the evaluated factors
// underflow to +0 and add +0 to an accumulator that is never -0, so they are unchanged.  A skipped CTA
// still writes its zero partials, so the reduce sums every chunk in order exactly as for one row.
// partial is (chunks, B, L): row b of chunk c at (c*B + b)*L, so smear_reduce_kernel over B*L columns
// gives the (B, L) output.  Rows past B in the last group are neither read nor stored.
template <int KIND>
__global__ void __launch_bounds__(kOutTile) smear_rows_partial_kernel(const double* __restrict__ wn,
                                                                      const double* __restrict__ inten,
                                                                      int64_t B, int64_t K,
                                                                      const double* __restrict__ out_wn, int64_t L,
                                                                      double width, double* __restrict__ partial) {
    __shared__ double s_wn[kInChunk];
    __shared__ __align__(16) double s_in[kRowSub][kRows];
    __shared__ double s_red[kOutTile / 32];
    const int64_t l = (int64_t)blockIdx.x * kOutTile + threadIdx.x;
    const int64_t i0 = (int64_t)blockIdx.y * kInChunk;
    const int n_in = (int)min((int64_t)kInChunk, K - i0);
    double lo_in = DBL_MAX, hi_in = -DBL_MAX;
    bool finite = true;
    for (int i = threadIdx.x; i < n_in; i += kOutTile) {
        const double w = wn[i0 + i];
        s_wn[i] = w;
        lo_in = fmin(lo_in, w);
        hi_in = fmax(hi_in, w);
        finite = finite && (w - w == 0.0);
    }
    const double o = (l < L) ? out_wn[l] : 0.0;
    bool far = false;  // every factor of the pair underflows to +0 (Gaussian only)
    if (KIND == 0) {
        const double lo_o = block_reduce_minmax((l < L) ? o : DBL_MAX, false, s_red);
        const double hi_o = block_reduce_minmax((l < L) ? o : -DBL_MAX, true, s_red);
        lo_in = block_reduce_minmax(lo_in, false, s_red);
        hi_in = block_reduce_minmax(hi_in, true, s_red);
        const int all_finite = __syncthreads_and(finite && (o - o == 0.0));
        const double cut = 39.0 * width;
        far = all_finite && (lo_in - hi_o > cut || lo_o - hi_in > cut);
    } else {
        __syncthreads();
    }
    const int64_t groups = (B + kRows - 1) / kRows;
    for (int64_t g = blockIdx.z; g < groups; g += gridDim.z) {
        const int64_t r0 = g * kRows;
        const int nr = (int)min((int64_t)kRows, B - r0);
        const double* rows = inten + r0 * K + i0;
        bool skip = false;
        if (KIND == 0 && far) {
            bool rows_finite = true;
            for (int j = threadIdx.x; j < nr * n_in; j += kOutTile) {
                const double v = rows[(int64_t)(j / n_in) * K + j % n_in];
                rows_finite = rows_finite && (v - v == 0.0);
            }
            skip = __syncthreads_and(rows_finite);
        }
        double acc[kRows];
#pragma unroll
        for (int r = 0; r < kRows; r++) acc[r] = 0.0;
        if (!skip) {
            for (int s0 = 0; s0 < n_in; s0 += kRowSub) {
                const int ns = min(kRowSub, n_in - s0);
                __syncthreads();  // the previous sub-tile (or group) has been read
                for (int j = threadIdx.x; j < kRows * kRowSub; j += kOutTile) {
                    const int r = j / kRowSub, i = j % kRowSub;
                    s_in[i][r] = (r < nr && i < ns) ? rows[(int64_t)r * K + s0 + i] : 0.0;
                }
                __syncthreads();
                if (l < L) {
                    if (KIND == 0) {
                        const double norm = (1 / width) * (1 / sqrt(2 * 3.141592653589793));
                        const double denom = 2 * (width * width);
                        for (int i = 0; i < ns; i++) {
                            const double dx = s_wn[s0 + i] - o;
                            const double f = norm * exp(-(dx * dx) / denom);
#pragma unroll
                            for (int r = 0; r < kRows; r++) acc[r] += f * s_in[i][r];
                        }
                    } else {
                        const double hw = 0.5 * width;
                        const double hw2 = hw * hw;
                        const double inv_pi = 1 / 3.141592653589793;
                        for (int i = 0; i < ns; i++) {
                            const double dx = s_wn[s0 + i] - o;
                            const double f = inv_pi * (hw / (dx * dx + hw2));
#pragma unroll
                            for (int r = 0; r < kRows; r++) acc[r] += f * s_in[i][r];
                        }
                    }
                }
            }
        }
        if (l < L) {
#pragma unroll
            for (int r = 0; r < kRows; r++)
                if (r < nr) partial[((int64_t)blockIdx.y * B + r0 + r) * L + l] = acc[r];
        }
    }
}

__global__ void smear_reduce_kernel(const double* __restrict__ partial, int64_t chunks, int64_t L,
                                    double* __restrict__ out) {
    for (int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; l < L; l += (int64_t)gridDim.x * blockDim.x) {
        double v = 0.0;
        for (int64_t c = 0; c < chunks; c++) v += partial[c * L + l];
        out[l] = v;
    }
}

}  // namespace rn

using namespace rn;

extern "C" size_t rn_convolve_workspace_size(int64_t num_in, int64_t num_out) {
    if (num_in <= 0 || num_out <= 0) return 0;
    const int64_t chunks = (num_in + kInChunk - 1) / kInChunk;
    return (size_t)chunks * (size_t)num_out * sizeof(double);
}

extern "C" int rn_convolve_spectrum(const double* d_wavenumbers, const double* d_intensities, int64_t num_in, int kind,
                                    double width, const double* d_out_wavenumbers, int64_t num_out,
                                    double* d_out_intensities, void* d_workspace, void* stream) {
    RN_CHECK_ARG(kind == 0 || kind == 1, "unsupported convolution type: %d", kind);
    RN_CHECK_ARG(width > 0, "invalid width: %g <= 0", width);
    RN_CHECK_ARG(num_in >= 0 && num_out >= 0, "negative size");
    if (num_out == 0) return RN_OK;
    RN_CHECK_ARG(d_out_wavenumbers && d_out_intensities, "null output pointer");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (num_in == 0) {
        RN_CUDA(cudaMemsetAsync(d_out_intensities, 0, sizeof(double) * num_out, s));
        return RN_OK;
    }
    RN_CHECK_ARG(d_wavenumbers && d_intensities && d_workspace, "null device pointer");
    const int64_t chunks = (num_in + kInChunk - 1) / kInChunk;
    RN_CHECK_ARG(chunks <= 65535, "too many input points for one call (%lld)", (long long)num_in);
    dim3 grid((unsigned)((num_out + kOutTile - 1) / kOutTile), (unsigned)chunks);
    double* partial = static_cast<double*>(d_workspace);
    if (kind == 0)
        smear_partial_kernel<0><<<grid, kOutTile, 0, s>>>(d_wavenumbers, d_intensities, num_in, d_out_wavenumbers,
                                                          num_out, width, partial);
    else
        smear_partial_kernel<1><<<grid, kOutTile, 0, s>>>(d_wavenumbers, d_intensities, num_in, d_out_wavenumbers,
                                                          num_out, width, partial);
    RN_LAUNCHED();
    const int rgrid = (int)std::min<int64_t>((num_out + 255) / 256, 148 * 8);
    smear_reduce_kernel<<<rgrid, 256, 0, s>>>(partial, chunks, num_out, d_out_intensities);
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    return RN_OK;
}

extern "C" size_t rn_convolve_spectra_workspace_size(int64_t num_rows, int64_t num_in, int64_t num_out) {
    if (num_rows <= 0) return 0;
    return (size_t)num_rows * rn_convolve_workspace_size(num_in, num_out);
}

extern "C" int rn_convolve_spectra(const double* d_wavenumbers, const double* d_intensities, int64_t num_rows,
                                   int64_t num_in, int kind, double width, const double* d_out_wavenumbers,
                                   int64_t num_out, double* d_out_intensities, void* d_workspace, void* stream) {
    RN_CHECK_ARG(kind == 0 || kind == 1, "unsupported convolution type: %d", kind);
    RN_CHECK_ARG(width > 0, "invalid width: %g <= 0", width);
    RN_CHECK_ARG(num_in >= 0 && num_out >= 0, "negative size");
    RN_CHECK_ARG(num_rows >= 0, "negative number of rows: %lld", (long long)num_rows);
    if (num_rows == 0 || num_out == 0) return RN_OK;
    if (num_rows == 1)  // one row: the single-row kernels, which carry no padded rows of a group
        return rn_convolve_spectrum(d_wavenumbers, d_intensities, num_in, kind, width, d_out_wavenumbers, num_out,
                                    d_out_intensities, d_workspace, stream);
    RN_CHECK_ARG(d_out_wavenumbers && d_out_intensities, "null output pointer");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (num_in == 0) {
        RN_CUDA(cudaMemsetAsync(d_out_intensities, 0, sizeof(double) * num_rows * num_out, s));
        return RN_OK;
    }
    RN_CHECK_ARG(d_wavenumbers && d_intensities && d_workspace, "null device pointer");
    const int64_t chunks = (num_in + kInChunk - 1) / kInChunk;
    RN_CHECK_ARG(chunks <= 65535, "too many input points for one call (%lld)", (long long)num_in);
    const int64_t groups = (num_rows + kRows - 1) / kRows;
    dim3 grid((unsigned)((num_out + kOutTile - 1) / kOutTile), (unsigned)chunks,
              (unsigned)std::min<int64_t>(groups, 65535));
    double* partial = static_cast<double*>(d_workspace);
    if (kind == 0)
        smear_rows_partial_kernel<0><<<grid, kOutTile, 0, s>>>(d_wavenumbers, d_intensities, num_rows, num_in,
                                                               d_out_wavenumbers, num_out, width, partial);
    else
        smear_rows_partial_kernel<1><<<grid, kOutTile, 0, s>>>(d_wavenumbers, d_intensities, num_rows, num_in,
                                                               d_out_wavenumbers, num_out, width, partial);
    RN_LAUNCHED();
    const int64_t columns = num_rows * num_out;  // (chunks, B, L) partials reduce like one row of B*L outputs
    const int rgrid = (int)std::min<int64_t>((columns + 255) / 256, 148 * 8);
    smear_reduce_kernel<<<rgrid, 256, 0, s>>>(partial, chunks, columns, d_out_intensities);
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    return RN_OK;
}
