// Self part of the Van Hove correlation G_s(r, t) and the displacement moments of atom groups
// (Trajectory.get_van_hove).
//
// Every membership (atom i of group g) is unwrapped with the minimum-image steps and exact integer image shifts of
// get_vdos / get_msd, then the displacements |r_i(n+t) - r_i(n)| of every origin n < S - t are binned, for each
// requested lag t, into integer histograms, and their squares and fourth powers are summed.  The arithmetic follows
// tests/van_hove_oracle.py operation for operation, with explicitly rounded intrinsics so that no multiply-add is
// fused:
//   k_j = ceil((x(j+1) - x(j)) - 0.5);  K(n) = sum_{j<n} k_j  (exact integers, any order)
//   w = (x(n) - x(0)) - K(n);  r_c = (w0 L[0,c] + w1 L[1,c]) + w2 L[2,c]
//   D_c = r_c(n+t) - r_c(n);  rr = (D0 D0 + D1 D1) + D2 D2;  k = floor(sqrt(rr) * (B / r_max)), counted when k < B
// so every count equals the oracle's exactly, whatever the grid, the chunking or the scheduling.
//
// Work decomposition.  The memberships (CSR list positions) run in chunks whose Cartesian paths fit the paths
// buffer of the workspace (kPathBudget bytes, at least one tile).  Per chunk:
//   1. vh_count_kernel: the image shifts of the steps of a block of kFrameBlock frames, summed per block;
//   2. vh_scan_kernel: one block per membership turns the block sums into exclusive prefix sums, K at each block start;
//   3. vh_unwrap_kernel: r(n) of every membership, stored component-planar (membership, c, frame) so that the reads
//      of consecutive origins coalesce;
//   4. vh_histogram_kernel: one persistent launch walks the chunk's items.
// An item is (member tile, origin range of kItemOrigins frames, lag): a tile holds up to kTile list positions of
// one group, and the items of all tiles are numbered ((tile * R) + range) * T + lag, R = ceil(S / kItemOrigins),
// so the numbering depends on S, the lags and the group sizes only.  A thread takes the origins of the range in
// strides of the block and loops over the tile's members; it bins into a shared uint32 histogram with one atomic per
// distinct bin of a warp (__match_any_sync: at short lags a rattling species puts nearly every displacement in a
// few bins) and flushes it with 64-bit atomics after the item (an item has at most kTile * kItemOrigins < 2^31
// displacements, so no shared counter can wrap).  Its sums of rr and rr^2 are reduced in a fixed order and
// written to the item's own slot.  5. vh_finish_kernel, once per call, sums the slots of each (group, lag) in item
// order and normalises the counts, so the moments are bit-identical for every chunking, grid and group set.
// Launches: 4 per membership chunk + 1.
#include <atomic>
#include <cmath>

#include "rn_common.cuh"

namespace rn {

constexpr int kVhThreads = 256;
constexpr int kFrameBlock = 256;         // frames per block of the count and unwrap passes
constexpr int kTile = 32;                // list positions of a group per member tile
constexpr int kItemOrigins = 2048;       // origins per item: kTile * kItemOrigins displacements < 2^31
constexpr int kMaxBins = 4096;           // one uint32 histogram: 16 KB of shared memory
constexpr size_t kPathBudget = 1ull << 30;  // bytes of unwrapped paths per membership chunk

static std::atomic<int64_t> g_van_hove_chunk{0};  // memberships per chunk (tests); 0 = automatic

struct VhTile {
    int64_t off;    // list position of the tile's first membership
    int32_t n;      // memberships of the tile
    int32_t group;
};

struct VhUnwrapParams {
    const double* pos;     // (S, N, 3) fractional
    const int64_t* atoms;  // the chunk's memberships (list positions p0 ..)
    double* shifts;        // (members, fblocks, 3) block sums of the step shifts, then their exclusive scan
    double* paths;         // (members, 3, S) Cartesian unwrapped paths
    int64_t num_frames, num_atoms, members, fblocks;
    double lattice[9];     // rows are lattice vectors
};

struct VhHistParams {
    const double* paths;     // the chunk's paths, membership p at (p - p0) * 3 * S
    const VhTile* tiles;
    const int64_t* lags;     // (T,)
    unsigned long long* counts;  // (G, T, B)
    double2* partials;       // one (sum rr, sum rr^2) per item
    int64_t num_frames, num_lags, ranges, p0;
    int64_t item0, item1;    // the chunk's items
    double inv;              // B / r_max
    double thr;              // rr above this cannot land in a bin: sqrt is skipped
    int num_bins;
};

__device__ __forceinline__ double vh_step_shift(double x1, double x0) {
    return ceil(__dsub_rn(__dsub_rn(x1, x0), 0.5));
}

// block b of membership m: the sums over the steps j -> j + 1, j in the block and j + 1 < S, of the three shifts
__global__ void __launch_bounds__(kVhThreads) vh_count_kernel(const VhUnwrapParams P) {
    __shared__ double sm[3][kVhThreads / 32];
    const int64_t m = blockIdx.x / P.fblocks, fb = blockIdx.x % P.fblocks;
    const int64_t j = fb * kFrameBlock + threadIdx.x;
    const double* x = P.pos + P.atoms[m] * 3;
    double k[3] = {0.0, 0.0, 0.0};
    if (j + 1 < P.num_frames) {
        const double* x0 = x + j * P.num_atoms * 3;
        const double* x1 = x0 + P.num_atoms * 3;
#pragma unroll
        for (int c = 0; c < 3; c++) k[c] = vh_step_shift(__ldg(x1 + c), __ldg(x0 + c));
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int c = 0; c < 3; c++) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) k[c] += __shfl_xor_sync(0xffffffffu, k[c], off);
        if (lane == 0) sm[c][warp] = k[c];
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        double s = 0.0;
        for (int w = 0; w < kVhThreads / 32; w++) s += sm[threadIdx.x][w];
        P.shifts[(m * P.fblocks + fb) * 3 + threadIdx.x] = s;
    }
}

// one block per membership: the block sums become exclusive prefix sums (integers, exact in any order)
__global__ void __launch_bounds__(kVhThreads) vh_scan_kernel(const VhUnwrapParams P) {
    __shared__ double sm[3][kVhThreads];
    double* row = P.shifts + blockIdx.x * P.fblocks * 3;
    double carry[3] = {0.0, 0.0, 0.0};
    for (int64_t base = 0; base < P.fblocks; base += kVhThreads) {
        const int64_t i = base + threadIdx.x;
#pragma unroll
        for (int c = 0; c < 3; c++) sm[c][threadIdx.x] = i < P.fblocks ? row[i * 3 + c] : 0.0;
        __syncthreads();
        for (int off = 1; off < kVhThreads; off <<= 1) {  // Hillis-Steele inclusive scan
            double v[3];
#pragma unroll
            for (int c = 0; c < 3; c++) v[c] = threadIdx.x >= off ? sm[c][threadIdx.x - off] : 0.0;
            __syncthreads();
#pragma unroll
            for (int c = 0; c < 3; c++) sm[c][threadIdx.x] += v[c];
            __syncthreads();
        }
#pragma unroll
        for (int c = 0; c < 3; c++) {
            const double exclusive = carry[c] + (threadIdx.x > 0 ? sm[c][threadIdx.x - 1] : 0.0);
            if (i < P.fblocks) row[i * 3 + c] = exclusive;
            carry[c] += sm[c][kVhThreads - 1];
        }
        __syncthreads();
    }
}

// r(n) of membership m for the frames of block fb: K(n) = K(block start) + the in-block inclusive scan of the shifts
// of the steps n' - 1 -> n', n' in the block
__global__ void __launch_bounds__(kVhThreads) vh_unwrap_kernel(const VhUnwrapParams P) {
    __shared__ double sm[3][kVhThreads];
    const int64_t m = blockIdx.x / P.fblocks, fb = blockIdx.x % P.fblocks;
    const int64_t n = fb * kFrameBlock + threadIdx.x;
    const double* x = P.pos + P.atoms[m] * 3;
    double xn[3] = {0.0, 0.0, 0.0}, k[3] = {0.0, 0.0, 0.0};
    if (n < P.num_frames) {
        const double* xr = x + n * P.num_atoms * 3;
#pragma unroll
        for (int c = 0; c < 3; c++) xn[c] = __ldg(xr + c);
        if (threadIdx.x > 0) {
#pragma unroll
            for (int c = 0; c < 3; c++) k[c] = vh_step_shift(xn[c], __ldg(xr - P.num_atoms * 3 + c));
        }
    }
#pragma unroll
    for (int c = 0; c < 3; c++) sm[c][threadIdx.x] = k[c];
    __syncthreads();
    for (int off = 1; off < kVhThreads; off <<= 1) {
        double v[3];
#pragma unroll
        for (int c = 0; c < 3; c++) v[c] = threadIdx.x >= off ? sm[c][threadIdx.x - off] : 0.0;
        __syncthreads();
#pragma unroll
        for (int c = 0; c < 3; c++) sm[c][threadIdx.x] += v[c];
        __syncthreads();
    }
    if (n >= P.num_frames) return;
    const double* base = P.shifts + (m * P.fblocks + fb) * 3;
    double w[3];
#pragma unroll
    for (int c = 0; c < 3; c++) {
        const double K = base[c] + sm[c][threadIdx.x];  // the step into the block's first frame is in base
        w[c] = __dsub_rn(__dsub_rn(xn[c], __ldg(x + c)), K);
    }
    const double* L = P.lattice;
    double* out = P.paths + m * 3 * P.num_frames + n;
#pragma unroll
    for (int c = 0; c < 3; c++)
        out[c * P.num_frames] = __dadd_rn(__dadd_rn(__dmul_rn(w[0], L[c]), __dmul_rn(w[1], L[3 + c])),
                                          __dmul_rn(w[2], L[6 + c]));
}

__global__ void __launch_bounds__(kVhThreads, 3) vh_histogram_kernel(const VhHistParams p) {
    __shared__ uint32_t hist[kMaxBins];
    __shared__ double2 red[kVhThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int k = threadIdx.x; k < p.num_bins; k += blockDim.x) hist[k] = 0u;
    const int64_t S = p.num_frames;
    for (int64_t item = p.item0 + blockIdx.x; item < p.item1; item += gridDim.x) {
        const int64_t ti = item % p.num_lags, range = (item / p.num_lags) % p.ranges;
        const VhTile tile = p.tiles[item / (p.num_lags * p.ranges)];
        const int64_t t = p.lags[ti];
        const int64_t n0 = range * kItemOrigins, n1 = min(n0 + kItemOrigins, S - t);
        double s2 = 0.0, s4 = 0.0;
        __syncthreads();  // hist is clear
        for (int64_t wbase = n0 + warp * 32; wbase < n1; wbase += blockDim.x) {  // warp-uniform bounds
            const int64_t n = wbase + lane;
            const bool valid = n < n1;
            const double* path = p.paths + (tile.off - p.p0) * 3 * S + (valid ? n : n0);
#pragma unroll 1
            for (int q = 0; q < tile.n; q++, path += 3 * S) {
                int key = -1;
                if (valid) {
                    const double d0 = __dsub_rn(path[t], path[0]);
                    const double d1 = __dsub_rn(path[S + t], path[S]);
                    const double d2 = __dsub_rn(path[2 * S + t], path[2 * S]);
                    const double rr = __dadd_rn(__dadd_rn(__dmul_rn(d0, d0), __dmul_rn(d1, d1)), __dmul_rn(d2, d2));
                    s2 = __dadd_rn(s2, rr);
                    s4 = __dadd_rn(s4, __dmul_rn(rr, rr));
                    if (rr <= p.thr) {  // false for NaN, as k < B is in the definition
                        const double s = __dmul_rn(__dsqrt_rn(rr), p.inv);
                        // floor(s) for 0 <= s < 2^52: 2^52 + s rounded down has floor(s) in its low word
                        if (s < (double)p.num_bins) key = __double2loint(__dadd_rd(s, 4503599627370496.0));
                    }
                }
                const unsigned peers = __match_any_sync(0xffffffffu, key);
                if (key >= 0 && lane == __ffs(peers) - 1) atomicAdd(&hist[key], (uint32_t)__popc(peers));
            }
        }
        // the item's sums in a fixed order: a butterfly over the warp, then the warps in order
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            s2 += __shfl_xor_sync(0xffffffffu, s2, off);
            s4 += __shfl_xor_sync(0xffffffffu, s4, off);
        }
        if (lane == 0) red[warp] = make_double2(s2, s4);
        __syncthreads();  // every displacement of the item is binned
        if (threadIdx.x == 0) {
            double2 total = red[0];
            for (int w = 1; w < kVhThreads / 32; w++) {
                total.x += red[w].x;
                total.y += red[w].y;
            }
            p.partials[item] = total;
        }
        unsigned long long* out = p.counts + (tile.group * p.num_lags + ti) * p.num_bins;
        for (int k = threadIdx.x; k < p.num_bins; k += blockDim.x) {
            const uint32_t v = hist[k];
            if (v) {
                atomicAdd(out + k, (unsigned long long)v);
                hist[k] = 0u;
            }
        }
    }
}

// G_s[g, t, k] = count / ((S - t) |g| shell_k); moments[g, t] = (sum rr, sum rr^2) / ((S - t) |g|), the item slots of
// (g, t) summed in item order
__global__ void vh_finish_kernel(const unsigned long long* __restrict__ counts, const double2* __restrict__ partials,
                                 const int64_t* __restrict__ group_tiles, const int64_t* __restrict__ offsets,
                                 const int64_t* __restrict__ lags, const double* __restrict__ shells, int64_t G,
                                 int64_t T, int64_t B, int64_t S, int64_t ranges, double* __restrict__ van_hove,
                                 double* __restrict__ moments) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t first = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    for (int64_t e = first; e < G * T * B; e += stride) {
        const int64_t gt = e / B, k = e - gt * B, g = gt / T, ti = gt - g * T;
        const double norm = (double)((S - lags[ti]) * (offsets[g + 1] - offsets[g]));
        van_hove[e] = __ddiv_rn((double)counts[e], __dmul_rn(norm, shells[k]));
    }
    for (int64_t gt = first; gt < G * T; gt += stride) {
        const int64_t g = gt / T, ti = gt - g * T;
        double s2 = 0.0, s4 = 0.0;
        for (int64_t tile = group_tiles[g]; tile < group_tiles[g + 1]; tile++)
            for (int64_t r = 0; r < ranges; r++) {
                const double2 v = partials[(tile * ranges + r) * T + ti];
                s2 = __dadd_rn(s2, v.x);
                s4 = __dadd_rn(s4, v.y);
            }
        const double norm = (double)((S - lags[ti]) * (offsets[g + 1] - offsets[g]));
        moments[gt * 2] = __ddiv_rn(s2, norm);
        moments[gt * 2 + 1] = __ddiv_rn(s4, norm);
    }
}

static size_t align256(size_t bytes) { return (bytes + 255) & ~(size_t)255; }

static int64_t max_tiles(int64_t num_groups, int64_t num_listed_atoms) { return num_groups + num_listed_atoms / kTile; }

// memberships per chunk: whole tiles whose paths fit kPathBudget, at least one tile, at most all memberships
static int64_t chunk_capacity(int64_t num_frames, int64_t num_listed_atoms) {
    const int64_t fit = (int64_t)(kPathBudget / (3 * sizeof(double) * (size_t)num_frames)) / kTile * kTile;
    return std::min(num_listed_atoms, std::max<int64_t>(kTile, fit));
}

static int64_t frame_blocks(int64_t num_frames) { return (num_frames + kFrameBlock - 1) / kFrameBlock; }

static int64_t origin_ranges(int64_t num_frames) { return (num_frames + kItemOrigins - 1) / kItemOrigins; }

}  // namespace rn

using namespace rn;

// Workspace layout: counts (G T B uint64), partials (items double2), tiles, group tile offsets (G + 1), group
// offsets (G + 1), lags (T), shells (B), atoms (M), shifts (capacity x fblocks x 3), paths (capacity x 3 x S).
extern "C" size_t rn_van_hove_workspace_size(int64_t num_frames, int64_t num_listed_atoms, int64_t num_groups,
                                             int64_t num_lags, int64_t num_bins) {
    if (num_frames < 2 || num_listed_atoms < 1 || num_groups < 1 || num_lags < 1 || num_bins < 1) return 0;
    const int64_t tiles = max_tiles(num_groups, num_listed_atoms);
    const int64_t cap = chunk_capacity(num_frames, num_listed_atoms);
    return align256((size_t)(num_groups * num_lags * num_bins) * sizeof(uint64_t)) +
           align256((size_t)(tiles * origin_ranges(num_frames) * num_lags) * sizeof(double2)) +
           align256((size_t)tiles * sizeof(VhTile)) + 2 * align256((size_t)(num_groups + 1) * sizeof(int64_t)) +
           align256((size_t)num_lags * sizeof(int64_t)) + align256((size_t)num_bins * sizeof(double)) +
           align256((size_t)num_listed_atoms * sizeof(int64_t)) +
           align256((size_t)(cap * frame_blocks(num_frames) * 3) * sizeof(double)) +
           (size_t)(cap * 3 * num_frames) * sizeof(double);
}

extern "C" int rn_van_hove(const double* d_positions, int64_t num_frames, int64_t num_atoms, const double* h_lattice,
                           const int64_t* h_lags, int64_t num_lags, double r_max, int64_t num_bins,
                           const int64_t* h_group_offsets, const int64_t* h_atoms, int64_t num_groups,
                           double* d_van_hove, double* d_moments, void* d_workspace, void* stream) {
    RN_CHECK_ARG(d_positions && h_lattice && h_lags && h_group_offsets && h_atoms && d_van_hove && d_moments &&
                     d_workspace,
                 "null pointer");
    RN_CHECK_ARG(num_frames >= 2, "num_frames must be at least 2 (got %lld)", (long long)num_frames);
    RN_CHECK_ARG(num_atoms >= 1 && num_atoms <= INT32_MAX, "invalid num_atoms %lld", (long long)num_atoms);
    RN_CHECK_ARG(num_groups >= 1 && num_groups <= 65535, "num_groups must be in 1..65535 (got %lld)",
                 (long long)num_groups);
    RN_CHECK_ARG(num_lags >= 1, "num_lags must be at least 1 (got %lld)", (long long)num_lags);
    for (int64_t i = 0; i < num_lags; i++) {
        RN_CHECK_ARG(h_lags[i] >= 0 && h_lags[i] < num_frames, "lag %lld out of range [0, %lld)",
                     (long long)h_lags[i], (long long)num_frames);
        RN_CHECK_ARG(i == 0 || h_lags[i] > h_lags[i - 1], "lags must be strictly increasing");
    }
    RN_CHECK_ARG(std::isfinite(r_max) && r_max > 0, "r_max must be finite and > 0 (got %g)", r_max);
    RN_CHECK_ARG(num_bins >= 1 && num_bins <= kMaxBins, "num_bins must be in 1..%d (got %lld)", kMaxBins,
                 (long long)num_bins);
    for (int i = 0; i < 9; i++) RN_CHECK_ARG(std::isfinite(h_lattice[i]), "lattice entry %d is not finite", i);
    const double* L = h_lattice;
    const double volume = std::fabs(L[0] * (L[4] * L[8] - L[5] * L[7]) + L[1] * (L[5] * L[6] - L[3] * L[8]) +
                                    L[2] * (L[3] * L[7] - L[4] * L[6]));
    RN_CHECK_ARG(volume > 0 && std::isfinite(volume), "the lattice has zero (or non-finite) cell volume");
    RN_CHECK_ARG(h_group_offsets[0] == 0, "group offsets must start at 0");
    for (int64_t g = 0; g < num_groups; g++)
        RN_CHECK_ARG(h_group_offsets[g + 1] > h_group_offsets[g], "group %lld is empty", (long long)g);
    const int64_t M = h_group_offsets[num_groups];
    RN_CHECK_ARG(M <= INT32_MAX, "too many listed atoms (%lld)", (long long)M);
    std::vector<int64_t> stamp((size_t)num_atoms, -1);
    for (int64_t g = 0; g < num_groups; g++)
        for (int64_t m = h_group_offsets[g]; m < h_group_offsets[g + 1]; m++) {
            const int64_t atom = h_atoms[m];
            RN_CHECK_ARG(atom >= 0 && atom < num_atoms, "atom index %lld of group %lld out of range [0, %lld)",
                         (long long)atom, (long long)g, (long long)num_atoms);
            RN_CHECK_ARG(stamp[(size_t)atom] != g, "group %lld repeats atom %lld", (long long)g, (long long)atom);
            stamp[(size_t)atom] = g;
        }

    const int64_t S = num_frames, T = num_lags, B = num_bins, G = num_groups;
    const int64_t R = origin_ranges(S), fblocks = frame_blocks(S);
    std::vector<VhTile> tiles;
    std::vector<int64_t> group_tiles(1, 0);
    for (int64_t g = 0; g < G; g++) {
        for (int64_t off = h_group_offsets[g]; off < h_group_offsets[g + 1]; off += kTile)
            tiles.push_back({off, (int32_t)std::min<int64_t>(kTile, h_group_offsets[g + 1] - off), (int32_t)g});
        group_tiles.push_back((int64_t)tiles.size());
    }
    const int64_t auto_cap = chunk_capacity(S, M);
    const int64_t forced = g_van_hove_chunk.load(std::memory_order_relaxed);
    const int64_t cap = forced > 0 ? std::min(forced, auto_cap) : auto_cap;
    std::vector<std::pair<size_t, size_t>> chunks;  // tile ranges; a tile never exceeds kTile <= auto_cap members
    for (size_t i = 0; i < tiles.size();) {
        size_t j = i + 1;
        while (j < tiles.size() && tiles[j].off + tiles[j].n - tiles[i].off <= cap) j++;
        chunks.push_back({i, j});
        i = j;
    }

    char* ws = static_cast<char*>(d_workspace);
    auto take = [&](size_t bytes) {
        char* at = ws;
        ws += align256(bytes);
        return at;
    };
    auto* d_counts = reinterpret_cast<unsigned long long*>(take((size_t)(G * T * B) * sizeof(uint64_t)));
    auto* d_partials = reinterpret_cast<double2*>(take((size_t)(max_tiles(G, M) * R * T) * sizeof(double2)));
    auto* d_tiles = reinterpret_cast<VhTile*>(take((size_t)max_tiles(G, M) * sizeof(VhTile)));
    auto* d_group_tiles = reinterpret_cast<int64_t*>(take((size_t)(G + 1) * sizeof(int64_t)));
    auto* d_offsets = reinterpret_cast<int64_t*>(take((size_t)(G + 1) * sizeof(int64_t)));
    auto* d_lags = reinterpret_cast<int64_t*>(take((size_t)T * sizeof(int64_t)));
    auto* d_shells = reinterpret_cast<double*>(take((size_t)B * sizeof(double)));
    auto* d_atoms = reinterpret_cast<int64_t*>(take((size_t)M * sizeof(int64_t)));
    auto* d_shifts = reinterpret_cast<double*>(take((size_t)(auto_cap * fblocks * 3) * sizeof(double)));
    auto* d_paths = reinterpret_cast<double*>(ws);

    // shell volumes (4 pi / 3) (e_{k+1}^3 - e_k^3), e_k = k * width, as rn_rdf
    const double width = r_max / (double)B;
    std::vector<double> shells((size_t)B);
    for (int64_t k = 0; k < B; k++) {
        const double e0 = (double)k * width, e1 = (double)(k + 1) * width;
        shells[(size_t)k] = 4 * M_PI / 3 * (e1 * e1 * e1 - e0 * e0 * e0);
    }

    cudaStream_t s = static_cast<cudaStream_t>(stream);
    // pageable sources: the copies return once the data is staged, so the vectors may go out of scope
    RN_CUDA(cudaMemcpyAsync(d_tiles, tiles.data(), sizeof(VhTile) * tiles.size(), cudaMemcpyHostToDevice, s));
    RN_CUDA(cudaMemcpyAsync(d_group_tiles, group_tiles.data(), sizeof(int64_t) * (size_t)(G + 1),
                            cudaMemcpyHostToDevice, s));
    RN_CUDA(cudaMemcpyAsync(d_offsets, h_group_offsets, sizeof(int64_t) * (size_t)(G + 1), cudaMemcpyHostToDevice, s));
    RN_CUDA(cudaMemcpyAsync(d_lags, h_lags, sizeof(int64_t) * (size_t)T, cudaMemcpyHostToDevice, s));
    RN_CUDA(cudaMemcpyAsync(d_shells, shells.data(), sizeof(double) * (size_t)B, cudaMemcpyHostToDevice, s));
    RN_CUDA(cudaMemcpyAsync(d_atoms, h_atoms, sizeof(int64_t) * (size_t)M, cudaMemcpyHostToDevice, s));
    RN_CUDA(cudaMemsetAsync(d_counts, 0, sizeof(uint64_t) * (size_t)(G * T * B), s));

    int device = 0, sms = 0, per_sm = 0;
    RN_CUDA(cudaGetDevice(&device));
    RN_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    RN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, vh_histogram_kernel, kVhThreads, 0));
    const int64_t grid_max = (int64_t)sms * std::max(per_sm, 1);

    VhUnwrapParams up;
    up.pos = d_positions;
    up.shifts = d_shifts;
    up.paths = d_paths;
    up.num_frames = S;
    up.num_atoms = num_atoms;
    up.fblocks = fblocks;
    for (int i = 0; i < 9; i++) up.lattice[i] = L[i];
    VhHistParams hp;
    hp.paths = d_paths;
    hp.tiles = d_tiles;
    hp.lags = d_lags;
    hp.counts = d_counts;
    hp.partials = d_partials;
    hp.num_frames = S;
    hp.num_lags = T;
    hp.ranges = R;
    hp.inv = (double)B / r_max;
    hp.thr = (r_max * (1 + 1e-6)) * (r_max * (1 + 1e-6));
    hp.num_bins = (int)B;
    for (const auto& chunk : chunks) {
        const int64_t p0 = tiles[chunk.first].off;
        const int64_t members = tiles[chunk.second - 1].off + tiles[chunk.second - 1].n - p0;
        up.atoms = d_atoms + p0;
        up.members = members;
        vh_count_kernel<<<(unsigned)(members * fblocks), kVhThreads, 0, s>>>(up);
        RN_LAUNCHED();
        vh_scan_kernel<<<(unsigned)members, kVhThreads, 0, s>>>(up);
        RN_LAUNCHED();
        vh_unwrap_kernel<<<(unsigned)(members * fblocks), kVhThreads, 0, s>>>(up);
        RN_LAUNCHED();
        hp.p0 = p0;
        hp.item0 = (int64_t)chunk.first * R * T;
        hp.item1 = (int64_t)chunk.second * R * T;
        vh_histogram_kernel<<<(unsigned)std::min(grid_max, hp.item1 - hp.item0), kVhThreads, 0, s>>>(hp);
        RN_LAUNCHED();
    }
    const int64_t outputs = G * T * B;
    vh_finish_kernel<<<(unsigned)std::min<int64_t>((outputs + 255) / 256, (int64_t)sms * 8), 256, 0, s>>>(
        d_counts, d_partials, d_group_tiles, d_offsets, d_lags, d_shells, G, T, B, S, R, d_van_hove, d_moments);
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    return RN_OK;
}

extern "C" void rn_debug_set_van_hove_chunk(int memberships) {
    rn::g_van_hove_chunk.store(memberships, std::memory_order_relaxed);
}
