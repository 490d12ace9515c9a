// Radial distribution functions g(r) of atom groups (Trajectory.get_rdf).
//
// For every group pair a <= b the pairs (i in a, j in b) of every frame are binned by their minimum-image distance
// into integer histograms; a finishing pass normalises the counts.  The distance follows the definition of
// tests/rdf_oracle.py operation for operation, with explicitly rounded intrinsics so that no multiply-add is fused:
//   d = x_j - x_i;  d -= ceil(d - 0.5)  (per component, wrap_disp of rn_device.cuh)
//   v_c = (d0 L[0,c] + d1 L[1,c]) + d2 L[2,c];  rr = (v0 v0 + v1 v1) + v2 v2;  k = floor(sqrt(rr) * inv)
// so every count equals the oracle's exactly, whatever the grid, the tiling or the scheduling.
//
// Work decomposition.  Each group is cut into tiles of up to kTile list positions.  An entry is one tile pair of
// one group pair: a rectangle (tile of a) x (tile of b), or for a == b on the diagonal the triangle p < q of one
// tile.  The frames of an entry are cut into items of about equal pair counts; one persistent launch walks the
// items with a grid-stride loop.  A block gathers the fractional positions of a batch of frames of the item's
// tiles into shared memory (structure of arrays), gives each thread rows (frame, p) and loops over the partners q,
// binning into a shared uint32 histogram that is flushed with 64-bit atomics at the end of every item (an item has
// fewer than 2^31 pairs, so no shared counter can wrap).
//
// The distinct part of the Van Hove correlation G_d(r, t) (Trajectory.get_distinct_van_hove,
// tests/distinct_van_hove_oracle.py) bins the same distance with x_i taken at origin n and x_j at n + t, for every
// ordered group pair, every requested lag t and every origin n < S - t.  Its kernels (dvh_*) reuse rdf_wrap, rdf_bin,
// rdf_rows and the entries above unchanged, and its host entry shares the checks, overlaps, tiles and shells of rn_rdf.
#include <cmath>

#include "rn_common.cuh"

namespace rn {

constexpr int kRdfThreads = 256;
constexpr int kTile = 256;             // list positions of a group per tile
constexpr int kSlots = 1024;           // (frame, atom) positions one block stages at a time
constexpr int kMaxBins = 4096;         // one uint32 histogram: 16 KB of shared memory
constexpr int64_t kItemPairs = 1LL << 31;  // pairs per item stay below this: the shared counters cannot wrap

struct RdfEntry {
    int64_t item0;    // first item of the entry
    int64_t a_off;    // list position (in the uploaded atom list) of the a-tile's first atom
    int64_t b_off;    // ... of the b-tile (rectangles only)
    int32_t np, nq;   // atoms of the a-tile and the b-tile; nq == 0: the triangle p < q of the a-tile
    int32_t pair;     // histogram of the group pair
    int32_t frames;   // frames per item
    int32_t overlap;  // rectangle of two groups that share atoms: i == j pairs are skipped
    int32_t pad;
};

struct RdfParams {
    const double* pos;  // (S, N, 3)
    const int64_t* atoms;
    const RdfEntry* entries;
    unsigned long long* counts;  // (P, B)
    int64_t num_entries, num_items, num_frames, num_atoms;
    double inv;  // B / r_max
    double thr;  // rr above this cannot land in a bin: sqrt is skipped
    int num_bins;
};

// d - ceil(d - 0.5) of d = xj - xi.  UNIT: both positions lie in [0, 1], so d - 0.5 lies in [-1.5, 0.5] and its
// ceiling is -1, 0 or 1: compare and select give the same value without the FRND instruction (only the sign of a
// zero may differ, which squaring removes).
template <bool UNIT>
__device__ __forceinline__ double rdf_wrap(double xj, double xi) {
    const double d = __dsub_rn(xj, xi);
    const double t = __dsub_rn(d, 0.5);
    if (UNIT) return t > 0.0 ? __dsub_rn(d, 1.0) : (t <= -1.0 ? __dadd_rn(d, 1.0) : d);
    return __dsub_rn(d, ceil(t));
}

template <bool UNIT>
__device__ __forceinline__ void rdf_bin(double xj, double yj, double zj, double xi, double yi, double zi,
                                        const double* L, const RdfParams& p, uint32_t* hist) {
    const double d0 = rdf_wrap<UNIT>(xj, xi), d1 = rdf_wrap<UNIT>(yj, yi), d2 = rdf_wrap<UNIT>(zj, zi);
    const double v0 = __dadd_rn(__dadd_rn(__dmul_rn(d0, L[0]), __dmul_rn(d1, L[3])), __dmul_rn(d2, L[6]));
    const double v1 = __dadd_rn(__dadd_rn(__dmul_rn(d0, L[1]), __dmul_rn(d1, L[4])), __dmul_rn(d2, L[7]));
    const double v2 = __dadd_rn(__dadd_rn(__dmul_rn(d0, L[2]), __dmul_rn(d1, L[5])), __dmul_rn(d2, L[8]));
    const double rr = __dadd_rn(__dadd_rn(__dmul_rn(v0, v0), __dmul_rn(v1, v1)), __dmul_rn(v2, v2));
    if (rr <= p.thr) {  // false for NaN, as k < B is in the definition
        const double s = __dmul_rn(__dsqrt_rn(rr), p.inv);
        if (s < (double)p.num_bins) {
            // floor(s) for 0 <= s < 2^52: 2^52 + s rounded down has floor(s) in its low word
            const int k = __double2loint(__dadd_rd(s, 4503599627370496.0));
            atomicAdd(&hist[k], 1u);
        }
    }
}

// The rows (frame f, position p) of a staged batch, one per thread at a time.  Triangle (nq == 0): the partners
// q = p+1 .. p+nc of p, taken mod np, where nc = np/2 and the last column stops at p < np/2 for an even np, visit
// every pair of the tile once; the lower list position is i.  Rectangle: every q of the b-tile.
template <bool TRI, bool OVERLAP, bool UNIT>
__device__ void rdf_rows(const RdfParams& p, const double* L, int np, int nq, int nfb, const double* sx,
                         const double* sy, const double* sz, const int* sid, uint32_t* hist) {
    const int rows = nfb * np;
    for (int r = threadIdx.x; r < rows; r += blockDim.x) {
        const int f = r / np, pa = r - f * np;
        const double xi = sx[r], yi = sy[r], zi = sz[r];
        if (TRI) {
            const int base = f * np;
            const int nc = (np & 1) == 0 && pa >= np / 2 ? np / 2 - 1 : np / 2;
            const int end = pa + nc;  // last partner, unwrapped
            const int hi = min(end, np - 1);
            for (int q = pa + 1; q <= hi; q++)  // q > p: i = p
                rdf_bin<UNIT>(sx[base + q], sy[base + q], sz[base + q], xi, yi, zi, L, p, hist);
            for (int q = 0; q <= end - np; q++)  // wrapped, q < p: i = q
                rdf_bin<UNIT>(xi, yi, zi, sx[base + q], sy[base + q], sz[base + q], L, p, hist);
        } else {
            const int base = nfb * np + f * nq;
            const int id = OVERLAP ? sid[r] : 0;
            for (int q = 0; q < nq; q++) {
                if (OVERLAP && sid[base + q] == id) continue;
                rdf_bin<UNIT>(sx[base + q], sy[base + q], sz[base + q], xi, yi, zi, L, p, hist);
            }
        }
    }
}

__global__ void __launch_bounds__(kRdfThreads) rdf_histogram_kernel(const RdfParams p, const double3 l0,
                                                                     const double3 l1, const double3 l2) {
    __shared__ uint32_t hist[kMaxBins];
    __shared__ double sx[kSlots], sy[kSlots], sz[kSlots];
    __shared__ int sid[kSlots];
    const double L[9] = {l0.x, l0.y, l0.z, l1.x, l1.y, l1.z, l2.x, l2.y, l2.z};
    for (int k = threadIdx.x; k < p.num_bins; k += blockDim.x) hist[k] = 0u;
    for (int64_t item = blockIdx.x; item < p.num_items; item += gridDim.x) {
        int64_t lo = 0, hi = p.num_entries - 1;  // the entry of the item: last item0 <= item
        while (lo < hi) {
            const int64_t mid = (lo + hi + 1) >> 1;
            if (p.entries[mid].item0 <= item) lo = mid;
            else hi = mid - 1;
        }
        const RdfEntry e = p.entries[lo];
        const int64_t f0 = (item - e.item0) * e.frames;
        const int64_t f1 = min(p.num_frames, f0 + e.frames);
        const int np = e.np, nq = e.nq;
        const int fb = kSlots / (np + nq);
        for (int64_t fs = f0; fs < f1; fs += fb) {
            const int nfb = (int)min((int64_t)fb, f1 - fs);
            __syncthreads();  // the previous batch has been read
            bool unit = true;
            const int na = nfb * np, total = na + nfb * nq;
            for (int k = threadIdx.x; k < total; k += blockDim.x) {
                int f, off;
                int64_t list;
                if (k < na) {
                    f = k / np;
                    off = k - f * np;
                    list = e.a_off + off;
                } else {
                    f = (k - na) / nq;
                    off = k - na - f * nq;
                    list = e.b_off + off;
                }
                const int64_t atom = p.atoms[list];
                const double* x = p.pos + ((fs + f) * p.num_atoms + atom) * 3;
                const double a = x[0], b = x[1], c = x[2];
                sx[k] = a;
                sy[k] = b;
                sz[k] = c;
                sid[k] = (int)atom;
                unit = unit && a >= 0.0 && a <= 1.0 && b >= 0.0 && b <= 1.0 && c >= 0.0 && c <= 1.0;
            }
            unit = __syncthreads_and(unit);
            if (nq == 0) {
                if (unit) rdf_rows<true, false, true>(p, L, np, nq, nfb, sx, sy, sz, sid, hist);
                else rdf_rows<true, false, false>(p, L, np, nq, nfb, sx, sy, sz, sid, hist);
            } else if (e.overlap) {
                if (unit) rdf_rows<false, true, true>(p, L, np, nq, nfb, sx, sy, sz, sid, hist);
                else rdf_rows<false, true, false>(p, L, np, nq, nfb, sx, sy, sz, sid, hist);
            } else {
                if (unit) rdf_rows<false, false, true>(p, L, np, nq, nfb, sx, sy, sz, sid, hist);
                else rdf_rows<false, false, false>(p, L, np, nq, nfb, sx, sy, sz, sid, hist);
            }
        }
        __syncthreads();  // every pair of the item is binned
        unsigned long long* out = p.counts + (int64_t)e.pair * p.num_bins;
        for (int k = threadIdx.x; k < p.num_bins; k += blockDim.x) {
            const uint32_t v = hist[k];
            if (v) {
                atomicAdd(out + k, (unsigned long long)v);
                hist[k] = 0u;
            }
        }
    }
}

// g[a, b, k] = count[a, b, k] * V / ((S n_ab) shell_k), the counts of a == b doubled (ordered pairs), a zero row
// where n_ab == 0; [b, a] mirrors [a, b].
__global__ void rdf_finish_kernel(const unsigned long long* __restrict__ counts, const int64_t* __restrict__ pair_norm,
                                  const double* __restrict__ shells, int64_t G, int64_t B, double volume,
                                  double* __restrict__ out) {
    const int64_t total = G * G * B;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t k = t % B, ab = t / B;
        const int64_t a0 = ab / G, b0 = ab % G;
        const int64_t a = min(a0, b0), b = max(a0, b0);
        const int64_t pair = a * G - a * (a - 1) / 2 + (b - a);
        const int64_t n_frames_pairs = pair_norm[pair];  // S * n_ab
        double g = 0.0;
        if (n_frames_pairs > 0) {
            const unsigned long long c = counts[pair * B + k] * (a == b ? 2ull : 1ull);
            g = __ddiv_rn(__dmul_rn((double)c, volume), __dmul_rn((double)n_frames_pairs, shells[k]));
        }
        out[t] = g;
    }
}

// Distinct part of the Van Hove correlation (Trajectory.get_distinct_van_hove): the pairs (i in a, j in b, i != j) of
// every ordered group pair, with x_i at origin n and x_j at n + t, binned as above.  Every entry is a rectangle (no
// triangle: [a, a, t] counts both orientations), with the overlap flag set whenever a n b is not empty, so that i == j
// is skipped by atom index.  An item is (entry, range of e.frames origins, lag), numbered (item0 + range) T + lag: the
// lag is fastest, so the items in flight share their origin frames in L2.  A batch stages the a-tile at the origins
// fs .. and the b-tile at fs + t .., the layout rdf_rows reads; the counts of item (pair, lag) go to row pair T + lag.
__global__ void __launch_bounds__(kRdfThreads) dvh_histogram_kernel(const RdfParams p, const int64_t* __restrict__ lags,
                                                                     int64_t num_lags, const double3 l0,
                                                                     const double3 l1, const double3 l2) {
    __shared__ uint32_t hist[kMaxBins];
    __shared__ double sx[kSlots], sy[kSlots], sz[kSlots];
    __shared__ int sid[kSlots];
    const double L[9] = {l0.x, l0.y, l0.z, l1.x, l1.y, l1.z, l2.x, l2.y, l2.z};
    for (int k = threadIdx.x; k < p.num_bins; k += blockDim.x) hist[k] = 0u;
    for (int64_t item = blockIdx.x; item < p.num_items; item += gridDim.x) {
        int64_t lo = 0, hi = p.num_entries - 1;  // the entry of the item: last item0 <= item / T
        const int64_t local = item / num_lags, ti = item - local * num_lags;
        while (lo < hi) {
            const int64_t mid = (lo + hi + 1) >> 1;
            if (p.entries[mid].item0 <= local) lo = mid;
            else hi = mid - 1;
        }
        const RdfEntry e = p.entries[lo];
        const int64_t t = lags[ti];
        const int64_t f0 = (local - e.item0) * e.frames;
        const int64_t f1 = min(p.num_frames - t, f0 + e.frames);  // origins n < S - t; the range may be empty
        const int np = e.np, nq = e.nq;
        const int fb = kSlots / (np + nq);
        for (int64_t fs = f0; fs < f1; fs += fb) {
            const int nfb = (int)min((int64_t)fb, f1 - fs);
            __syncthreads();  // the previous batch has been read
            bool unit = true;
            const int na = nfb * np, total = na + nfb * nq;
            for (int k = threadIdx.x; k < total; k += blockDim.x) {
                int f, off;
                int64_t list, frame;
                if (k < na) {
                    f = k / np;
                    off = k - f * np;
                    list = e.a_off + off;
                    frame = fs + f;
                } else {
                    f = (k - na) / nq;
                    off = k - na - f * nq;
                    list = e.b_off + off;
                    frame = fs + t + f;
                }
                const int64_t atom = p.atoms[list];
                const double* x = p.pos + (frame * p.num_atoms + atom) * 3;
                const double a = x[0], b = x[1], c = x[2];
                sx[k] = a;
                sy[k] = b;
                sz[k] = c;
                sid[k] = (int)atom;
                unit = unit && a >= 0.0 && a <= 1.0 && b >= 0.0 && b <= 1.0 && c >= 0.0 && c <= 1.0;
            }
            unit = __syncthreads_and(unit);
            if (e.overlap) {
                if (unit) rdf_rows<false, true, true>(p, L, np, nq, nfb, sx, sy, sz, sid, hist);
                else rdf_rows<false, true, false>(p, L, np, nq, nfb, sx, sy, sz, sid, hist);
            } else {
                if (unit) rdf_rows<false, false, true>(p, L, np, nq, nfb, sx, sy, sz, sid, hist);
                else rdf_rows<false, false, false>(p, L, np, nq, nfb, sx, sy, sz, sid, hist);
            }
        }
        __syncthreads();  // every pair of the item is binned
        // e.pair = a G + b < 65535^2 < 2^32, read unsigned
        unsigned long long* out = p.counts + ((int64_t)(uint32_t)e.pair * num_lags + ti) * p.num_bins;
        for (int k = threadIdx.x; k < p.num_bins; k += blockDim.x) {
            const uint32_t v = hist[k];
            if (v) {
                atomicAdd(out + k, (unsigned long long)v);
                hist[k] = 0u;
            }
        }
    }
}

// g_d[a, b, t, k] = count[a, b, t, k] * V / (((S - t) n_ab) shell_k), a zero row where n_ab == 0: at t = 0 the
// expression, and so every bit, of rdf_finish_kernel.
__global__ void dvh_finish_kernel(const unsigned long long* __restrict__ counts, const int64_t* __restrict__ pair_norm,
                                  const int64_t* __restrict__ lags, const double* __restrict__ shells, int64_t GG,
                                  int64_t T, int64_t B, int64_t S, double volume, double* __restrict__ out) {
    const int64_t total = GG * T * B;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = e / B, k = e - row * B, pair = row / T, ti = row - pair * T;
        const int64_t n_ab = pair_norm[pair];
        double g = 0.0;
        if (n_ab > 0)
            g = __ddiv_rn(__dmul_rn((double)counts[e], volume), __dmul_rn((double)((S - lags[ti]) * n_ab), shells[k]));
        out[e] = g;
    }
}

// Workspace layout: S n_ab per pair (P int64), shells (B doubles), entries, atoms (M int64), counts (P x B uint64).
static int64_t rdf_max_entries(int64_t num_groups, int64_t num_listed_atoms) {
    const int64_t tiles = num_groups + num_listed_atoms / kTile;  // >= the sum of the groups' tile counts
    return tiles * tiles;
}

static size_t align256(size_t bytes) { return (bytes + 255) & ~(size_t)255; }

// ---- host parts shared by rn_rdf and rn_distinct_van_hove ----

static int check_sizes(int64_t num_frames, int64_t num_atoms, int64_t num_groups, int64_t num_bins) {
    RN_CHECK_ARG(num_frames >= 1, "num_frames must be at least 1 (got %lld)", (long long)num_frames);
    RN_CHECK_ARG(num_atoms >= 1 && num_atoms <= INT32_MAX, "invalid num_atoms %lld", (long long)num_atoms);
    RN_CHECK_ARG(num_groups >= 1 && num_groups <= 65535, "num_groups must be in 1..65535 (got %lld)",
                 (long long)num_groups);
    RN_CHECK_ARG(num_bins >= 1 && num_bins <= kMaxBins, "num_bins must be in 1..%d (got %lld)", kMaxBins,
                 (long long)num_bins);
    return RN_OK;
}

// the lattice, its volume V = |L_0 . (L_1 x L_2)| and 0 < r_max <= w_min / 2
static int check_cell(const double* L, double r_max, double* volume_out) {
    for (int i = 0; i < 9; i++) RN_CHECK_ARG(std::isfinite(L[i]), "lattice entry %d is not finite", i);
    double cross[3][3];  // cross[c] = L[c+1] x L[c+2]
    for (int c = 0; c < 3; c++) {
        const double* u = L + 3 * ((c + 1) % 3);
        const double* w = L + 3 * ((c + 2) % 3);
        cross[c][0] = u[1] * w[2] - u[2] * w[1];
        cross[c][1] = u[2] * w[0] - u[0] * w[2];
        cross[c][2] = u[0] * w[1] - u[1] * w[0];
    }
    const double volume = std::fabs(L[0] * cross[0][0] + L[1] * cross[0][1] + L[2] * cross[0][2]);
    RN_CHECK_ARG(volume > 0 && std::isfinite(volume), "the lattice has zero (or non-finite) cell volume");
    double w_min = INFINITY;
    for (int c = 0; c < 3; c++)
        w_min = std::min(w_min, volume / std::sqrt(cross[c][0] * cross[c][0] + cross[c][1] * cross[c][1] +
                                                   cross[c][2] * cross[c][2]));
    RN_CHECK_ARG(r_max > 0 && r_max <= 0.5 * w_min * (1 + 1e-12),
                 "r_max must be in (0, %.17g] Å, half the smallest perpendicular width of the cell (got %g)",
                 0.5 * w_min, r_max);
    *volume_out = volume;
    return RN_OK;
}

// groups: sizes, ranges and repeats
static int check_groups(const int64_t* offsets, const int64_t* atoms, int64_t num_groups, int64_t num_atoms) {
    RN_CHECK_ARG(offsets[0] == 0, "group offsets must start at 0");
    for (int64_t g = 0; g < num_groups; g++)
        RN_CHECK_ARG(offsets[g + 1] > offsets[g], "group %lld is empty", (long long)g);
    const int64_t M = offsets[num_groups];
    RN_CHECK_ARG(M <= INT32_MAX, "too many listed atoms (%lld)", (long long)M);
    std::vector<int64_t> stamp((size_t)num_atoms, -1);
    for (int64_t g = 0; g < num_groups; g++)
        for (int64_t m = offsets[g]; m < offsets[g + 1]; m++) {
            const int64_t atom = atoms[m];
            RN_CHECK_ARG(atom >= 0 && atom < num_atoms, "atom index %lld of group %lld out of range [0, %lld)",
                         (long long)atom, (long long)g, (long long)num_atoms);
            RN_CHECK_ARG(stamp[(size_t)atom] != g, "group %lld repeats atom %lld", (long long)g, (long long)atom);
            stamp[(size_t)atom] = g;
        }
    return RN_OK;
}

// |a n b| of the group pairs a <= b, in the order a G - a (a - 1) / 2 + (b - a) of rdf_finish_kernel
static std::vector<int64_t> group_overlaps(const int64_t* offsets, const int64_t* atoms, int64_t num_groups,
                                           int64_t num_atoms) {
    std::vector<int64_t> stamp((size_t)num_atoms, -1);
    std::vector<int64_t> overlap((size_t)(num_groups * (num_groups + 1) / 2));
    for (int64_t a = 0, pair = 0; a < num_groups; a++) {
        for (int64_t m = offsets[a]; m < offsets[a + 1]; m++) stamp[(size_t)atoms[m]] = a;
        for (int64_t b = a; b < num_groups; b++, pair++) {
            int64_t shared = 0;
            for (int64_t m = offsets[b]; m < offsets[b + 1]; m++) shared += stamp[(size_t)atoms[m]] == a;
            overlap[(size_t)pair] = shared;
        }
    }
    return overlap;
}

struct Tile {
    int64_t off;
    int32_t n;
};

static std::vector<Tile> group_tiles(const int64_t* offsets, int64_t g) {
    std::vector<Tile> t;
    for (int64_t off = offsets[g]; off < offsets[g + 1]; off += kTile)
        t.push_back({off, (int32_t)std::min<int64_t>(kTile, offsets[g + 1] - off)});
    return t;
}

// shell volumes (4 pi / 3) (e_{k+1}^3 - e_k^3), e_k = k * width
static std::vector<double> shell_volumes(double r_max, int64_t num_bins) {
    const double width = r_max / (double)num_bins;
    std::vector<double> shells((size_t)num_bins);
    for (int64_t k = 0; k < num_bins; k++) {
        const double e0 = (double)k * width, e1 = (double)(k + 1) * width;
        shells[(size_t)k] = 4 * M_PI / 3 * (e1 * e1 * e1 - e0 * e0 * e0);
    }
    return shells;
}

// SMs x resident blocks of a histogram kernel
template <typename Kernel>
static int histogram_grid(Kernel kernel, int* sms, int64_t* grid_max) {
    int device = 0, per_sm = 0;
    RN_CUDA(cudaGetDevice(&device));
    RN_CUDA(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, device));
    RN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kRdfThreads, 0));
    *grid_max = (int64_t)*sms * std::max(per_sm, 1);
    return RN_OK;
}

static RdfParams histogram_params(const double* positions, const int64_t* atoms, const RdfEntry* entries,
                                  unsigned long long* counts, int64_t num_entries, int64_t num_items,
                                  int64_t num_frames, int64_t num_atoms, double r_max, int64_t num_bins) {
    RdfParams p;
    p.pos = positions;
    p.atoms = atoms;
    p.entries = entries;
    p.counts = counts;
    p.num_entries = num_entries;
    p.num_items = num_items;
    p.num_frames = num_frames;
    p.num_atoms = num_atoms;
    p.inv = (double)num_bins / r_max;
    p.thr = (r_max * (1 + 1e-6)) * (r_max * (1 + 1e-6));
    p.num_bins = (int)num_bins;
    return p;
}

}  // namespace rn

using namespace rn;

extern "C" size_t rn_rdf_workspace_size(int64_t num_groups, int64_t num_listed_atoms, int64_t num_bins) {
    if (num_groups < 1 || num_listed_atoms < 1 || num_bins < 1) return 0;
    const size_t pairs = (size_t)(num_groups * (num_groups + 1) / 2);
    return align256(pairs * sizeof(int64_t)) + align256((size_t)num_bins * sizeof(double)) +
           align256((size_t)rdf_max_entries(num_groups, num_listed_atoms) * sizeof(RdfEntry)) +
           align256((size_t)num_listed_atoms * sizeof(int64_t)) + pairs * (size_t)num_bins * sizeof(uint64_t);
}

extern "C" int rn_rdf(const double* d_positions, int64_t num_frames, int64_t num_atoms, const double* h_lattice,
                      double r_max, int64_t num_bins, const int64_t* h_group_offsets, const int64_t* h_atoms,
                      int64_t num_groups, double* d_rdf, void* d_workspace, void* stream) {
    RN_CHECK_ARG(d_positions && h_lattice && h_group_offsets && h_atoms && d_rdf && d_workspace, "null pointer");
    int status = check_sizes(num_frames, num_atoms, num_groups, num_bins);
    if (status != RN_OK) return status;
    double volume = 0.0;
    status = check_cell(h_lattice, r_max, &volume);
    if (status != RN_OK) return status;
    status = check_groups(h_group_offsets, h_atoms, num_groups, num_atoms);
    if (status != RN_OK) return status;
    const double* L = h_lattice;
    const int64_t M = h_group_offsets[num_groups];
    const int64_t P = num_groups * (num_groups + 1) / 2;
    const std::vector<int64_t> overlap = group_overlaps(h_group_offsets, h_atoms, num_groups, num_atoms);
    std::vector<int64_t> pair_norm((size_t)P);  // S n_ab, n_ab = |a||b| - |a n b|
    for (int64_t a = 0, pair = 0; a < num_groups; a++)
        for (int64_t b = a; b < num_groups; b++, pair++) {
            const int64_t na = h_group_offsets[a + 1] - h_group_offsets[a];
            const int64_t nb = h_group_offsets[b + 1] - h_group_offsets[b];
            pair_norm[(size_t)pair] = num_frames * (na * nb - overlap[(size_t)pair]);
        }

    // entries: tile pairs of every group pair, with their pair counts per frame
    std::vector<RdfEntry> entries;
    std::vector<int64_t> per_frame;
    for (int64_t a = 0, pair = 0; a < num_groups; a++) {
        const std::vector<Tile> ta = group_tiles(h_group_offsets, a);
        for (int64_t b = a; b < num_groups; b++, pair++) {
            const std::vector<Tile> tb = b == a ? ta : group_tiles(h_group_offsets, b);
            for (size_t i = 0; i < ta.size(); i++)
                for (size_t j = (b == a ? i : 0); j < tb.size(); j++) {
                    RdfEntry e{};
                    e.a_off = ta[i].off;
                    e.np = ta[i].n;
                    e.pair = (int32_t)pair;
                    if (b == a && i == j) {
                        if (e.np < 2) continue;  // a one-atom tile has no pair with itself
                        e.nq = 0;
                        per_frame.push_back((int64_t)e.np * (e.np - 1) / 2);
                    } else {
                        e.b_off = tb[j].off;
                        e.nq = tb[j].n;
                        e.overlap = overlap[(size_t)pair] > 0;
                        per_frame.push_back((int64_t)e.np * e.nq);
                    }
                    entries.push_back(e);
                }
        }
    }

    char* ws = static_cast<char*>(d_workspace);
    int64_t* d_pair_norm = reinterpret_cast<int64_t*>(ws);
    ws += align256((size_t)P * sizeof(int64_t));
    double* d_shells = reinterpret_cast<double*>(ws);
    ws += align256((size_t)num_bins * sizeof(double));
    RdfEntry* d_entries = reinterpret_cast<RdfEntry*>(ws);
    ws += align256((size_t)rdf_max_entries(num_groups, M) * sizeof(RdfEntry));
    int64_t* d_atoms = reinterpret_cast<int64_t*>(ws);
    ws += align256((size_t)M * sizeof(int64_t));
    unsigned long long* d_counts = reinterpret_cast<unsigned long long*>(ws);

    const std::vector<double> shells = shell_volumes(r_max, num_bins);

    int sms = 0;
    int64_t grid_max = 0;
    status = histogram_grid(rdf_histogram_kernel, &sms, &grid_max);
    if (status != RN_OK) return status;
    // items of about equal pair counts, four per block
    int64_t total_pairs = 0;
    for (int64_t c : per_frame) total_pairs += c * num_frames;
    const int64_t target = std::max<int64_t>(1, total_pairs / (4 * grid_max));
    int64_t items = 0;
    for (size_t e = 0; e < entries.size(); e++) {
        const int64_t c = per_frame[e];
        const int64_t frames = std::min<int64_t>({std::max<int64_t>(1, target / c), num_frames, kItemPairs / c});
        entries[e].frames = (int32_t)frames;
        entries[e].item0 = items;
        items += (num_frames + frames - 1) / frames;
    }

    cudaStream_t s = static_cast<cudaStream_t>(stream);
    // pageable sources: the copies return once the data is staged, so the vectors may go out of scope
    RN_CUDA(cudaMemcpyAsync(d_pair_norm, pair_norm.data(), sizeof(int64_t) * (size_t)P, cudaMemcpyHostToDevice, s));
    RN_CUDA(cudaMemcpyAsync(d_shells, shells.data(), sizeof(double) * (size_t)num_bins, cudaMemcpyHostToDevice, s));
    if (!entries.empty())
        RN_CUDA(cudaMemcpyAsync(d_entries, entries.data(), sizeof(RdfEntry) * entries.size(), cudaMemcpyHostToDevice,
                                s));
    RN_CUDA(cudaMemcpyAsync(d_atoms, h_atoms, sizeof(int64_t) * (size_t)M, cudaMemcpyHostToDevice, s));
    RN_CUDA(cudaMemsetAsync(d_counts, 0, sizeof(uint64_t) * (size_t)P * (size_t)num_bins, s));

    const RdfParams p = histogram_params(d_positions, d_atoms, d_entries, d_counts, (int64_t)entries.size(), items,
                                         num_frames, num_atoms, r_max, num_bins);
    const double3 l0 = make_double3(L[0], L[1], L[2]), l1 = make_double3(L[3], L[4], L[5]),
                  l2 = make_double3(L[6], L[7], L[8]);
    // launched even without items (every group a single atom), so that a call always makes the same launches
    rdf_histogram_kernel<<<(unsigned)std::max<int64_t>(1, std::min(grid_max, items)), kRdfThreads, 0, s>>>(p, l0, l1,
                                                                                                        l2);
    RN_LAUNCHED();
    const int64_t outputs = num_groups * num_groups * num_bins;
    rdf_finish_kernel<<<(unsigned)std::min<int64_t>((outputs + 255) / 256, (int64_t)sms * 8), 256, 0, s>>>(
        d_counts, d_pair_norm, d_shells, num_groups, num_bins, volume, d_rdf);
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    return RN_OK;
}

// Workspace layout: n_ab per ordered pair (G G int64), lags (T int64), shells (B doubles), entries, atoms (M int64),
// counts (G G T x B uint64).
extern "C" size_t rn_distinct_van_hove_workspace_size(int64_t num_listed_atoms, int64_t num_groups, int64_t num_lags,
                                                      int64_t num_bins) {
    if (num_listed_atoms < 1 || num_groups < 1 || num_lags < 1 || num_bins < 1) return 0;
    const size_t pairs = (size_t)(num_groups * num_groups);
    return align256(pairs * sizeof(int64_t)) + align256((size_t)num_lags * sizeof(int64_t)) +
           align256((size_t)num_bins * sizeof(double)) +
           align256((size_t)rdf_max_entries(num_groups, num_listed_atoms) * sizeof(RdfEntry)) +
           align256((size_t)num_listed_atoms * sizeof(int64_t)) +
           pairs * (size_t)num_lags * (size_t)num_bins * sizeof(uint64_t);
}

extern "C" int rn_distinct_van_hove(const double* d_positions, int64_t num_frames, int64_t num_atoms,
                                    const double* h_lattice, const int64_t* h_lags, int64_t num_lags, double r_max,
                                    int64_t num_bins, const int64_t* h_group_offsets, const int64_t* h_atoms,
                                    int64_t num_groups, double* d_out, void* d_workspace, void* stream) {
    RN_CHECK_ARG(d_positions && h_lattice && h_lags && h_group_offsets && h_atoms && d_out && d_workspace,
                 "null pointer");
    int status = check_sizes(num_frames, num_atoms, num_groups, num_bins);
    if (status != RN_OK) return status;
    RN_CHECK_ARG(num_lags >= 1, "num_lags must be at least 1 (got %lld)", (long long)num_lags);
    for (int64_t i = 0; i < num_lags; i++) {
        RN_CHECK_ARG(h_lags[i] >= 0 && h_lags[i] < num_frames, "lag %lld out of range [0, %lld)",
                     (long long)h_lags[i], (long long)num_frames);
        RN_CHECK_ARG(i == 0 || h_lags[i] > h_lags[i - 1], "lags must be strictly increasing");
    }
    double volume = 0.0;
    status = check_cell(h_lattice, r_max, &volume);
    if (status != RN_OK) return status;
    status = check_groups(h_group_offsets, h_atoms, num_groups, num_atoms);
    if (status != RN_OK) return status;
    const double* L = h_lattice;
    const int64_t S = num_frames, T = num_lags, B = num_bins, G = num_groups, M = h_group_offsets[G];
    const std::vector<int64_t> overlap = group_overlaps(h_group_offsets, h_atoms, G, num_atoms);
    auto shared = [&](int64_t a, int64_t b) {
        const int64_t lo = std::min(a, b), hi = std::max(a, b);
        return overlap[(size_t)(lo * G - lo * (lo - 1) / 2 + (hi - lo))];
    };
    std::vector<int64_t> pair_norm((size_t)(G * G));  // n_ab = |a||b| - |a n b|
    for (int64_t a = 0; a < G; a++)
        for (int64_t b = 0; b < G; b++)
            pair_norm[(size_t)(a * G + b)] = (h_group_offsets[a + 1] - h_group_offsets[a]) *
                                                 (h_group_offsets[b + 1] - h_group_offsets[b]) -
                                             shared(a, b);

    // entries: every tile pair of every ordered group pair is a rectangle
    std::vector<std::vector<Tile>> tiles((size_t)G);
    for (int64_t g = 0; g < G; g++) tiles[(size_t)g] = group_tiles(h_group_offsets, g);
    std::vector<RdfEntry> entries;
    for (int64_t a = 0; a < G; a++)
        for (int64_t b = 0; b < G; b++)
            for (const Tile& ta : tiles[(size_t)a])
                for (const Tile& tb : tiles[(size_t)b]) {
                    RdfEntry e{};
                    e.a_off = ta.off;
                    e.np = ta.n;
                    e.b_off = tb.off;
                    e.nq = tb.n;
                    e.pair = (int32_t)(uint32_t)(a * G + b);
                    e.overlap = shared(a, b) > 0;
                    entries.push_back(e);
                }

    char* ws = static_cast<char*>(d_workspace);
    auto take = [&](size_t bytes) {
        char* at = ws;
        ws += align256(bytes);
        return at;
    };
    auto* d_pair_norm = reinterpret_cast<int64_t*>(take((size_t)(G * G) * sizeof(int64_t)));
    auto* d_lags = reinterpret_cast<int64_t*>(take((size_t)T * sizeof(int64_t)));
    auto* d_shells = reinterpret_cast<double*>(take((size_t)B * sizeof(double)));
    auto* d_entries = reinterpret_cast<RdfEntry*>(take((size_t)rdf_max_entries(G, M) * sizeof(RdfEntry)));
    auto* d_atoms = reinterpret_cast<int64_t*>(take((size_t)M * sizeof(int64_t)));
    auto* d_counts = reinterpret_cast<unsigned long long*>(ws);

    const std::vector<double> shells = shell_volumes(r_max, B);

    int sms = 0;
    int64_t grid_max = 0;
    status = histogram_grid(dvh_histogram_kernel, &sms, &grid_max);
    if (status != RN_OK) return status;
    // items of about equal pair counts, four per block: an entry's origins n < S - lags[0] are cut into ranges of
    // e.frames origins, one item per (range, lag); ranges beyond S - t are empty for lag t
    int64_t origins = 0;
    for (int64_t i = 0; i < T; i++) origins += S - h_lags[i];
    int64_t total_pairs = 0;
    for (const RdfEntry& e : entries) total_pairs += (int64_t)e.np * e.nq * origins;
    const int64_t target = std::max<int64_t>(1, total_pairs / (4 * grid_max));
    const int64_t first_origins = S - h_lags[0];
    int64_t ranges = 0;
    for (RdfEntry& e : entries) {
        const int64_t c = (int64_t)e.np * e.nq;
        const int64_t frames = std::min<int64_t>({std::max<int64_t>(1, target / c), first_origins, kItemPairs / c});
        e.frames = (int32_t)frames;
        e.item0 = ranges;
        ranges += (first_origins + frames - 1) / frames;
    }
    const int64_t items = ranges * T;

    cudaStream_t s = static_cast<cudaStream_t>(stream);
    // pageable sources: the copies return once the data is staged, so the vectors may go out of scope
    RN_CUDA(cudaMemcpyAsync(d_pair_norm, pair_norm.data(), sizeof(int64_t) * (size_t)(G * G), cudaMemcpyHostToDevice,
                            s));
    RN_CUDA(cudaMemcpyAsync(d_lags, h_lags, sizeof(int64_t) * (size_t)T, cudaMemcpyHostToDevice, s));
    RN_CUDA(cudaMemcpyAsync(d_shells, shells.data(), sizeof(double) * (size_t)B, cudaMemcpyHostToDevice, s));
    RN_CUDA(cudaMemcpyAsync(d_entries, entries.data(), sizeof(RdfEntry) * entries.size(), cudaMemcpyHostToDevice, s));
    RN_CUDA(cudaMemcpyAsync(d_atoms, h_atoms, sizeof(int64_t) * (size_t)M, cudaMemcpyHostToDevice, s));
    RN_CUDA(cudaMemsetAsync(d_counts, 0, sizeof(uint64_t) * (size_t)(G * G * T * B), s));

    const RdfParams p = histogram_params(d_positions, d_atoms, d_entries, d_counts, (int64_t)entries.size(), items, S,
                                         num_atoms, r_max, B);
    const double3 l0 = make_double3(L[0], L[1], L[2]), l1 = make_double3(L[3], L[4], L[5]),
                  l2 = make_double3(L[6], L[7], L[8]);
    dvh_histogram_kernel<<<(unsigned)std::min(grid_max, items), kRdfThreads, 0, s>>>(p, d_lags, T, l0, l1, l2);
    RN_LAUNCHED();
    const int64_t outputs = G * G * T * B;
    dvh_finish_kernel<<<(unsigned)std::min<int64_t>((outputs + 255) / 256, (int64_t)sms * 8), 256, 0, s>>>(
        d_counts, d_pair_norm, d_lags, d_shells, G * G, T, B, S, volume, d_out);
    RN_LAUNCHED();
    RN_CUDA(cudaGetLastError());
    return RN_OK;
}
