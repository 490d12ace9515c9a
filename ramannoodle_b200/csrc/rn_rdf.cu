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

// Workspace layout: S n_ab per pair (P int64), shells (B doubles), entries, atoms (M int64), counts (P x B uint64).
static int64_t rdf_max_entries(int64_t num_groups, int64_t num_listed_atoms) {
    const int64_t tiles = num_groups + num_listed_atoms / kTile;  // >= the sum of the groups' tile counts
    return tiles * tiles;
}

static size_t align256(size_t bytes) { return (bytes + 255) & ~(size_t)255; }

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
    RN_CHECK_ARG(num_frames >= 1, "num_frames must be at least 1 (got %lld)", (long long)num_frames);
    RN_CHECK_ARG(num_atoms >= 1 && num_atoms <= INT32_MAX, "invalid num_atoms %lld", (long long)num_atoms);
    RN_CHECK_ARG(num_groups >= 1 && num_groups <= 65535, "num_groups must be in 1..65535 (got %lld)",
                 (long long)num_groups);
    RN_CHECK_ARG(num_bins >= 1 && num_bins <= kMaxBins, "num_bins must be in 1..%d (got %lld)", kMaxBins,
                 (long long)num_bins);
    for (int i = 0; i < 9; i++) RN_CHECK_ARG(std::isfinite(h_lattice[i]), "lattice entry %d is not finite", i);
    const double* L = h_lattice;
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

    // groups: sizes, ranges, repeats and the pairwise overlaps |a n b|
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
    const int64_t P = num_groups * (num_groups + 1) / 2;
    std::vector<int64_t> pair_norm((size_t)P);  // S n_ab, n_ab = |a||b| - |a n b|
    std::fill(stamp.begin(), stamp.end(), -1);
    std::vector<int64_t> overlap((size_t)P);
    for (int64_t a = 0, pair = 0; a < num_groups; a++) {
        for (int64_t m = h_group_offsets[a]; m < h_group_offsets[a + 1]; m++) stamp[(size_t)h_atoms[m]] = a;
        for (int64_t b = a; b < num_groups; b++, pair++) {
            int64_t shared = 0;
            for (int64_t m = h_group_offsets[b]; m < h_group_offsets[b + 1]; m++) shared += stamp[(size_t)h_atoms[m]] == a;
            const int64_t na = h_group_offsets[a + 1] - h_group_offsets[a];
            const int64_t nb = h_group_offsets[b + 1] - h_group_offsets[b];
            overlap[(size_t)pair] = shared;
            pair_norm[(size_t)pair] = num_frames * (na * nb - shared);
        }
    }

    // entries: tile pairs of every group pair, with their pair counts per frame
    struct Tile {
        int64_t off;
        int32_t n;
    };
    std::vector<RdfEntry> entries;
    std::vector<int64_t> per_frame;
    auto tiles_of = [&](int64_t g) {
        std::vector<Tile> t;
        for (int64_t off = h_group_offsets[g]; off < h_group_offsets[g + 1]; off += kTile)
            t.push_back({off, (int32_t)std::min<int64_t>(kTile, h_group_offsets[g + 1] - off)});
        return t;
    };
    for (int64_t a = 0, pair = 0; a < num_groups; a++) {
        const std::vector<Tile> ta = tiles_of(a);
        for (int64_t b = a; b < num_groups; b++, pair++) {
            const std::vector<Tile> tb = b == a ? ta : tiles_of(b);
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

    // shell volumes (4 pi / 3) (e_{k+1}^3 - e_k^3), e_k = k * width
    const double width = r_max / (double)num_bins;
    std::vector<double> shells((size_t)num_bins);
    for (int64_t k = 0; k < num_bins; k++) {
        const double e0 = (double)k * width, e1 = (double)(k + 1) * width;
        shells[(size_t)k] = 4 * M_PI / 3 * (e1 * e1 * e1 - e0 * e0 * e0);
    }

    int device = 0, sms = 0, per_sm = 0;
    RN_CUDA(cudaGetDevice(&device));
    RN_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    RN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, rdf_histogram_kernel, kRdfThreads, 0));
    const int64_t grid_max = (int64_t)sms * std::max(per_sm, 1);
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

    RdfParams p;
    p.pos = d_positions;
    p.atoms = d_atoms;
    p.entries = d_entries;
    p.counts = d_counts;
    p.num_entries = (int64_t)entries.size();
    p.num_items = items;
    p.num_frames = num_frames;
    p.num_atoms = num_atoms;
    p.inv = (double)num_bins / r_max;
    p.thr = (r_max * (1 + 1e-6)) * (r_max * (1 + 1e-6));
    p.num_bins = (int)num_bins;
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
