"""CPU oracle of the distinct Van Hove correlation (``Trajectory.get_distinct_van_hove``): for every ordered group pair
(a, b), lag t and origin n < S - t, the minimum-image distances of x_j(n + t) - x_i(n), i in a, j in b, i != j, binned
into exact integer counts and normalised like ``rdf_oracle.rdf``.  The distance takes the operations of
``rdf_oracle.pair_bins`` in their order.  No reference counterpart; plain numpy (elementwise operations never fuse a
multiply-add).  Test infrastructure only."""
import numpy as np

from rdf_oracle import bin_edges, cell_widths, pair_norms

ORIGIN_CHUNK_PAIRS = 1 << 24  # (origins x N x N) bin indices formed at a time


def lag_pair_bins(x0, x1, lattice, r_max, num_bins):
    """Origin frames x0 and partner frames x1 (F,N,3) -> (F,N,N) float bin index k[f, i, j] of x1_j - x0_i."""
    inv = num_bins / r_max
    d = x1[:, None, :, :] - x0[:, :, None, :]  # d[f, i, j] = x1_j - x0_i
    d = d - np.ceil(d - 0.5)
    v = [(d[..., 0] * lattice[0, c] + d[..., 1] * lattice[1, c]) + d[..., 2] * lattice[2, c] for c in range(3)]
    rr = (v[0] * v[0] + v[1] * v[1]) + v[2] * v[2]
    return np.floor(np.sqrt(rr) * inv)


def _groups(atom_groups, num_atoms):
    if atom_groups is None:
        return [np.arange(num_atoms)]
    return [np.asarray(list(g), dtype=np.int64) for g in atom_groups]


def distinct_counts(positions_ts, lattice, lags, r_max, num_bins, atom_groups=None):
    """(G, G, T, B) int64 counts of the ordered group pairs."""
    x = np.asarray(positions_ts, dtype=np.float64)
    frames, num_atoms = x.shape[:2]
    groups = _groups(atom_groups, num_atoms)
    G = len(groups)
    counts = np.zeros((G, G, len(lags), num_bins), dtype=np.int64)
    chunk = max(1, ORIGIN_CHUNK_PAIRS // (num_atoms * num_atoms))
    for ti, t in enumerate(lags):
        for n0 in range(0, frames - t, chunk):
            n1 = min(frames - t, n0 + chunk)
            k = lag_pair_bins(x[n0:n1], x[n0 + t:n1 + t], lattice, r_max, num_bins)
            for a in range(G):
                for b in range(G):
                    keep = groups[a][:, None] != groups[b][None, :]
                    values = k[:, groups[a]][:, :, groups[b]][:, keep]
                    values = values[values < num_bins].astype(np.int64)
                    counts[a, b, ti] += np.bincount(values, minlength=num_bins)
    return counts


def normalise(counts, frames, lattice, lags, r_max, atom_groups, num_atoms):
    """g_d (G, G, T, B) = count * V / ((S - t) n_ab shell_k), zero where n_ab = 0."""
    volume, _ = cell_widths(lattice)
    _, _, shell = bin_edges(r_max, counts.shape[3])
    norms = pair_norms(atom_groups, num_atoms)
    g = np.zeros(counts.shape)
    for a in range(counts.shape[0]):
        for b in range(counts.shape[1]):
            if norms[a, b] > 0:
                for ti, t in enumerate(lags):
                    g[a, b, ti] = counts[a, b, ti] * volume / ((frames - int(t)) * int(norms[a, b]) * shell)
    return g


def distinct_van_hove(positions_ts, lattice, lags, r_max, num_bins, atom_groups=None):
    """(r, g_d, counts): r (B,) the bin centres, g_d (G, G, T, B) and the counts (G, G, T, B) int64."""
    x = np.asarray(positions_ts, dtype=np.float64)
    frames, num_atoms = x.shape[:2]
    lags = np.asarray(lags, dtype=np.int64)
    counts = distinct_counts(x, lattice, lags, r_max, num_bins, atom_groups)
    r, _, _ = bin_edges(r_max, num_bins)
    return r, normalise(counts, frames, lattice, lags, r_max, atom_groups, num_atoms), counts
