"""CPU oracle of the radial distribution functions (``Trajectory.get_rdf``): per-frame minimum-image pair distances of
atom groups, binned into exact integer counts and normalised by the ideal-gas shell counts.  No reference counterpart;
plain numpy (elementwise operations never fuse a multiply-add, so every product and sum is rounded on its own).  Test
infrastructure only."""
import numpy as np

FRAME_CHUNK_PAIRS = 1 << 24  # (frames x N x N) bin indices formed at a time


def cell_widths(lattice):
    """(V, w): V = |det L| = |L_0 . (L_1 x L_2)| and the perpendicular widths w_c = V / |L_{c+1} x L_{c+2}|."""
    volume = abs(np.dot(lattice[0], np.cross(lattice[1], lattice[2])))
    cross = np.cross(lattice[[1, 2, 0]], lattice[[2, 0, 1]])
    return volume, volume / np.sqrt(np.sum(cross * cross, axis=1))


def bin_edges(r_max, num_bins):
    """(r, e, shell): bin centres (B,), edges (B+1,) and shell volumes (B,)."""
    width = r_max / num_bins
    edges = np.arange(num_bins + 1) * width
    shell = 4 * np.pi / 3 * (edges[1:] * edges[1:] * edges[1:] - edges[:-1] * edges[:-1] * edges[:-1])
    return (np.arange(num_bins) + 0.5) * width, edges, shell


def pair_bins(x, lattice, r_max, num_bins):
    """(F,N,3) fractional positions -> (F,N,N) float bin index k[f, i, j] = floor(|wrap(x_j - x_i) @ L| * inv)."""
    inv = num_bins / r_max
    d = x[:, None, :, :] - x[:, :, None, :]  # d[f, i, j] = x_j - x_i
    d = d - np.ceil(d - 0.5)
    v = [(d[..., 0] * lattice[0, c] + d[..., 1] * lattice[1, c]) + d[..., 2] * lattice[2, c] for c in range(3)]
    rr = (v[0] * v[0] + v[1] * v[1]) + v[2] * v[2]
    return np.floor(np.sqrt(rr) * inv)


def _groups(atom_groups, num_atoms):
    if atom_groups is None:
        return [np.arange(num_atoms)]
    return [np.asarray(list(g), dtype=np.int64) for g in atom_groups]


def rdf_counts(positions_ts, lattice, r_max, num_bins, atom_groups=None):
    """(G, G, B) int64 counts: ordered pairs, so a group with itself counts every pair p < q twice."""
    x = np.asarray(positions_ts, dtype=np.float64)
    frames, num_atoms = x.shape[:2]
    groups = _groups(atom_groups, num_atoms)
    G = len(groups)
    counts = np.zeros((G, G, num_bins), dtype=np.int64)
    chunk = max(1, FRAME_CHUNK_PAIRS // (num_atoms * num_atoms))
    for f0 in range(0, frames, chunk):
        k = pair_bins(x[f0:f0 + chunk], lattice, r_max, num_bins)
        for a in range(G):
            for b in range(a, G):
                sub = k[:, groups[a]][:, :, groups[b]]
                if a == b:
                    keep = np.triu(np.ones(sub.shape[1:], dtype=bool), 1)
                else:
                    keep = groups[a][:, None] != groups[b][None, :]
                values = sub[:, keep]
                values = values[values < num_bins].astype(np.int64)
                counts[a, b] += np.bincount(values, minlength=num_bins) * (2 if a == b else 1)
    for a in range(G):
        for b in range(a):
            counts[a, b] = counts[b, a]
    return counts


def pair_norms(atom_groups, num_atoms):
    """n_ab = |a| |b| - |a n b| (G, G) int64."""
    groups = _groups(atom_groups, num_atoms)
    return np.array([[len(a) * len(b) - len(np.intersect1d(a, b)) for b in groups] for a in groups], dtype=np.int64)


def rdf(positions_ts, lattice, r_max, num_bins, atom_groups=None, counts=None):
    """(r, g, counts): r (B,), g (G, G, B) = count * V / (S n_ab shell_k), zero where n_ab = 0."""
    x = np.asarray(positions_ts, dtype=np.float64)
    frames, num_atoms = x.shape[:2]
    if counts is None:
        counts = rdf_counts(x, lattice, r_max, num_bins, atom_groups)
    volume, _ = cell_widths(lattice)
    r, _, shell = bin_edges(r_max, num_bins)
    norms = pair_norms(atom_groups, num_atoms)
    g = np.zeros(counts.shape)
    for a in range(counts.shape[0]):
        for b in range(counts.shape[1]):
            if norms[a, b] > 0:
                g[a, b] = counts[a, b] * volume / (frames * int(norms[a, b]) * shell)
    return r, g, counts
