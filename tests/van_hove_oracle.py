"""CPU oracle of the self Van Hove correlation (``Trajectory.get_van_hove``): per-group histograms of the single-atom
displacements |r_i(n+t) - r_i(n)| along the paths unwrapped as in ``get_msd``, and their second and fourth moments.
No reference counterpart; plain numpy, elementwise, so that every product and sum is rounded on its own and the
counts are exact integers.  Test infrastructure only."""
import numpy as np

from oracle import numpy_port as ora
from rdf_oracle import bin_edges

ORIGIN_CHUNK = 1 << 22  # (origins x atoms) displacements formed at a time


def unwrapped_paths(x, lattice):
    """(S,N,3) fractional positions, taken as given (``Trajectory`` passes its wrapped ``positions_ts``) -> r (S,N,3)
    in Å.  The image shifts are those of ``msd_oracle.unwrapped_paths``; ``w = (x(n) - x(0)) - K(n)`` and
    ``r_c = (w0 L[0,c] + w1 L[1,c]) + w2 L[2,c]``, the operation order of ``rdf_oracle.pair_bins``."""
    x = np.asarray(x, dtype=np.float64)
    step = np.diff(x, axis=0)
    k = np.rint(step - ora.apply_pbc_displacement(step))  # exact integers
    shifts = np.concatenate([np.zeros_like(x[:1]), np.cumsum(k, axis=0)])  # K(n), K(0) = 0
    w = (x - x[:1]) - shifts
    return np.stack([(w[..., 0] * lattice[0, c] + w[..., 1] * lattice[1, c]) + w[..., 2] * lattice[2, c]
                     for c in range(3)], axis=-1)


def _groups(atom_groups, num_atoms):
    if atom_groups is None:
        return [np.arange(num_atoms)]
    return [np.asarray(list(g), dtype=np.int64) for g in atom_groups]


def van_hove_counts(positions_ts, lattice, lags, r_max, num_bins, atom_groups=None):
    """(counts (G,T,B) int64, sums (G,T,2)): the bin counts and the sums of rr and rr^2 over every membership and
    every origin n < S - t."""
    r = unwrapped_paths(positions_ts, lattice)
    frames, num_atoms = r.shape[:2]
    groups = _groups(atom_groups, num_atoms)
    inv = num_bins / r_max
    counts = np.zeros((len(groups), len(lags), num_bins), dtype=np.int64)
    sums = np.zeros((len(groups), len(lags), 2))
    chunk = max(1, ORIGIN_CHUNK // num_atoms)
    for ti, t in enumerate(lags):
        for n0 in range(0, frames - t, chunk):
            n1 = min(frames - t, n0 + chunk)
            d = r[n0 + t:n1 + t] - r[n0:n1]
            rr = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]  # (origins, N)
            k = np.floor(np.sqrt(rr) * inv)
            for g, atoms in enumerate(groups):
                sub, kg = rr[:, atoms], k[:, atoms]
                sums[g, ti, 0] += np.sum(sub)
                sums[g, ti, 1] += np.sum(sub * sub)
                values = kg[kg < num_bins].astype(np.int64)
                counts[g, ti] += np.bincount(values, minlength=num_bins)
    return counts, sums


def van_hove(positions_ts, lattice, lags, r_max, num_bins, atom_groups=None):
    """(r, g_s, moments, counts): r (B,) the bin centres, g_s (G,T,B) = count / ((S - t) |g| shell_k) in Å^-3,
    moments (G,T,2) = (sum rr, sum rr^2) / ((S - t) |g|), counts (G,T,B) int64."""
    x = np.asarray(positions_ts, dtype=np.float64)
    frames, num_atoms = x.shape[:2]
    lags = np.asarray(lags, dtype=np.int64)
    counts, sums = van_hove_counts(x, lattice, lags, r_max, num_bins, atom_groups)
    r, _, shell = bin_edges(r_max, num_bins)
    sizes = np.array([len(g) for g in _groups(atom_groups, num_atoms)], dtype=np.int64)
    norm = (frames - lags)[None, :] * sizes[:, None]  # (G,T) int64
    g_s = counts / (norm[:, :, None] * shell)
    return r, g_s, sums / norm[:, :, None], counts


def alpha2(moments):
    """The non-Gaussian parameter 3 <rr^2> / (5 <rr>^2) - 1 of moments (..., 2)."""
    return 3 * moments[..., 1] / (5 * moments[..., 0] ** 2) - 1
