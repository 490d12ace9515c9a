"""CPU oracle of the mean squared displacement (``Trajectory.get_msd``): the per-group mean, over atoms and time
origins, of the squared displacement along the path unwrapped with the minimum-image steps of ``get_vdos``.  No
reference counterpart; written with calls ``oracle/numpy_port.py`` already has.  Test infrastructure only."""
import numpy as np

from oracle import numpy_port as ora


def unwrapped_paths(positions_ts, lattice):
    """(S,N,3) fractional positions -> r (S,N,3) in Å: ``(x(n) - x(0) - K(n)) @ lattice`` with K the running sum of the
    integer image shifts of the minimum-image steps."""
    x = ora.apply_pbc(positions_ts)  # what Trajectory stores
    step = np.diff(x, axis=0)
    d = ora.apply_pbc_displacement(step)  # (S-1,N,3) in (-0.5, 0.5], the steps of get_vdos
    k = np.rint(step - d)  # exact integers
    shifts = np.concatenate([np.zeros_like(x[:1]), np.cumsum(k, axis=0)])  # K(n), K(0) = 0
    return (x - x[:1] - shifts) @ lattice


def _group_rows(per_atom, atom_groups):
    return np.stack([np.mean(per_atom[list(atoms)], axis=0) for atoms in atom_groups])


def msd_direct(positions_ts, lattice, timestep, atom_groups):
    """Direct form (small S): lag_times (S,), msd (G,S)."""
    r = unwrapped_paths(positions_ts, lattice)
    frames, num_atoms = r.shape[:2]
    per_atom = np.zeros((num_atoms, frames))
    for m in range(1, frames):
        per_atom[:, m] = np.mean(np.sum((r[m:] - r[:-m]) ** 2, axis=2), axis=0)
    return np.arange(frames) * timestep, _group_rows(per_atom, atom_groups)


def msd_fft(positions_ts, lattice, timestep, atom_groups):
    """numpy FFT form (long trajectories): |r(n+m) - r(n)|^2 summed over n < S-m as
    sum_{n<S-m} D(n) + sum_{n>=m} D(n) - 2 C(m), D = |r|^2, C the zero-padded autocorrelation."""
    r = unwrapped_paths(positions_ts, lattice)
    frames = r.shape[0]
    n = 1 << int(2 * frames - 1).bit_length()
    spectrum = np.fft.rfft(r, n=n, axis=0)
    c = np.sum(np.fft.irfft(spectrum.real ** 2 + spectrum.imag ** 2, n=n, axis=0)[:frames], axis=2).T  # (N,S)
    prefix = np.concatenate([np.zeros((1, r.shape[1])), np.cumsum(np.sum(r * r, axis=2), axis=0)]).T  # (N,S+1)
    lags = np.arange(frames)
    a = prefix[:, frames - lags] + (prefix[:, -1:] - prefix[:, lags])
    per_atom = (a - 2 * c) / (frames - lags)
    per_atom[:, 0] = 0.0
    return lags * timestep, _group_rows(per_atom, atom_groups)


def energies(positions_ts, lattice, atom_groups):
    """E_g = sum over the group's atoms and all frames of |r_i(n)|^2: the scale of an FFT correlation's error."""
    r = unwrapped_paths(positions_ts, lattice)
    per_atom = np.sum(r * r, axis=(0, 2))
    return np.array([np.sum(per_atom[list(atoms)]) for atoms in atom_groups])


def error_ratio(got, want, positions_ts, lattice, atom_groups):
    """max |got - want| / scale_g(m), scale_g(m) = 2 E_g / ((S - m) |g|); lag 0 is compared exactly."""
    frames = want.shape[1]
    sizes = np.array([len(list(atoms)) for atoms in atom_groups], dtype=np.float64)
    scale = 2 * energies(positions_ts, lattice, atom_groups)[:, None] / ((frames - np.arange(frames))[None] * sizes[:, None])
    scale = np.maximum(scale, np.finfo(np.float64).tiny)
    return float(np.max(np.abs(got - want) / scale))
