"""CPU oracle of the projected VDOS (``Trajectory.get_projected_vdos``): ``calc_signal_spectrum`` of the minimum-image
velocities of ``vdos_oracle`` projected on K vectors.  No reference counterpart; written with calls
``oracle/numpy_port.py`` already has.  Test infrastructure only."""
import numpy as np

from oracle import numpy_port as ora


def velocities(positions_ts, lattice, timestep):
    """(S,N,3) fractional positions -> (S-1,N,3) Cartesian velocities in Å/fs, formed as ``vdos_oracle.vdos`` does."""
    x = ora.apply_pbc(positions_ts)  # what Trajectory stores
    d = ora.apply_pbc_displacement(np.diff(x, axis=0))  # (M,N,3) fractional, minimum image
    return (d @ lattice) / timestep  # lattice rows are vectors


def projected_vdos(positions_ts, lattice, timestep, vectors):
    """-> wavenumbers (P,), rows (K,P): row k is calc_signal_spectrum(sum_{i,c} vectors[k,i,c] v[:,i,c])[1:]."""
    q = np.einsum("kic,nic->kn", np.asarray(vectors, dtype=np.float64), velocities(positions_ts, lattice, timestep))
    wn = ora.calc_signal_spectrum(q[0], timestep)[0][1:]
    rows = np.stack([ora.calc_signal_spectrum(q[k], timestep)[1][1:] for k in range(q.shape[0])])
    return wn, rows
