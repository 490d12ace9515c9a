"""CPU oracle of the vibrational density of states (``Trajectory.get_vdos``): the weighted sum, over the atoms of a
group and the three Cartesian components, of ``calc_signal_spectrum`` of the minimum-image velocities.  No reference
counterpart; written with calls ``oracle/numpy_port.py`` already has.  Test infrastructure only."""
import numpy as np

from oracle import numpy_port as ora


def vdos(positions_ts, lattice, timestep, atom_groups, atom_weights):
    """(S,N,3) fractional positions -> wavenumbers (P,), VDOS (G,P); 0 cm^-1 bin dropped as in ``md_measure``."""
    x = ora.apply_pbc(positions_ts)  # what Trajectory stores
    d = ora.apply_pbc_displacement(np.diff(x, axis=0))  # (M,N,3) fractional, minimum image
    v = (d @ lattice) / timestep  # Cartesian, Å/fs; lattice rows are vectors
    wn = ora.calc_signal_spectrum(v[:, 0, 0], timestep)[0][1:]
    out = np.zeros((len(atom_groups), len(wn)))
    for g, atoms in enumerate(atom_groups):
        for i in atoms:
            for c in range(3):
                out[g] += atom_weights[i] * ora.calc_signal_spectrum(v[:, i, c], timestep)[1][1:]
    return wn, out
