/*
 * ramannoodle_b200 — test and tuning hooks of libramannoodle_b200.so.
 *
 * Not part of the drop-in boundary (include/ramannoodle_b200.h): these entries let the parity
 * tests force the fallback kernels / alternative schedules and check the FFT core directly.
 * The A/B switches are process-wide atomics that every launch reads once; flipping one while
 * another thread is inside a call only changes which (equally correct) kernel the NEXT launch uses.
 */
#ifndef RAMANNOODLE_B200_DEBUG_H
#define RAMANNOODLE_B200_DEBUG_H

#include "ramannoodle_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* route the affine (linear-DOF) term through affine_generic_kernel instead of the TMA kernel */
void rn_debug_force_generic_affine(int on);
/* frames-per-tile multiplier (1, 2; 0 = automatic) of the TMA affine kernel */
void rn_debug_set_affine_config(int mt, int stages);
/* dense kernel generation: 1 = first, 3 = warp-specialised + Horner epilogue, 4 = chained-DMMA epilogue */
void rn_debug_set_dense_config(int version, int variant);  /* variant (generation 4): bit 0 = one-DADD wrap with a branch in the producers, bit 1 = DOF padding computed, bits 4-7 = ring slots (4..7, 0 = automatic) */
/* local 16-frame tiles that phase 0 / 1 of rn_calc_polarizabilities_routed_phase evaluates, in launch order (host only) */
int64_t rn_debug_phase_tiles(int64_t num_frames, int64_t first_frame, int64_t stripe, int phase, int64_t* tiles,
                             int64_t capacity);
/* unit-balanced dense schedule: 0 = never, 1 = automatic, 2 = always */
void rn_debug_set_dense_split(int mode);
/* mask sweeps: fused sweep kernels on/off; shortest run of linear models worth fusing (2..4) */
void rn_debug_set_sweep_fused(int on);
void rn_debug_set_sweep_min_run(int run);
/* memberships per chunk of rn_van_hove (whole member tiles, at least one; 0 = automatic) */
void rn_debug_set_van_hove_chunk(int memberships);
/* FFT core of the spectrum path (csrc/rn_fft.cuh), single-GPU plans: forward transform of 2^info[2]
 * complex values left in the transform's own digit-reversed order, and IFFT(FFT(in) * H) (unnormalised,
 * natural order) with H the plan's chirp filter spectrum.  d_out must not alias d_in. */
int rn_debug_fft_forward(rn_spectrum_plan* plan, const double* d_in, double* d_out, void* stream);
int rn_debug_fft_convolve(rn_spectrum_plan* plan, const double* d_in, double* d_out, void* stream);

#ifdef __cplusplus
}
#endif

#endif /* RAMANNOODLE_B200_DEBUG_H */
