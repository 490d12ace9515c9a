/*
 * ramannoodle_b200 — C-ABI of the B200 (sm_100a) MD-Raman hot path.
 *
 * The reference (wolearyc/ramannoodle v0.5.0) is pure Python and has no FFI; its plugin
 * boundary is three ABCs plus one free function (ramannoodle/abstract.py:10-83,
 * ramannoodle/spectrum/utils.py:12-18).  Each entry point below names the reference
 * interface it replaces (file:line relative to the reference tree).  The reference-side
 * binding a maintainer would add (a ctypes stub) is shown in INTEGRATION.md.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / numpy types cross this boundary;
 *   - all arithmetic is IEEE fp64; arrays are C-contiguous (row-major);
 *   - `d_` pointers are device pointers on the model's / plan's device, `h_` are host;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); device
 *     entry points enqueue work and return without synchronising;
 *   - every function returns RN_OK (0) or a negative rn_status; the message of the last
 *     failure on the calling thread is available from rn_last_error().
 */
#ifndef RAMANNOODLE_B200_H
#define RAMANNOODLE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum rn_status {
    RN_OK = 0,
    RN_ERR_INVALID_ARGUMENT = -1,
    RN_ERR_CUDA = -2,
    RN_ERR_UNSUPPORTED = -3,
    RN_ERR_OUT_OF_MEMORY = -4
} rn_status;

/* Flags for rn_model_create. */
#define RN_MODEL_DEFAULT 0
/* Evaluate every DOF through the dense DMMA projection + spline epilogue, even DOFs whose
 * interpolant is a single linear piece (disables the affine collapse; used to benchmark
 * and cross-check the dense path on ARTModels). */
#define RN_MODEL_FORCE_DENSE 1

typedef struct rn_model rn_model;
typedef struct rn_spectrum_plan rn_spectrum_plan;

/* Human-readable message of the last error raised on this thread ("" if none). */
const char* rn_last_error(void);

/* Library / device probe: writes the CUDA runtime version, the device count and the
 * compute capability (major*10+minor) of `device`.  Used by the loader to fail loudly. */
int rn_device_info(int device, int* runtime_version, int* device_count, int* compute_capability,
                   int* sm_count);

/* ------------------------------------------------------------------------------------
 * Polarizability model — replaces InterpolationModel / ARTModel evaluation state
 * (ramannoodle/pmodel/_interpolation.py:110-115; ARTModel inherits, pmodel/_art.py:48).
 *
 *   h_ref_positions  (N,3)  fractional positions of the ReferenceStructure
 *   h_lattice        (3,3)  rows are lattice vectors (Å)   (structure/_reference.py:285)
 *   h_basis          (J,3N) Cartesian basis vectors, one row per DOF (_cart_basis_vectors)
 *   h_degree         (J,)   B-spline degree k_j of DOF j    (_interpolations[j].k)
 *   h_knot_off       (J+1,) knots of DOF j are h_knots[h_knot_off[j] .. h_knot_off[j+1])
 *   h_coef_off       (J+1,) coefficients of DOF j are rows h_coef_off[j] .. h_coef_off[j+1]
 *                           of h_coefs, an (sum n_j, 9) array (c reshaped (n_j,3,3)->(n_j,9))
 *   h_weight         (J,)   1 - mask_j                      (_interpolation.py:242)
 *   h_ref_polarizability (3,3)
 * Splines use extrapolate=True semantics (scipy BSpline as called at _interpolation.py:243).
 * ------------------------------------------------------------------------------------ */
int rn_model_create(const double* h_ref_positions, int64_t num_atoms, const double* h_lattice,
                    const double* h_basis, int64_t num_dofs, const int32_t* h_degree,
                    const int64_t* h_knot_off, const double* h_knots, const int64_t* h_coef_off,
                    const double* h_coefs, const double* h_weight,
                    const double* h_ref_polarizability, int device, int flags, rn_model** out);
int rn_model_destroy(rn_model* model);

/* info[0]=num_atoms, [1]=num_dofs, [2]=DOFs folded into the affine term, [3]=DOFs evaluated by
 * the dense path, [4]=max spline degree on the dense path, [5]=device, [6]=1 if the TMA
 * affine kernel is eligible for this model size, [7]=max pieces of any dense-path DOF. */
int rn_model_info(const rn_model* model, int64_t info[8]);

/* PolarizabilityModel.calc_polarizabilities(positions_batch)  (abstract.py:13-29;
 * _interpolation.py:191-252): d_positions (S,N,3) fractional -> d_alpha (S,3,3). */
int rn_calc_polarizabilities(const rn_model* model, const double* d_positions, int64_t num_frames,
                             double* d_alpha, void* stream);

/* The "displacements already computed" entry BASELINE.json's north_star names
 * (pmodel.get_polarizability(cart_displacements)): d_cart_displacements (S,3N) in Å as
 * produced at _interpolation.py:217-223 -> d_alpha (S,3,3)  (= _interpolation.py:233-252). */
int rn_get_polarizability(const rn_model* model, const double* d_cart_displacements,
                          int64_t num_frames, double* d_alpha, void* stream);

/* Host-buffer form of rn_calc_polarizabilities: streams h_positions to the device in
 * chunks (copies overlapped with evaluation).  The result is written to h_alpha (host,
 * may be NULL) and/or d_alpha (device, may be NULL); at least one must be given.
 * Synchronous.  Pinned (page-locked) host buffers give full PCIe bandwidth; see
 * rn_host_register.  chunk_frames <= 0 picks ~64 MiB chunks. */
int rn_calc_polarizabilities_host(const rn_model* model, const double* h_positions,
                                  int64_t num_frames, double* h_alpha, double* d_alpha,
                                  int64_t chunk_frames);

/* Multi-destination forms for frame-sharded multi-GPU runs: the evaluated rows are stored to
 * every pointer of d_alpha_outputs (num_outputs in 1..8).  outputs[0] is the local series, the
 * others are the same buffer on peer GPUs (peer-mapped device memory, e.g. symmetric memory over
 * NVLink); all pointers are pre-offset to this rank's first frame.  The hot kernels write the
 * peers' rows themselves (ld/st.global on mapped peer pointers): the all-gather of the
 * (S,3,3) series is fused into the evaluation.  The caller synchronises the ranks afterwards. */
int rn_calc_polarizabilities_multi(const rn_model* model, const double* d_positions,
                                   int64_t num_frames, double* const* d_alpha_outputs,
                                   int num_outputs, void* stream);
int rn_calc_polarizabilities_host_multi(const rn_model* model, const double* h_positions,
                                        int64_t num_frames, double* const* d_alpha_outputs,
                                        int num_outputs, int64_t chunk_frames, void* stream);

/* Routed form for the shared multi-GPU spectrum (rn_spectrum_dist_*): the rows are stored to
 * d_alpha (this rank's block inside its own full (S,3,3) series buffer, i.e. buffer + first_frame*9)
 * and, by the kernels themselves over NVLink, to the series buffers of the ranks whose spectrum
 * stage consumes them: row n = first_frame + local row goes to owner(n) and owner(n-1) with
 * owner(n) = (n mod period) / width  (rn_spectrum_dist_route).  peer_series[r] is the BASE of rank r's
 * full series buffer (peer-mapped); NULL for this rank itself and for ranks that own nothing.
 * The host form streams h_positions like rn_calc_polarizabilities_host; its private streams start
 * after the work already enqueued on `stream` (e.g. a cross-rank barrier) and it returns when done. */
int rn_calc_polarizabilities_routed(const rn_model* model, const double* d_positions,
                                    int64_t num_frames, double* d_alpha, double* const* peer_series,
                                    int world, int64_t first_frame, int64_t period, int64_t width,
                                    void* stream);
int rn_calc_polarizabilities_host_routed(const rn_model* model, const double* h_positions,
                                         int64_t num_frames, double* d_alpha,
                                         double* const* peer_series, int world, int64_t first_frame,
                                         int64_t period, int64_t width, int64_t chunk_frames,
                                         void* stream);
/* The routed evaluation in two phases, for a schedule that overlaps the spectrum stage's (NVLink-bound)
 * pack with the (HBM-bound) evaluation: phase 0 evaluates the frames n with (n mod 2*stripe) < stripe + 16
 * — every row the packs of phase 0 read (rn_spectrum_dist_pack, rn_spectrum_dist_stripe) — phase 1 the
 * others; each phase is ONE launch whose tiles map onto the selected frames.  Needs the TMA affine path
 * (a purely linear model, 16-byte aligned rows) and blocks that start and end on multiples of 16 frames:
 * rn_routed_phases_supported() says whether a model / block qualifies (else RN_ERR_UNSUPPORTED). */
int rn_routed_phases_supported(const rn_model* model, const double* d_positions, int64_t num_frames,
                               int64_t first_frame, int64_t stripe);
int rn_calc_polarizabilities_routed_phase(const rn_model* model, const double* d_positions,
                                          int64_t num_frames, double* d_alpha,
                                          double* const* peer_series, int world, int64_t first_frame,
                                          int64_t period, int64_t width, int64_t stripe, int phase,
                                          void* stream);

/* Mask sweeps (SURVEY.md §8f N3): num_models models of ONE structure — in practice the
 * get_masked_model copies of a model (pmodel/_interpolation.py:697-708; ARTModel.get_dof_indexes,
 * pmodel/_art.py:335-365), which differ only in `weight` — evaluated on the same positions;
 * d_alpha_outputs[g] (num_frames*9 doubles, device) receives exactly what
 * rn_calc_polarizabilities(models[g], ...) writes.  Runs of up to four purely linear models
 * (every ARTModel) share one kernel: the trajectory is read and wrapped once and contracted with
 * the stacked (3N x 9G) table.  The host form streams h_positions across PCIe once for all models. */
int rn_calc_polarizabilities_sweep(const rn_model* const* models, int num_models,
                                   const double* d_positions, int64_t num_frames,
                                   double* const* d_alpha_outputs, void* stream);
int rn_calc_polarizabilities_host_sweep(const rn_model* const* models, int num_models,
                                        const double* h_positions, int64_t num_frames,
                                        double* const* d_alpha_outputs, int64_t chunk_frames);
/* Routed mask sweep for the shared multi-GPU spectrum: d_alpha_outputs[g] receives what
 * rn_calc_polarizabilities_sweep writes (this rank's block of mask g's series; spline models always take the
 * whole-tile schedule here, so short blocks may differ from the plain sweep's unit-balanced one in the last
 * bits), and row n of mask g is
 * also stored to peer_series[g*world + r] for r = owner(n) and r = owner(n-1) — the rule of
 * rn_calc_polarizabilities_routed, one row of `world` base pointers per mask (NULL for this rank and
 * for ranks that own nothing).  The host form sends each chunk across PCIe once for all masks; its
 * private streams start after the work already enqueued on `stream` and it returns when done. */
int rn_calc_polarizabilities_sweep_routed(const rn_model* const* models, int num_models,
                                          const double* d_positions, int64_t num_frames,
                                          double* const* d_alpha_outputs, double* const* peer_series,
                                          int world, int64_t first_frame, int64_t period, int64_t width,
                                          void* stream);
int rn_calc_polarizabilities_host_sweep_routed(const rn_model* const* models, int num_models,
                                               const double* h_positions, int64_t num_frames,
                                               double* const* d_alpha_outputs,
                                               double* const* peer_series, int world,
                                               int64_t first_frame, int64_t period, int64_t width,
                                               int64_t chunk_frames, void* stream);

/* Trajectory.__init__ stores apply_pbc(positions_ts) (dynamics/_trajectory.py:45;
 * structure/utils.py:27: p - p // 1).  Elementwise, in place allowed (d_out == d_in). */
int rn_apply_pbc(const double* d_in, double* d_out, int64_t count, void* stream);


/* ------------------------------------------------------------------------------------
 * MD Raman spectrum — replaces MDRamanSpectrum.measure (spectrum/_raman.py:241-309) with
 * calc_signal_spectrum (spectrum/utils.py:95-124) evaluated through the identity
 *   Re FFT_M(autocorr+(x))[k] = (|FFT_M(x)[k]|^2 + sum x^2) / 2,  M = S - 1,
 * using an arbitrary-length (Bluestein) FFT written for this library (in-place DIF/DIT convolution,
 * csrc/rn_fft.cuh).  A plan owns the tables and work buffers for one series length S on one device;
 * calls on one plan must not overlap (one stream at a time).
 * ------------------------------------------------------------------------------------ */
int rn_spectrum_plan_create(int64_t num_frames, int device, rn_spectrum_plan** out);
int rn_spectrum_plan_destroy(rn_spectrum_plan* plan);
/* Number of output points: ceil((S-1)/2) - 1  (the 0 cm^-1 bin is dropped, _raman.py:299-301). */
int64_t rn_spectrum_num_points(int64_t num_frames);
/* d_alpha (S,3,3) -> d_wavenumbers (P,), d_intensities (P,), P = rn_spectrum_num_points(S).
 * laser_correction / bose_einstein_correction follow _raman.py:13-69,303-307. */
int rn_md_spectrum(rn_spectrum_plan* plan, const double* d_alpha, double timestep_fs,
                   int laser_correction, double laser_wavelength_nm, int bose_einstein_correction,
                   double temperature_K, double* d_wavenumbers, double* d_intensities, void* stream);
/* Windowed spectra (no reference counterpart; each row is rn_md_spectrum of one slice).
 * rn_spectrum_plan_create_batched: a single-GPU plan for windows of window_frames frames whose work,
 * power, energy-partial and ticket buffers hold `batch` windows (1 .. 65535; batch = 1 is
 * rn_spectrum_plan_create).  rn_md_spectrum also accepts such a plan.
 * rn_md_spectrum_windows: d_alpha (num_frames,3,3) -> d_wavenumbers (P,), d_intensities (W,P) with
 * P = rn_spectrum_num_points(window_frames), W = 1 + (num_frames - window_frames) / hop_frames;
 * row w is rn_md_spectrum of frames [w hop_frames, w hop_frames + window_frames).  Trailing frames
 * that fill no window are not read.  The windows run in chunks of `batch` on `stream`. */
int rn_spectrum_plan_create_batched(int64_t window_frames, int64_t batch, int device, rn_spectrum_plan** out);
int rn_md_spectrum_windows(rn_spectrum_plan* plan, const double* d_alpha, int64_t num_frames, int64_t hop_frames,
                           double timestep_fs, int laser_correction, double laser_wavelength_nm,
                           int bose_einstein_correction, double temperature_K, double* d_wavenumbers,
                           double* d_intensities, void* stream);
/* Cross spectra of G series (extends _raman.py:241-309 and spectrum/utils.py:95-124; no reference
 * counterpart).  d_alpha is a contiguous (G,S,3,3) array, plan a single-GPU plan of S frames whose batch
 * is at least G (rn_spectrum_plan_create_batched(S, G, ...)).  -> d_wavenumbers (P,), d_intensities
 * (G,G,P), P = rn_spectrum_num_points(S).  Row (g,h) is _raman.py:241-309 with every
 * calc_signal_spectrum(sig) replaced by the spectrum of the symmetrised cross-correlation
 * (correlate(sig_g, sig_h) + correlate(sig_h, sig_g)) / 2 of the same signals: symmetric in g and h,
 * bilinear in the series, and row (g,g) is bit-identical to rn_md_spectrum of series g.  For series whose
 * differences add up to those of a total series, the G x G rows add up to its spectrum.  The plan keeps
 * G(G-1)/2 * (ceil((S-1)/256) + 1) doubles of energy partials between calls. */
int rn_md_cross_spectra(rn_spectrum_plan* plan, const double* d_alpha, int64_t num_series, double timestep_fs,
                        int laser_correction, double laser_wavelength_nm, int bose_einstein_correction,
                        double temperature_K, double* d_wavenumbers, double* d_intensities, void* stream);
/* Vibrational density of states of G atom groups (no reference counterpart).  d_positions is a contiguous
 * (S,N,3) array of fractional positions, plan a single-GPU plan of S frames (rn_spectrum_plan_create or
 * rn_spectrum_plan_create_batched); h_lattice the (3,3) lattice in Angstrom, rows are lattice vectors;
 * h_weights (N,) finite and >= 0, NULL = all 1; group g is the atoms h_atoms[h_group_offsets[g] ..
 * h_group_offsets[g+1]-1] (CSR, non-empty, indices in [0, N)).  -> d_wavenumbers (P,), d_intensities (G,P),
 * P = rn_spectrum_num_points(S): row g is sum over its atoms i and c = x, y, z of
 * w_i calc_signal_spectrum(v_ic, timestep)[1:] (spectrum/utils.py:95-124) with the minimum-image velocity
 * v = (wrap(x[n+1] - x[n]) @ lattice) / timestep in Angstrom/fs; the wavenumbers are those of rn_md_spectrum.
 * Two memberships of a group form a slot; slots run in chunks of the plan's batch (one pack, the transform
 * and one combine per chunk) and the result is bit-identical for every batch.  The plan keeps the slot
 * table (24 bytes per slot plus 8 (G+1)) between calls.  P = 0 launches nothing. */
int rn_vdos(rn_spectrum_plan* plan, const double* d_positions, int64_t num_atoms, const double* h_lattice,
            const double* h_weights, const int64_t* h_group_offsets, const int64_t* h_atoms, int64_t num_groups,
            double timestep_fs, double* d_wavenumbers, double* d_intensities, void* stream);
/* One transform shared by the ranks of a multi-GPU run (one process per GPU; no reference
 * counterpart — same result as rn_md_spectrum on the whole series).  The chirp-z transform of
 * length L is decimated in frequency over the G = 2, 4 or 8 ranks of the group (the largest power
 * of two <= world; further ranks only receive the result):
 *   1. the evaluation kernels store every series row n to the rank whose block of n' = n mod (L/G)
 *      contains it (rn_spectrum_dist_route: owner(n) = (n mod period) / width; a rank also needs row
 *      n+1 of its last n) — rn_calc_polarizabilities_routed;
 *   2. rn_spectrum_dist_pack: np.diff, signal packing, chirp pre-multiply, G-point DFT over the blocks
 *      and twiddle for this rank's n'; residue r is stored into peer_work[r] (rank r's work buffer);
 *   3. rn_spectrum_dist_transform: the local length-L/G convolution with this rank's decimated
 *      filter, in place in d_work; its last pass stores every value to the rank that owns that m'
 *      (peer_recv[owner]).  Ownership of m' is mirror-symmetric about (M mod L/G) / 2, so that the owner
 *      of bin m also owns bin M - m;
 *   4. rn_spectrum_dist_final: the G-point inverse DFT over the residues for this rank's pairs of m',
 *      I[k] = (P[k] + P[M-k]) / (4 L^2) + E/2 with P[m] = sum_p |y_p[m]|^2 and the optional corrections,
 *      stored to every destination's spectrum buffer (half the bytes of P, and nothing left to combine);
 *      the wavenumbers are written locally (d_wavenumbers, may be NULL);
 *   5. rn_spectrum_dist_finish (every rank): copies the finished intensities out of the spectrum buffer
 *      (and writes the wavenumbers if d_wavenumbers is given: ranks that did not run step 4) — together
 *      exactly what rn_md_spectrum returns.
 * The caller separates the steps with a cross-rank barrier (the buffers are peer-mapped device memory,
 * e.g. symmetric memory over NVLink) and provides, per rank, a work buffer, a receive buffer and a
 * spectrum buffer of rn_spectrum_dist_sizes bytes (the spectrum buffer starts with 16 doubles: the series
 * energy shares of the ranks and pack phases, stored to every destination by step 2).  All ranks of the world call every
 * step; for spectator ranks (rank >= G) steps 2-4 return immediately.  Steps 2 and 3 take `seq`: -1
 * handles the three packed sequences in one go; 0, 1, 2 handle one sequence, so that a caller can
 * pipeline them on several streams (the NVLink-bound stores of one sequence overlap the transform of
 * another; the pass with seq = 0 also sums the series energies, and must be among the passes). */
int rn_spectrum_plan_create_dist(int64_t num_frames, int device, int world, int rank,
                                 rn_spectrum_plan** out);
/* info[0]=log2 L, [1]=ranks sharing the transform, [2]=log2 of the local length, [3]=strided levels,
 * [4],[5]=log2 of their radices, [6]=block of n' / m' one rank owns, [7]=M. */
int rn_spectrum_plan_info(const rn_spectrum_plan* plan, int64_t info[8]);
int rn_spectrum_dist_sizes(const rn_spectrum_plan* plan, int64_t* work_bytes, int64_t* recv_bytes,
                           int64_t* spectrum_bytes);
int rn_spectrum_dist_route(const rn_spectrum_plan* plan, int64_t* period, int64_t* width);
/* phase: -1 packs the rank's whole block of n'; 0 / 1 pack the first / second half (rn_spectrum_dist_stripe
 * elements each) — phase 0 reads only rows that rn_calc_polarizabilities_routed_phase(..., phase 0) stores, so
 * it can run (on a second stream) while phase 1 of the evaluation is still streaming frames. */
int rn_spectrum_dist_stripe(const rn_spectrum_plan* plan, int64_t* stripe);
int rn_spectrum_dist_pack(rn_spectrum_plan* plan, const double* d_series, double* const* peer_work,
                          double* const* dest_spectrum, int num_dest, int seq, int phase, void* stream);
int rn_spectrum_dist_transform(rn_spectrum_plan* plan, double* d_work, double* const* peer_recv,
                               int seq, void* stream);
int rn_spectrum_dist_final(rn_spectrum_plan* plan, const double* d_recv, const double* d_spectrum,
                           double* const* dest_spectrum, int num_dest, double timestep_fs,
                           int laser_correction, double laser_wavelength_nm,
                           int bose_einstein_correction, double temperature_K,
                           double* d_wavenumbers, void* stream);
int rn_spectrum_dist_finish(const rn_spectrum_plan* plan, const double* d_spectrum, double timestep_fs,
                            double* d_wavenumbers, double* d_intensities, void* stream);
/* calc_signal_spectrum(signal, sampling_rate) (spectrum/utils.py:95-124) for one real signal of
 * length M = S-1 of the plan: outputs ceil(M/2) points (bin 0 included). */
int rn_signal_spectrum(rn_spectrum_plan* plan, const double* d_signal, double sampling_rate,
                       double* d_wavenumbers, double* d_intensities, void* stream);

/* convolve_spectrum (spectrum/utils.py:12-73): kind 0 = gaussian, 1 = lorentzian.
 * d_workspace must hold rn_convolve_workspace_size(K, L) bytes (may be NULL if that is 0). */
size_t rn_convolve_workspace_size(int64_t num_in, int64_t num_out);
int rn_convolve_spectrum(const double* d_wavenumbers, const double* d_intensities, int64_t num_in,
                         int kind, double width, const double* d_out_wavenumbers, int64_t num_out,
                         double* d_out_intensities, void* d_workspace, void* stream);
/* convolve_spectrum (spectrum/utils.py:12-73) of num_rows rows that share one input and one output grid:
 * d_intensities (B,K) row-major -> d_out_intensities (B,L).  Row b is bit-identical to rn_convolve_spectrum
 * of row b.  Two launches whatever B is.  d_workspace must hold rn_convolve_spectra_workspace_size(B, K, L)
 * bytes.  num_rows == 0 or num_out == 0: nothing is launched; num_in == 0: one memset of the output;
 * num_rows == 1 runs the kernels of rn_convolve_spectrum. */
size_t rn_convolve_spectra_workspace_size(int64_t num_rows, int64_t num_in, int64_t num_out);
int rn_convolve_spectra(const double* d_wavenumbers, const double* d_intensities, int64_t num_rows, int64_t num_in,
                        int kind, double width, const double* d_out_wavenumbers, int64_t num_out,
                        double* d_out_intensities, void* d_workspace, void* stream);

/* Trajectory ingest — replaces the Python text parsing of io.vasp.xdatcar.read_positions_ts
 * (ramannoodle/io/vasp/xdatcar.py:21-56; header/frames as io/vasp/poscar.py:_read_lattice,
 * _read_atomic_symbols, _read_positions).  Host-only (no GPU needed): mmap + a thread pool
 * running a correctly rounded decimal parser (values equal Python's float(token)).
 * rn_xdatcar_scan returns the frame count, atom count and the scaled lattice (9 doubles, may
 * be NULL); rn_xdatcar_read fills h_positions (S,N,3) — e.g. a pinned buffer — with the
 * fractional coordinates as written, or wrapped into [0,1) like Trajectory.__init__
 * (dynamics/trajectory.py:58) when wrap != 0 (num_threads <= 0: all cores).
 * Direct-coordinate frames only. */
int rn_xdatcar_scan(const char* path, int64_t* num_frames, int64_t* num_atoms, double* lattice);
int rn_xdatcar_read(const char* path, double* h_positions, int64_t num_frames, int64_t num_atoms,
                    int num_threads, int wrap);

/* OUTCAR molecular-dynamics trajectories — replaces the line-by-line Python parsing of
 * io.vasp.outcar.read_trajectory (ramannoodle/io/vasp/outcar.py:497-538; header fields as
 * :46-86 atom count, :481-494 timestep, :212-241 lattice; ML/ab-initio step rule :520-527).
 * rn_outcar_scan returns the number of kept frames, the atom count, the lattice (9 doubles, rows are
 * lattice vectors, may be NULL) and the timestep in fs (may be NULL).  rn_outcar_read fills
 * h_positions (S,N,3): the Cartesian coordinates as written when inv_lattice is NULL, else
 * cart @ inv_lattice (row-major 3x3, the reference's np.linalg.inv(lattice)), wrapped into [0,1)
 * when wrap != 0.  Host-only. */
int rn_outcar_scan(const char* path, int64_t* num_frames, int64_t* num_atoms, double* lattice,
                   double* timestep_fs);
int rn_outcar_read(const char* path, double* h_positions, int64_t num_frames, int64_t num_atoms,
                   const double* inv_lattice, int num_threads, int wrap);

/* vasprun.xml molecular-dynamics trajectories (ramannoodle/io/vasp/vasprun.py:298-330, _parse_positions
 * :53-70, _parse_timestep :281-295): every unnamed `structure` element directly under the root is a frame
 * (rows of its first `varray`), POTIM is the timestep.  Host-only, same pattern as the XDATCAR reader:
 * scan (frame / atom counts, timestep in fs), then read into a (num_frames, num_atoms, 3) buffer.
 * RN_ERR_INVALID_ARGUMENT: what the reference reports as InvalidFileException; RN_ERR_UNSUPPORTED: markup
 * the tokenizer does not handle — the caller re-reads the file with a full XML parser. */
int rn_vasprun_scan(const char* path, int64_t* num_frames, int64_t* num_atoms, double* timestep_fs);
int rn_vasprun_read(const char* path, double* h_positions, int64_t num_frames, int64_t num_atoms,
                    int num_threads, int wrap);

/* Host-side Trajectory.__init__ wrap (dynamics/_trajectory.py:45; structure/utils.py:27:
 * positions - positions // 1) with a thread pool: h_out[i] = h_in[i] - floor(h_in[i]), identical to
 * numpy's result; h_out may be pinned memory, in place allowed.  num_threads <= 0: all cores. */
int rn_host_apply_pbc(const double* h_in, double* h_out, int64_t count, int num_threads);

/* Page-lock / unlock a caller-owned host buffer (cudaHostRegister) for fast transfers. */
int rn_host_register(void* h_ptr, size_t bytes);
int rn_host_unregister(void* h_ptr);

/* Host-only helper (no GPU needed): converts one B-spline (t, c (n,9), k) into the piecewise
 * polynomial table the kernels evaluate.  out_breaks gets the (pieces-1) interior break
 * points, out_x0 the expansion point of each piece and out_coefs (pieces, k+1, 9) the local
 * power-basis coefficients.  Returns the number of pieces, or a negative rn_status.
 * Capacity: out_breaks/out_x0 need n entries, out_coefs n*(k+1)*9. */
int rn_bspline_to_pp(const double* h_knots, int num_knots, const double* h_coefs, int degree,
                     double* out_breaks, double* out_x0, double* out_coefs);

/* Kernel-launch counter (incremented by every kernel this library launches); used by
 * bench.py for its "gpu_launches" claim. */
int64_t rn_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* RAMANNOODLE_B200_H */
