/*
 * professad_b200.h -- C ABI of the B200-native OFDFT hot path (drop-in for PROFESS-AD's
 * energy-functional evaluation and density-optimisation loop).
 *
 * The reference (PROFESS-AD v1.0.1) is pure Python/PyTorch: it has no FFI of its own.  Its
 * "operator interface" for this path is the Python callable contract
 *     f(box_vecs, den) -> scalar energy,   differentiated by torch.autograd        (docs/source/functionals.rst:13-15)
 * plus the optimisation loop in System.optimize_density (src/professad/system.py:774-908).
 * Every entry point below replaces one such callable (energy AND analytic dE/dn in one call) or
 * one stage of that loop; the citation on each says which.  The Python binding a reference
 * maintainer would add (ctypes) is shown in INTEGRATION.md and shipped in
 * profess_ad_b200/_native.py.
 *
 * Conventions
 *   - all arrays are DEVICE pointers to fp64, C-contiguous (n0, n1, n2) grids, N = n0*n1*n2;
 *     `box` is a HOST pointer to the 3x3 row-major lattice (rows = lattice vectors, bohr);
 *   - energies are written to a DEVICE double (Hartree) -- no call synchronises the host;
 *   - `v_out` may be NULL (energy only).  With `accumulate != 0` the call does E += ..., v += ...;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all work is
 *     enqueued on it and the call returns immediately;
 *   - return value 0 = ok, otherwise an error code; pad_last_error() gives the message
 *     (thread-local).  Nothing here falls back to the CPU.
 */
#ifndef PROFESSAD_B200_H
#define PROFESSAD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pad_plan pad_plan;

#define PAD_OK 0
#define PAD_ERR_CUDA 1
#define PAD_ERR_CUFFT 2
#define PAD_ERR_ARG 3
#define PAD_ERR_NCCL 4

/* parts of a Wang-Teter style kinetic functional to include (functionals.py:669-670) */
#define PAD_PART_TF 1
#define PAD_PART_VW 2
#define PAD_PART_NL 4
#define PAD_PART_ALL 7

/* local terms for pad_eval_local */
#define PAD_LOCAL_TF 1          /* ThomasFermi               functionals.py:207-224  */
#define PAD_LOCAL_LDAX 2        /* lda_exchange              functionals.py:1510-1512 */
#define PAD_LOCAL_PZC 4         /* perdew_zunger_correlation functionals.py:1515-1521 */
#define PAD_LOCAL_IONEL 8       /* IonElectron               functionals.py:31-46     */

const char* pad_version(void);
const char* pad_last_error(void);
/* kernels this library has launched so far in this process (own kernels; cuFFT execs counted separately) */
unsigned long long pad_launch_count(void);
unsigned long long pad_fft_exec_count(void);
/* 1 (default): use the hand-written fused FFT pipeline where the grid allows (n2 in 128/256);
 * 0: plain cuFFT 3-D transforms + separate elementwise kernels.  Returns the previous setting. */
int pad_set_fast_fft(int on);
/* tuning switches (process-wide): "fast_fft" (as above), "own_xy" (1: hand-written strided x/y passes with the
 * reciprocal-space multiply fused into the x pass; 0: batched 2-D cuFFT), "pipe" (1: the z and y passes of an x-plane run
 * as items of ONE persistent kernel and hand the plane over through the L2, csrc/zy_pipe.cuh; 0: one kernel per pass),
 * "pipe_lpi" / "pipe_tpi" (lines per z item / tiles per y item, 0: default), "fuse_terms" (1: pad_eval_total evaluates
 * IonElectron / LDA exchange / PZ correlation inside the WGC99 mid pass and Hartree as a fourth field of its second
 * transform batch; 0: one call per term).  Returns the previous value, -1 on error. */
int pad_set_option(const char* name, int value);
/* Live per-stage device timing (CUDA events on the launch stream between the kernels of the fused WGC99
 * pipeline).  pad_profile_begin() switches it on and clears the sums; pad_profile_end() switches it off and
 * returns, for each stage i < *n_out (at most cap), the mean milliseconds per evaluation in ms_out[i] and its
 * name in names_out[i * 48 ...] (NUL-terminated).  Used by bench.py for the dominant-kernel roofline. */
int pad_profile_begin(void);
int pad_profile_end(char* names_out, double* ms_out, int cap, int* n_out, int* evals_out);

/* ---- plan: replaces wavevecs(box_vecs, shape) (functional_tools.py:135-162) and owns the cuFFT
 *      plans, scratch fields and cached reciprocal-space kernels for one (box, shape, device). ---- */
int pad_plan_create(pad_plan** plan, const double* box_host, const int* shape_host, int device);
int pad_plan_destroy(pad_plan* plan);

/* ---- slab plan: one large grid split over `world` ranks (one process per GPU).  Real space is split along
 *      axis 0 (n0 / world planes per rank), the half spectrum along axis 1 (n1 / world rows, all of axis 0);
 *      every 3-D transform is a local batched 2-D (y, z) cuFFT, ONE all-to-all, and a local strided 1-D (x)
 *      cuFFT.  The library does not link a communication library: the caller supplies `fn`, which must, on
 *      `stream`'s device and ordered with `stream`,
 *        op == PAD_COMM_ALL_TO_ALL : exchange send_buf -> recv_buf, `count` complex128 per peer (peer r's block
 *                                    is send_buf[r * count ...]; block r of recv_buf comes from peer r)
 *        op == PAD_COMM_ALL_REDUCE : sum comm_scratch[0 .. count) over the ranks, in place
 *        op == PAD_COMM_ALL_REDUCE_MAX : maximum of comm_scratch[0 .. count) over the ranks, in place
 *      and return 0.  Python binds it to torch.distributed (NCCL over NVLink).  Every functional entry point
 *      below then takes LOCAL slabs (den, v: n0/world x n1 x n2) and returns GLOBAL energies on every rank;
 *      pad_denopt_* keeps each rank's slab of chi, the gradient and the L-BFGS history and all-reduces the
 *      inner products of an iteration in one batch.  The fused FFT pipeline runs on slab plans once
 *      pad_plan_set_slab_fast_buffers has been called. ---- */
#define PAD_COMM_ALL_TO_ALL 0
#define PAD_COMM_ALL_REDUCE 1
#define PAD_COMM_ALL_REDUCE_MAX 2
#define PAD_COMM_ALL_TO_ALL_2 3          /* as PAD_COMM_ALL_TO_ALL, on the second buffer pair (pad_plan_set_overlap_buffers) */
#define PAD_COMM_ALL_TO_ALL_FAST 16      /* + 8 * dst + src: exchange slab_fast buffer `src` -> `dst` (pad_plan_set_slab_fast_buffers),
                                           `count` complex128 per peer */
#define PAD_COMM_SCRATCH 64
typedef int (*pad_comm_fn)(void* user, int op, long long count, void* stream);
int pad_plan_create_slab(pad_plan** plan, const double* box_host, const int* global_shape_host, int device,
                         int rank, int world, void* send_buf, void* recv_buf, double* comm_scratch,
                         pad_comm_fn fn, void* user);
/* Optional second exchange buffer pair (Nk complex each, caller-owned).  With it, batches of transforms inside one
 * evaluation are software-pipelined: the all-to-all of one field is issued on a communication stream of the plan's own
 * (`fn` is then called with THAT stream and op PAD_COMM_ALL_TO_ALL / PAD_COMM_ALL_TO_ALL_2) while the local FFTs of the
 * neighbouring fields run on the caller's stream. */
int pad_plan_set_overlap_buffers(pad_plan* plan, void* send_buf2, void* recv_buf2);
/* Buffers for the fused FFT pipeline on a slab plan (functional_tools.py:381-423 / functionals.py:941-985 on one grid over several
 * GPUs): six caller-owned device buffers of pad_slab_fast_elements(plan) complex128 each -- four spectrum fields and two exchange
 * stagings.  With them (and n0, n1 in {64 ... 512}, n2 in {128, 256, 512}) WangGovindCarter99 and the Wang-Teter family run the
 * hand-written z / y / x passes on the slabs: the y pass stores its rows blocked by destination rank, so the all-to-all (op
 * PAD_COMM_ALL_TO_ALL_FAST + 8 * dst + src, issued on the plan's communication stream field by field while the neighbouring
 * fields' passes run) needs no pack / unpack kernel, and the kernel mix is fused into the x pass of the transposed layout. */
size_t pad_slab_fast_elements(const pad_plan* plan);
/* Same pipeline with the transposition fused into the passes (the B200 / NVSwitch form): base_ptrs[r] is rank r's symmetric
 * allocation of 8 * pad_slab_fast_elements(plan) complex128 -- four spectrum fields in the local layout followed by the same four
 * in the transposed layout -- mapped into THIS process (peer access over NVLink; torch symmetric memory in parallel.py).  The
 * forward y pass then stores every result row straight into the owner rank's transposed buffer and the fused x pass stores its
 * inverse transform straight into the owner ranks' local buffers; the only collective left is a barrier (fn with op
 * PAD_COMM_BARRIER) between producer and consumer passes.  world <= 8. */
#define PAD_COMM_BARRIER 4
#define PAD_COMM_BARRIER_2 5          /* the same on the plan's communication stream (a second signal channel: barriers of the two streams may be in flight together) */
int pad_plan_set_slab_peer_buffers(pad_plan* plan, void* const* base_ptrs, int world);
/* The same idea for the cuFFT slab path (every functional, any grid): recv_ptrs[r] / recv2_ptrs[r] are the addresses, in THIS
 * process, of rank r's recv_buf / second receive buffer (pad_plan_set_overlap_buffers must have been called; both pairs live in
 * symmetric memory).  The pack kernel of a forward transform then stores every element straight into the owner rank's receive
 * buffer, an inverse transform copies its blocks there, and the all-to-all becomes a barrier (op PAD_COMM_BARRIER); consecutive
 * transforms alternate between the two receive buffers, which is what makes one barrier per transform enough. */
int pad_plan_set_slab_peer_recv(pad_plan* plan, void* const* recv_ptrs, void* const* recv2_ptrs, int world);
int pad_plan_set_slab_fast_buffers(pad_plan* plan, void* const* six_buffers);
int pad_plan_set_box(pad_plan* plan, const double* box_host);      /* same grid, new lattice (strain scans) */
/* Repeated pad_eval_wgc99 / pad_eval_total calls with unchanged arguments are captured once and replayed as one CUDA graph (option
 * "graphs"); counters of captures and replays since the library was loaded. */
int pad_graph_stats(unsigned long long* captures, unsigned long long* replays);
size_t pad_plan_workspace_bytes(const pad_plan* plan);

/* ---- single functionals: E (+)= F[n],  v (+)= dF/dn --------------------------------------- */
/* IonElectron / ThomasFermi / lda_exchange / perdew_zunger_correlation in one pass over n.
 * `terms` is a mask of PAD_LOCAL_*; v_ext may be NULL unless PAD_LOCAL_IONEL is set.
 * PerdewZunger (functionals.py:1540-1554) = PAD_LOCAL_LDAX | PAD_LOCAL_PZC. */
int pad_eval_local(pad_plan* plan, const double* den, const double* v_ext, int terms,
                   double* E_out, double* v_out, int accumulate, void* stream);
/* Hartree (functionals.py:49-72) */
int pad_eval_hartree(pad_plan* plan, const double* den, double* E_out, double* v_out, int accumulate, void* stream);
/* Weizsaecker (functionals.py:227-246) */
int pad_eval_weizsaecker(pad_plan* plan, const double* den, double* E_out, double* v_out, int accumulate, void* stream);
/* WangTeter / Perrot / SmargiassiMadden / WangGovindCarter98 and non_local_KEF
 * (functionals.py:644-725): `parts` selects TF, vW and the non-local term. */
int pad_eval_wt(pad_plan* plan, const double* den, double alpha, double beta, int parts,
                double* E_out, double* v_out, int accumulate, void* stream);
/* WangTeterStyleFunctional building blocks (functionals.py:771-782): writes TF, vW, T_NL to
 * E3_out[0..2] and the three potentials to v3_out (3*N doubles, may be NULL). */
int pad_eval_wt_components(pad_plan* plan, const double* den, double alpha, double beta,
                           double* E3_out, double* v3_out, void* stream);
/* WangGovindCarter99.forward (functionals.py:941-985), 14-FFT analytic form; the kernel
 * (generate_kernel, functionals.py:845-939) is built on the device and cached in the plan. */
int pad_eval_wgc99(pad_plan* plan, const double* den, double alpha, double beta, double gamma, double kappa,
                   double* E_out, double* v_out, int accumulate, void* stream);
/* PerdewBurkeErnzerhof (functionals.py:1597-1635); `which`: 1 = exchange, 2 = correlation, 3 = both */
int pad_eval_pbe(pad_plan* plan, const double* den, int which, double* E_out, double* v_out, int accumulate, void* stream);
/* Semilocal kinetic functionals T = int C_TF n^(5/3) F(p, q), p = s^2, q the reduced Laplacian (functional_tools.py:122-135):
 *   PAD_SEMILOCAL_LKT  LuoKarasievTrickey (functionals.py:309):  F = 1/cosh(p0 s) + (5/3) p            (a = p0 = 1.3)
 *   PAD_SEMILOCAL_PG   PauliGaussian      (functionals.py:336):  F = (5/3) p + exp(-p0 p) + p1 q^2     (mu = 40/27, beta = 0.25)
 * Potential e_n - div(2 e_sigma grad n) + lap(e_L) from one gradient (and Laplacian) and one divergence round trip. */
#define PAD_SEMILOCAL_LKT 0
#define PAD_SEMILOCAL_PG 1
int pad_eval_semilocal_kinetic(pad_plan* plan, const double* den, int variant, double p0, double p1, double* E_out, double* v_out,
                               int accumulate, void* stream);

/* HuangCarter.forward (variant 0: p0 = lambda) / RevisedHuangCarter.forward (variant 1: p0 = a, p1 = b)
 * (functionals.py:1232-1269, 1331-1365) with field_dependent_convolution + interpolate_kernel +
 * interpolate (functional_tools.py:292-423) fused into node-wise convolutions and a per-voxel
 * 4-node Hermite gather.  table_dev: DEVICE pointer to 2*n_eta doubles [eta | omega(eta)], eta uniform
 * from 0.  geometric != 0 selects the geometric node progression (what HC/revHC use), else arithmetic.
 * Does one device->host read (min/max of xi), as the reference does.  n_nodes_out (host, may be NULL). */
int pad_eval_hc(pad_plan* plan, const double* den, int variant, double p0, double p1, double beta, double kappa,
                int geometric, const double* table_dev, int n_eta, double* E_out, double* v_out, int accumulate,
                int* n_nodes_out, void* stream);

/* ---- spectral tools (functional_tools.py:166-227) ------------------------------------------ */
int pad_gradient(pad_plan* plan, const double* f, double* gx, double* gy, double* gz, void* stream);
int pad_laplacian(pad_plan* plan, const double* f, double* out, void* stream);

/* ---- hand-written 3-D real FFT (z passes own, (x,y) batched cuFFT) over the padded half-spectrum layout
 *      (n0, n1, nzp = n2/2 + 8) complex; unnormalised like cuFFT.  Exposed for tests and profiling. -------- */
int pad_fast_fft_supported(const pad_plan* plan);
int pad_rfft3_fast(pad_plan* plan, const double* in, double* out_cplx_padded, int* nzp_out, void* stream);
int pad_irfft3_fast(pad_plan* plan, double* in_cplx_padded /* destroyed */, double* out, void* stream);
/* one strided pass on its own: in-place complex FFT of a padded half-spectrum along axis 0 or 1 (length 64/128/256),
 * dir = -1 forward, +1 inverse, unnormalised (torch.fft.fft / ifft * n along that axis) */
int pad_fft_axis_fast(pad_plan* plan, double* cplx_padded, int axis, int dir, void* stream);
/* 1 if the software-pipelined (z, y) kernels serve this plan's shape (and the "pipe" option is on), else 0 */
int pad_pipe_supported(const pad_plan* plan);
/* synchronises `stream` and returns the watchdog word of the pipelined kernels' control block: 0 = every launch on this
 * plan ran to completion, 1 = a CTA gave up waiting for work (the results are then invalid); -1: no pipelined launch yet */
int pad_pipe_status(pad_plan* plan, void* stream);
/* test hook: the table-driven pow / sqrt / reciprocal of csrc/fastmath.cuh next to the CUDA library results */
int pad_dbg_fastmath(const double* x, size_t n, double e, double* out3n, double* ref3n, void* stream);

/* ---- ionic potential and ion-electron forces: replaces System.__potential_from_ions (system.py:183-205) ->
 *      interpolate_recpot (ion_utils.py:49-81) -> lattice_sum (ion_utils.py:88-118) -> structure_factor
 *      (ion_utils.py:121-137), and the IonElectron part of System.__compute_forces (system.py:913-925).
 *      Exact structure factor, O(N_k N_ion) complex multiply-adds from per-ion 1-D phase tables; no N_k x N_ion
 *      temporary.  Works on slab plans (v_ext_out is then the local slab; forces_out holds this rank's PARTIAL
 *      sums, which the caller adds over the ranks). ---- */
typedef struct pad_species {
    const double* table_dev;   /* DEVICE, 2 * n_table doubles [k | v(k)]: k uniform from 0 to k_max (1/bohr), v the
                                  tabulated local pseudopotential (Ha bohr^3) with the Coulomb tail -4 pi z / k^2
                                  ADDED BACK (the smooth part the reference interpolates, ion_utils.py:62-66)      */
    int n_table;
    double k_max;
    double z;                  /* ion charge: the tail is removed again after the interpolation                  */
    const double* frac_dev;    /* DEVICE, n_ions x 3 fractional coordinates                                      */
    int n_ions;
} pad_species;
/* v_ext(r) = irfftn(sum_s v_s(|k|) S_s(k)) / vol over the plan's grid; v_ext_out: N doubles */
int pad_ionic_potential(pad_plan* plan, const pad_species* species, int n_species, double* v_ext_out, void* stream);
/* Particle-mesh Ewald variants (System(pme_order=n), system.py:183-205 -> structure_factor_spline, ion_utils.py:218-286):
 * B-spline spreading + one r2c + exponential-spline factors instead of the O(N_k N_ion) exact structure factor.  order: even,
 * 2..32.  On slab plans every rank sweeps all ions and keeps the stencil points on its own planes (frac_dev holds ALL ions on
 * every rank; forces come out as per-rank partial sums).  pad_pme_structure_factor returns S(k) itself (n0 x n1 x (n2/2+1) complex), the quantity the
 * reference's tests/test_particle_mesh_ewald.py:46-63 compares with the exact structure factor. */
int pad_ionic_potential_pme(pad_plan* plan, const pad_species* species, int n_species, int order, double* v_ext_out, void* stream);
int pad_pme_structure_factor(pad_plan* plan, const double* frac_dev, int n_ions, int order, double* S_out_cplx, void* stream);
/* Forces and stress of the IonElectron term WITH the particle-mesh structure factor: what the reference's autograd gives when
 * pme_order is set (system.py:913-935 through structure_factor_spline).  Forces: one r2c of the density, per species one k-space
 * pass, one c2r and a gather of the B-spline derivative weights over every ion's order^3 stencil -- O(N log N + N_ion order^3);
 * stress: pad_ion_stress with S(k) taken from the mesh (fixed fractional coordinates: S does not depend on the cell). */
int pad_ion_forces_pme(pad_plan* plan, const pad_species* species, int n_species, int order, const double* den,
                       double* forces_out, void* stream);
int pad_ion_stress_pme(pad_plan* plan, const pad_species* species, int n_species, int order, const double* den,
                       double* stress_out, int accumulate, void* stream);
/* F_I = -d/dR_I of IonElectron(den, v_ext[R]) at fixed density, Cartesian, Ha/bohr; forces_out: DEVICE,
 * 3 * (total number of ions) doubles in species order */
int pad_ion_forces(pad_plan* plan, const pad_species* species, int n_species, const double* den, double* forces_out,
                   void* stream);

/* IonElectron part of the stress (system.py:927-935) at fixed fractional coordinates and electron number;
 * stress_out: DEVICE, 9 doubles (row-major symmetric 3 x 3, Ha/bohr^3), overwritten unless accumulate != 0 */
int pad_ion_stress(pad_plan* plan, const pad_species* species, int n_species, const double* den, double* stress_out,
                   int accumulate, void* stream);

/* ---- fused evaluation of a whole term list: replaces System.__compute_energy + autograd
 *      (system.py:759-772, 830-838).  E_out = sum of terms, v_out = total dE/dn. ---------------- */
typedef struct pad_terms {
    int local_mask;      /* PAD_LOCAL_* bits (IonElectron needs v_ext)                       */
    int hartree;         /* 0/1                                                              */
    int kinetic;         /* 0 none, 1 Wang-Teter family (alpha, beta, kinetic_parts), 2 WGC99,
                            3 Huang-Carter family (hc_* below; beta, kappa from the shared fields),
                            4 semilocal (sl_* at the end; with pbe set both share one gradient / divergence round trip) */
    int kinetic_parts;   /* PAD_PART_* mask for kinetic == 1 (e.g. PAD_PART_VW alone = Weizsaecker) */
    int pbe;             /* 0 none, 1 exchange, 2 correlation, 3 both                        */
    double alpha, beta, gamma, kappa;
    /* kinetic == 3: arguments of pad_eval_hc */
    int hc_variant;              /* 0 HuangCarter (hc_p0 = lambda), 1 RevisedHuangCarter (hc_p0 = a, hc_p1 = b) */
    int hc_geometric;
    int hc_n_eta;
    double hc_p0, hc_p1;
    const double* hc_table_dev;  /* DEVICE, 2 * hc_n_eta doubles [eta | omega(eta)]                             */
    /* kinetic == 4: arguments of pad_eval_semilocal_kinetic */
    int sl_variant;              /* PAD_SEMILOCAL_LKT or PAD_SEMILOCAL_PG                                      */
    double sl_p0, sl_p1;
} pad_terms;
int pad_eval_total(pad_plan* plan, const pad_terms* terms, const double* den, const double* v_ext,
                   double* E_out, double* v_out, void* stream);

/* Analytic stress sigma_ij = (1/vol) dE/d eps_ij of the terms of a pad_terms descriptor (everything except
 * IonElectron, see pad_ion_stress): replaces get_stress / System.__compute_stress (functional_tools.py:73-100,
 * system.py:927-935; formulas tests/tools_for_tests.py:212-472).  stress_out: DEVICE, 9 doubles, overwritten.
 * Every kinetic kind is covered: Wang-Teter family, WangGovindCarter99 (kernel regenerated for the strained cell) and the
 * Huang-Carter family (xi-node list held fixed, as the reference's autograd sees it, functional_tools.py:408-416) and the
 * semilocal kind (LuoKarasievTrickey, PauliGaussian: gradient and Laplacian terms). */
int pad_stress_terms(pad_plan* plan, const pad_terms* terms, const double* den, double* stress_out, void* stream);

/* ---- ion-ion interaction: replaces ion_interaction_sum (ion_utils.py:293-333; torch_nl pair list + autograd) with a
 *      direct sweep over (ion j, image shift) candidates per ion i and closed-form derivatives.  box_host: 9 doubles (rows =
 *      lattice vectors); cart_dev: n x 3 Cartesian coordinates (DEVICE); charges_dev: n (DEVICE); charge_total: their sum.
 *      E_out_dev: 1 double.  dcart_dev (n x 3) = dE/dcoords, dbox_dev (9) = dE/dbox_vecs AT FIXED coords (what autograd needs
 *      for a function of the two tensors; the stress follows through coords = frac @ box_vecs) -- either may be null.
 *      work_dev: pad_ion_ion_work_doubles(...) doubles of DEVICE scratch.  Reference vectors: tests/test_ion_utils.py:12-147. */
size_t pad_ion_ion_work_doubles(const double* box_host, int n, double Rc);
int pad_ion_ion(const double* box_host, const double* cart_dev, const double* charges_dev, int n, double charge_total,
                double Rc, double Rd, double* E_out_dev, double* dcart_dev, double* dbox_dev, double* work_dev, int device,
                void* stream);

/* ---- chi-parametrisation (system.py:830-854): n = N chi^2 / int chi^2 and the projected gradient
 *      dE/dchi_ijk = dV (N/Ntilde) 2 chi (v - mu), mu = int v n / N.  grad_out = N doubles. -------- */
int pad_chi_to_density(pad_plan* plan, const double* chi, double n_elec, double* den_out, void* stream);
int pad_chi_project(pad_plan* plan, const double* chi, const double* den, const double* v, double n_elec,
                    double* grad_out, double* stats_out /* device, 4: |g|_1, g.g, max|dE/dchi|, max|mu - v| */,
                    void* stream);

/* ---- device-resident density optimisation: replaces the loop of System.optimize_density
 *      (system.py:866-901) driving LBFGSNew.step (lbfgsnew.py:512-769, fixed step) or TPGD.step
 *      (two_point_gradient_descent.py:25-65).  The host only enqueues work and polls a pinned
 *      status word a few evaluations behind the GPU; there is no synchronisation inside an outer
 *      iteration. ------------------------------------------------------------------------------ */
typedef struct pad_denopt pad_denopt;
typedef struct pad_denopt_params {
    double n_elec;             /* electrons in the cell                                         */
    double ntol;               /* optimize_density(ntol)                                        */
    int n_conv_cond_count;
    int method;                /* 0 = LBFGS, 1 = TPGD                                           */
    double step_size;          /* n_step_size (lr)                                              */
    int n_maxiter;
    int conv_target;           /* 0 = dE [eV], 1 = max|dE/dchi|, 2 = max|mu - dE/dn|            */
    int history;               /* L-BFGS history (reference: 8); <= 8                           */
    int max_iter;              /* L-BFGS inner iterations per step (reference: 6)               */
    double tolerance_grad;     /* 1e-5 */
    double tolerance_change;   /* 1e-9 */
} pad_denopt_params;
typedef struct pad_denopt_result {
    int iterations;            /* outer iterations executed                                     */
    int converged;             /* 1 if the stop rule fired, 0 if n_maxiter was reached          */
    int closures;              /* energy+potential evaluations                                  */
    double energy;             /* functional energy (without ion-ion) of the final density [Ha] */
    double last_dE_eV, last_dEdchi, last_euler;
} pad_denopt_result;
int pad_denopt_create(pad_denopt** opt, pad_plan* plan, const pad_terms* terms, const pad_denopt_params* params);
/* den_inout: initial density in, optimised density out (device).  trace_host (may be NULL) receives
 * 4 doubles per outer iteration: E [eV], dE [eV], max|dE/dchi|, max|mu - dE/dn|. Blocks until done. */
int pad_denopt_run(pad_denopt* opt, double* den_inout, const double* v_ext, pad_denopt_result* result_host,
                   double* trace_host, void* stream);
int pad_denopt_destroy(pad_denopt* opt);

#ifdef __cplusplus
}
#endif
#endif
