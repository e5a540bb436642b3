// Shared device/host helpers for the B200 OFDFT hot path.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <cufft.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>

#include "../../include/professad_b200.h"

#define PAD_MAX_RED 8            // reductions per kernel
#define PAD_MAX_BLOCKS 1184      // 148 SMs x 8 resident 256-thread CTAs
#define PAD_THREADS 256
#define PAD_N_RBUF 8             // real scratch fields
#define PAD_N_CBUF 4             // half-spectrum scratch fields
#define PAD_N_SCAL 64            // device scalars

constexpr double kPi = 3.14159265358979323846;
// 0.3 (3 pi^2)^(2/3)
constexpr double kCTF = 2.871234000188191;

void pad_set_error(const char* fmt, ...);
extern unsigned long long g_pad_launches;   // kernels launched by this library (own kernels + cuFFT execs)
extern unsigned long long g_pad_fft_execs;

#define PAD_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e_ = (call);                                                                \
        if (e_ != cudaSuccess) {                                                                \
            pad_set_error("CUDA error %s at %s:%d (%s)", cudaGetErrorString(e_), __FILE__, __LINE__, #call); \
            return PAD_ERR_CUDA;                                                                \
        }                                                                                       \
    } while (0)

#define PAD_CUFFT(call)                                                                         \
    do {                                                                                        \
        cufftResult r_ = (call);                                                                \
        if (r_ != CUFFT_SUCCESS) {                                                              \
            pad_set_error("cuFFT error %d at %s:%d (%s)", (int)r_, __FILE__, __LINE__, #call);  \
            return PAD_ERR_CUFFT;                                                               \
        }                                                                                       \
    } while (0)

#define PAD_TRY(call)                \
    do {                             \
        int rc_ = (call);            \
        if (rc_ != PAD_OK) return rc_; \
    } while (0)

// ---------------------------------------------------------------------------------------------
//  reciprocal-space geometry: restates wavevecs() (functional_tools.py:135-162) per k-point
// ---------------------------------------------------------------------------------------------
struct KGeom {
    int n0, n1, n2, nzh;     // grid and half-spectrum length along axis 2
    int e0, e1, e2;          // axis length even?
    double b[9];             // reciprocal lattice, rows = b_i = 2 pi inv(box^T)[i]
    double inv_n;            // 1 / (n0 n1 n2): cuFFT transforms are unnormalised
    int nzp_pad;             // padded row length (complex) of the fused-pipeline spectra: n2/2 + 8
    int n1_loc, j1_off;      // half-spectrum rows held by this plan: (n0, n1_loc, nzh), j1 = local index + j1_off
                             // (single-GPU plans: n1_loc = n1, j1_off = 0; slab plans: the rank's y range)
};

struct KPoint {
    double kx, ky, kz;       // k(p) with the reference's "Nyquist made positive" convention
    double px, py, pz;       // k(pbar), the Hermitian partner on a self-conjugate plane
    bool special;            // p lies on a self-conjugate plane AND carries a Nyquist index
    int j0, j1, j2;
};

__device__ __forceinline__ KPoint make_kpoint_at(const KGeom& g, int j0, int j1, int j2) {
    KPoint p;
    p.j0 = j0; p.j1 = j1; p.j2 = j2;
    const double f0 = (double)(p.j0 <= g.n0 / 2 ? p.j0 : p.j0 - g.n0);
    const double f1 = (double)(p.j1 <= g.n1 / 2 ? p.j1 : p.j1 - g.n1);
    const double f2 = (double)p.j2;
    p.kx = f0 * g.b[0] + f1 * g.b[3] + f2 * g.b[6];
    p.ky = f0 * g.b[1] + f1 * g.b[4] + f2 * g.b[7];
    p.kz = f0 * g.b[2] + f1 * g.b[5] + f2 * g.b[8];
    const bool nyq0 = g.e0 && (p.j0 == g.n0 / 2);
    const bool nyq1 = g.e1 && (p.j1 == g.n1 / 2);
    const bool nyq2 = g.e2 && (p.j2 == g.n2 / 2);
    const bool selfconj = (p.j2 == 0) || nyq2;
    p.special = selfconj && (nyq0 || nyq1 || nyq2);
    p.px = p.kx; p.py = p.ky; p.pz = p.kz;
    if (p.special) {
        const double q0 = nyq0 ? f0 : -f0;
        const double q1 = nyq1 ? f1 : -f1;
        p.px = q0 * g.b[0] + q1 * g.b[3] + f2 * g.b[6];
        p.py = q0 * g.b[1] + q1 * g.b[4] + f2 * g.b[7];
        p.pz = q0 * g.b[2] + q1 * g.b[5] + f2 * g.b[8];
    }
    return p;
}

__device__ __forceinline__ KPoint make_kpoint(const KGeom& g, uint32_t idx) {
    const uint32_t row = idx / (uint32_t)g.nzh;
    const int j2 = (int)(idx - row * (uint32_t)g.nzh);
    const int j0 = (int)(row / (uint32_t)g.n1_loc);
    const int j1 = (int)(row - (uint32_t)j0 * (uint32_t)g.n1_loc) + g.j1_off;
    return make_kpoint_at(g, j0, j1, j2);
}

// Effective real multiplier M(|k|^2-like even function) on the half spectrum: on special points the
// reference's irfftn sees the Hermitian part (M(p) + M(pbar)) / 2  (DESIGN.md "Nyquist semantics").
template <class M>
__device__ __forceinline__ double sym_even(const KPoint& p, M mult) {
    double m = mult(p.kx, p.ky, p.kz);
    if (p.special) m = 0.5 * (m + mult(p.px, p.py, p.pz));
    return m;
}

// |k|^2 along a line of the half spectrum with fixed (j1, j2) and running j0: k(p) = f0 b0 + C, C = f1 b1 + f2 b2, so
// |k|^2 = f0^2 |b0|^2 + 2 f0 (b0.C) + |C|^2 -- two FMAs per point instead of a make_kpoint_at; same for the Hermitian
// partner pbar = (-j0, -j1, j2) (Nyquist indices keep their sign) that special points average with (sym_even).
struct KLine {
    double B00, d, cc, db, ccb;
    int n0, half0;
    bool e0, selfconj, nyq12;
};
__device__ __forceinline__ KLine make_kline(const KGeom& g, int j1, int j2) {
    KLine L;
    const double f1 = (double)(j1 <= g.n1 / 2 ? j1 : j1 - g.n1), f2 = (double)j2;
    const bool nyq1 = g.e1 && (j1 == g.n1 / 2), nyq2 = g.e2 && (j2 == g.n2 / 2);
    const double q1 = nyq1 ? f1 : -f1;
    const double cx = f1 * g.b[3] + f2 * g.b[6], cy = f1 * g.b[4] + f2 * g.b[7], cz = f1 * g.b[5] + f2 * g.b[8];
    const double px = q1 * g.b[3] + f2 * g.b[6], py = q1 * g.b[4] + f2 * g.b[7], pz = q1 * g.b[5] + f2 * g.b[8];
    L.B00 = g.b[0] * g.b[0] + g.b[1] * g.b[1] + g.b[2] * g.b[2];
    L.d = g.b[0] * cx + g.b[1] * cy + g.b[2] * cz;
    L.cc = cx * cx + cy * cy + cz * cz;
    L.db = g.b[0] * px + g.b[1] * py + g.b[2] * pz;
    L.ccb = px * px + py * py + pz * pz;
    L.n0 = g.n0; L.half0 = g.n0 / 2; L.e0 = g.e0;
    L.selfconj = (j2 == 0) || nyq2;
    L.nyq12 = nyq1 || nyq2;
    return L;
}
// sym_even for a multiplier that depends on k only through |k|^2
template <class M>
__device__ __forceinline__ double kline_sym_even(const KLine& L, int j0, M mult_of_k2) {
    const double f0 = (double)(j0 <= L.half0 ? j0 : j0 - L.n0);
    const double k2 = fma(f0, fma(f0, L.B00, 2.0 * L.d), L.cc);
    double m = mult_of_k2(k2);
    const bool nyq0 = L.e0 && (j0 == L.half0);
    if (L.selfconj && (L.nyq12 || nyq0)) {
        const double q0 = nyq0 ? f0 : -f0;
        m = 0.5 * (m + mult_of_k2(fma(q0, fma(q0, L.B00, 2.0 * L.db), L.ccb)));
    }
    return m;
}

// Effective wave-vector for the gradient multiplier i*k_c:  (k(p) - k(pbar)) / 2 on special points.
__device__ __forceinline__ void sym_kvec(const KPoint& p, double& kx, double& ky, double& kz) {
    kx = p.kx; ky = p.ky; kz = p.kz;
    if (p.special) {
        kx = 0.5 * (p.kx - p.px);
        ky = 0.5 * (p.ky - p.py);
        kz = 0.5 * (p.kz - p.pz);
    }
}

// ---------------------------------------------------------------------------------------------
//  block reduction: warp shuffles, then one shared-memory hop.  Deterministic for a fixed grid.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <int NRED>
__device__ __forceinline__ void block_reduce_store(const double (&acc)[NRED], double* __restrict__ partials) {
    __shared__ double sm[NRED][PAD_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int t = 0; t < NRED; ++t) {
        double v = warp_sum(acc[t]);
        if (lane == 0) sm[t][warp] = v;
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int t = 0; t < NRED; ++t) {
            double v = lane < PAD_THREADS / 32 ? sm[t][lane] : 0.0;
            v = warp_sum(v);
            if (lane == 0) partials[(size_t)t * PAD_MAX_BLOCKS + blockIdx.x] = v;
        }
    }
}

// real-space elementwise kernel: f(i, acc) for every grid point, NRED block-reduced sums
template <int NRED, class F>
__global__ void __launch_bounds__(PAD_THREADS) ew_kernel(size_t n, F f, double* __restrict__ partials) {
    double acc[NRED > 0 ? NRED : 1];
#pragma unroll
    for (int t = 0; t < (NRED > 0 ? NRED : 1); ++t) acc[t] = 0.0;
    const size_t stride = (size_t)gridDim.x * PAD_THREADS;
    for (size_t i = (size_t)blockIdx.x * PAD_THREADS + threadIdx.x; i < n; i += stride) f(i, acc);
    if (NRED > 0) block_reduce_store<(NRED > 0 ? NRED : 1)>(acc, partials);
}

// reciprocal-space kernel: f(idx, kpoint) for every half-spectrum point
template <class F>
__global__ void __launch_bounds__(PAD_THREADS) ks_kernel(KGeom g, uint32_t nk, F f) {
    const uint32_t stride = gridDim.x * PAD_THREADS;
    for (uint32_t idx = blockIdx.x * PAD_THREADS + threadIdx.x; idx < nk; idx += stride) {
        KPoint p = make_kpoint(g, idx);
        f(idx, p);
    }
}

inline int pad_grid_for(size_t n) {
    size_t b = (n + PAD_THREADS - 1) / PAD_THREADS;
    if (b > PAD_MAX_BLOCKS) b = PAD_MAX_BLOCKS;
    if (b < 1) b = 1;
    return (int)b;
}

// ---------------------------------------------------------------------------------------------
//  the plan
// ---------------------------------------------------------------------------------------------
struct pad_plan {
    int n0, n1, n2, nzh;
    size_t N, Nk;
    double box[9], recip[9], vol, dV;
    int device;
    KGeom geom;
    cufftHandle d2z, z2d;
    bool fft_ready;
    void* fft_work;
    size_t fft_work_bytes;
    cudaStream_t fft_stream;
    double* rbuf[PAD_N_RBUF];
    cufftDoubleComplex* cbuf[PAD_N_CBUF];
    double* partials;            // PAD_MAX_RED * PAD_MAX_BLOCKS
    double* scal;                // PAD_N_SCAL device scalars
    // WGC99 kernel cache: 4 half-spectrum real arrays W0, K1, K2, K3 and the key they were built for
    double* wgc_kern;
    double* wgc_kern4;           // same kernels, interleaved (W0,K1,K2,K3) per k-point over the PADDED half-spectrum layout
    double wgc_key[6];           // alpha, beta, gamma, kappa, + box generation, valid flag
    uint64_t box_generation;
    // fused Wang-Teter pipeline: 1/G^-1(eta) - 3 eta^2 - 1 per k-point over the padded half-spectrum layout
    double* wt_kern;
    uint64_t wt_kern_generation;
    // Huang-Carter scratch: xi-node list (+ min/max words), table slopes, n_xi convolution fields
    double* hc_scratch;
    double* hc_slopes;
    int hc_slopes_n;
    double* hc_conv;
    int hc_conv_nodes;
    // fused z-pass pipeline (fftz.cu): padded half-spectrum buffers and the batched 2-D (x, y) cuFFT plan
    int nzp;
    cufftHandle xy;
    bool xy_ready;
    void* xy_work;
    cudaStream_t xy_stream;
    cufftDoubleComplex* zbuf[4];
    size_t bytes_allocated;
    // software-pipelined (z, y) kernels (zy_pipe.cuh): control block, per-item partial sums
    void* pipe_ctl;
    double* pipe_part;
    size_t pipe_part_n;
    // ionic potential / forces (ions.cu): per-ion 1-D phase tables + table slopes, force partial sums
    void* ion_scratch;
    size_t ion_scratch_bytes;
    double* ion_partial;
    size_t ion_partial_bytes;
    // slab decomposition over `world` ranks (plan.cu, "slab plans"): real space is split along axis 0
    // (n0_loc planes per rank), reciprocal space along axis 1 (n1_loc rows per rank, all of axis 0).
    // N and Nk above are then the LOCAL point counts; dV, vol, geom.inv_n stay global.
    bool dist;
    int rank, world, n0_loc, n1_loc;
    cufftHandle d2z_yz, z2d_yz, z2z_x;
    void *send_buf, *recv_buf;   // Nk complex each, owned by the caller
    // second exchange buffer pair + a communication stream: batches of transforms are software-pipelined so that the
    // all-to-all of one field runs while the local FFTs of its neighbours do (pad_fft_forward_many / _inverse_many)
    void *send_buf2, *recv_buf2;
    void* peer_recv[2][8];       // cuFFT slab path over peer memory: every rank's two receive buffers (pad_plan_set_slab_peer_recv)
    bool recv_push;              // ... registered: the permute kernel stores straight into the owners' receive buffers
    bool recv_after_pipeline;    // a pipelined batch has used the receive pair since the last single transform
    int recv_parity;             // receive buffer the next transform uses (alternating: see fft_forward_slab)
    // CUDA graphs of whole evaluations (pad_eval_wgc99 / the fused term list): one instantiated graph per distinct argument set
    struct GraphSlot {
        unsigned long long key[14];
        void* exec;                  // cudaGraphExec_t
        unsigned long long launches; // kernels in the graph (pad_launch_count goes up by this per replay)
        unsigned long long stamp;    // last use (LRU)
        int state;                   // 0 empty, 1 argument set seen once (run directly), 2 captured, -1 capture failed: always direct
    } graphs[16];
    cudaStream_t graph_stream;   // private capture stream (the caller's may be the legacy default stream, which cannot capture)
    unsigned long long graph_clock;
    bool slab_push;              // peer pointers registered (pad_plan_set_slab_peer_buffers): transposition by NVLink stores of the y / x passes
    void *peer_B[4][8], *peer_T[4][8];      // [field][rank]: local-layout and transposed-layout spectrum buffers of every rank
    void* slab_fast[6];          // fused pipeline on slabs: 4 spectrum buffers + 2 exchange stagings of n0_loc * n1 * nzp complex, owned by the caller
    cudaStream_t comm_stream;
    cudaEvent_t ev_ready[2], ev_a2a[2], ev_free[2];
    bool comm_ready;
    double* comm_scratch;        // PAD_COMM_SCRATCH doubles, owned by the caller
    pad_comm_fn comm_fn;
    void* comm_user;
};

// scalar slots (device doubles in plan->scal)
enum {
    S_SUM_RHO = 0,      // sum of n over the grid
    S_N0 = 1,           // mean density
    S_NREF = 2,         // WGC99 reference density kappa * round(N_elec) / vol
    S_NREF_KEY = 3,     // n_ref the cached WGC99 kernel was built for
    S_WT_KEY = 4,       // n0 the cached Lindhard kernel table of the fused Wang-Teter pipeline was built for
    S_GRAPH_E = 6,      // energy output of a replayed evaluation graph (copied to the caller's scalar after the launch)
    S_CTR = 5,          // two 32-bit arrival counters of "last CTA finishes the job" kernels (zero between launches)
    S_TMP0 = 8,         // 8 slots of per-call temporaries
    S_E_PARTS = 16      // component energies
};

int pad_get_rbuf(pad_plan* p, int i, double** out);
int pad_get_cbuf(pad_plan* p, int i, cufftDoubleComplex** out);
int pad_fft_forward(pad_plan* p, const double* in, cufftDoubleComplex* out, cudaStream_t s);
int pad_fft_inverse(pad_plan* p, cufftDoubleComplex* in, double* out, cudaStream_t s);
// n independent transforms; on slab plans with a second exchange buffer pair the all-to-all of field f overlaps the
// local transforms of fields f - 1 and f + 1 (otherwise a plain loop)
int pad_fft_forward_many(pad_plan* p, const double* const* in, cufftDoubleComplex* const* out, int n, cudaStream_t s);
int pad_fft_inverse_many(pad_plan* p, cufftDoubleComplex* const* in, double* const* out, int n, cudaStream_t s);
extern int g_pad_own_xy;
extern int g_pad_pipe;             // 1: software-pipelined (z, y) kernels where the shape allows (default)
extern int g_pad_zinv_stream;      // 1: streamed inverse z kernel (results folded as they arrive, 3 CTAs/SM), 0: batch form
extern int g_pad_local_tail;       // 1: fused term list with the local terms in the one-field Hartree inverse pass (0: inside the mid pass)
extern int g_pad_pbe_fast;         // 1: PerdewBurkeErnzerhof on the fused passes where they cover the grid
extern int g_pad_xone;             // 1: one-field x passes (-k^2, 4 pi / k^2) as the two-transform plain pass
extern int g_pad_ywide;            // 1: y pass at L = 256 with 32 threads per line (8 points each)
extern int g_pad_graphs;           // 1: repeated evaluations with the same arguments replay a CUDA graph
extern unsigned long long g_pad_option_epoch;      // bumped by pad_set_option (part of the graph keys)
extern int g_pad_fuse_mid;         // 1: WGC99 mid pass and the forward z pass of the second batch in one kernel
extern int g_pad_fold_table;       // 1: orthorhombic cells read only the |kx|, |ky| quarter of the WGC99 kernel table
extern int g_pad_fuse_terms;       // 1: pad_eval_total folds local terms + Hartree into the WGC99 pipeline where it can
extern int g_pad_pipe_lpi;         // lines per z item (0: default)
extern int g_pad_pipe_tpi;         // tiles per y item (0: default)
extern int g_pad_profile;          // 1: record CUDA events between pipeline stages (pad_profile_begin/end)
void pad_stage_begin(cudaStream_t s);
void pad_stage_mark(const char* name, cudaStream_t s);
extern int g_pad_fast_fft;    // 1: use the fused z-pass pipeline where the shape allows (default), 0: plain cuFFT 3-D
int pad_wgc99_fast_supported(const pad_plan* p);
int pad_local_fast(pad_plan* p, const double* den, const double* v_ext, int mask, double* E_out, double* v_out, int accumulate, cudaStream_t s);
int pad_pbe_pointwise(pad_plan* p, cudaStream_t s, const double* den, double* gx, double* gy, double* gz, double* v, int which,
                      int accumulate, int* grid_out);
int pad_pbe_fast_supported(const pad_plan* p);
int pad_pbe_fast(pad_plan* p, const double* den, int which, double* E_out, double* v_out, int accumulate, cudaStream_t s);
// semilocal kinetic functional (PAD_SEMILOCAL_*, parameters p0, p1) plus, with pbe != 0, the PBE terms (1 x, 2 c, 3 both) in the
// same point kernel
struct pad_semilocal_args {
    int variant;
    double p0, p1;
    int pbe;
};
int pad_semilocal_pointwise(pad_plan* p, cudaStream_t s, const double* den, double* gx, double* gy, double* gz, double* lap, double* v,
                            const pad_semilocal_args& P, int accumulate, int* grid_out);
int pad_semilocal_fast(pad_plan* p, const double* den, const pad_semilocal_args& P, double* E_out, double* v_out, int accumulate,
                       cudaStream_t s);
int pad_eval_semilocal_ex(pad_plan* p, const double* den, const pad_semilocal_args& P, double* E_out, double* v_out, int accumulate,
                          void* stream);
int pad_hartree_fast_supported(const pad_plan* p);
int pad_hartree_fast(pad_plan* p, const double* den, double* E_out, double* v_out, int accumulate, cudaStream_t s);
int pad_wt_fast_supported(const pad_plan* p);
int pad_wt_fast(pad_plan* p, const double* den, double alpha, double beta, double* E_out, double* v_out, int accumulate,
                cudaStream_t s);
// extra terms evaluated inside the WGC99 pipeline (fused term list): local terms in the mid pass, Hartree as a fourth
// field of the second batch
struct pad_wgc_extras {
    int local_mask;            // PAD_LOCAL_LDAX | PAD_LOCAL_PZC | PAD_LOCAL_IONEL (not TF: WGC99 carries its own)
    const double* v_ext;       // for PAD_LOCAL_IONEL
    int hartree;
};
int pad_wgc99_total_supported(const pad_plan* p);
int pad_wgc99_fast(pad_plan* p, const double* den, double alpha, double beta, const double* kern, double* E_out,
                   double* v_out, int accumulate, cudaStream_t s, const pad_wgc_extras* ex);
int pad_eval_wgc99_ex(pad_plan* p, const double* den, double alpha, double beta, double gamma, double kappa, double* E_out,
                      double* v_out, int accumulate, void* stream, const pad_wgc_extras* ex);

// finalize: E_out (+)= sum_t coef[t] * (sum over blocks of partials[t]); optionally store raw sums
struct FinalizeArgs {
    int nblocks, nterms, accumulate;
    double coef[PAD_MAX_RED];
    double* sums_out;     // nterms raw sums (may be null)
    double* E_out;        // may be null
};
void pad_launch_finalize(pad_plan* p, const FinalizeArgs& a, cudaStream_t s);
// slab plans (no-ops otherwise): combine `n` device values over the ranks, in place and ordered with `s`.
// max: non-negative doubles held as their bit patterns (the atomicMax convention of the reduction kernels).
int pad_allreduce_max_bits(pad_plan* p, unsigned long long* bits, int n, cudaStream_t s);
int pad_slab_comm(pad_plan* p, int op, long long count, cudaStream_t s);
int pad_ensure_comm_stream(pad_plan* p);      // plan-owned communication stream + the events of the pipelined exchanges
// stress.cu: the 7 block-reduced sums [iso, xx, yy, zz, xy, xz, yz] left in p->partials by a kernel with `nblocks`
// CTAs are finished (all-reduced on slab plans) and added to the row-major 3 x 3 device tensor `sig`:
// sig_ij += c_t T_ij + c_iso iso delta_ij
int pad_stress_accumulate(pad_plan* p, cudaStream_t s, int nblocks, double c_iso, double c_t, double* sig);
// hc.cu: stress of the non-local term of the Huang-Carter family, added to sig[9]
int pad_stress_hc_nl(pad_plan* p, const double* den, int variant, double p0, double p1, double beta, double kappa, int geometric,
                     const double* table_dev, int n_eta, double* sig, cudaStream_t s);
// functionals.cu (needs the WGC99 series constants of that translation unit): non-local WGC99 stress, added to sig[9]
int pad_stress_wgc99_nl(pad_plan* p, const double* den, double alpha, double beta, double gamma, double kappa, double* sig,
                        cudaStream_t s);
