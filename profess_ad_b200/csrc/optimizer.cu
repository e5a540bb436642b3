// Fused evaluation of a term list, the chi-parametrisation kernels, and the device-resident
// density optimiser (L-BFGS with fixed step / Barzilai-Borwein TPGD).
//
// Replaces the loop of System.optimize_density (system.py:866-901) driving LBFGSNew.step
// (lbfgsnew.py:512-769, line_search_fn=False) or TPGD.step (two_point_gradient_descent.py:25-65).
//
// Design (DESIGN.md "device-resident optimiser"):
//  * all optimiser scalars live in one device struct (OptState); the branches of the reference
//    (curvature test, six break conditions, outer stop rule) are taken by one-thread "transition"
//    kernels, and the vector kernels are predicated on the flags those set;
//  * the L-BFGS two-loop recursion runs in coefficient space ("vector-free" L-BFGS): one fused pass
//    forms s = t d, y = g - g_prev and ALL inner products the recursion needs (Gram rows of the new
//    pair, S.g, Y.g), a scalar kernel turns them into the coefficients of d in the basis
//    {s_i, y_i, g}, and one fused pass assembles d, steps chi and updates g_prev.  Two passes over
//    the history instead of ~4 m sequential dot/axpy launches with a host sync each;
//  * the host enqueues "ticks" (closure + transition + move) and polls a pinned copy of the status
//    a few ticks behind the GPU: no host synchronisation inside an outer iteration.
#include <stdlib.h>

#include "common.cuh"

#define OPT_M 8                 // max history
#define OPT_SLOTS (OPT_M + 1)   // one spare slot for the provisional (s, y) pair
#define OPT_NACC (5 + 5 * OPT_SLOTS)
#define OPT_LOOKAHEAD 3
#define OPT_RING 8

namespace {

constexpr double kEvPerHa = 4.3597447222071e-18 / 1.602176634e-19;

struct OptState {
    // ---- closure outputs
    double sum_chi2, sum_vrho, E, g_l1, gg;
    unsigned long long max_dEdchi_bits, max_euler_bits;
    // ---- L-BFGS
    int k, order[OPT_M], free_slot;
    double SY[OPT_SLOTS][OPT_SLOTS], YY[OPT_SLOTS][OPT_SLOTS], Sg[OPT_SLOTS], Yg[OPT_SLOTS];
    double cS[OPT_SLOTS], cY[OPT_SLOTS], cg;
    double H, t, loss, prev_loss, gtd, d_l1;
    int n_iter_total, it, evals, phase, do_move, do_pass1;
    // ---- TPGD
    int tp_iter;
    double tp_alpha;
    // ---- outer loop
    int outer_iter, conv_count, done, converged, closures;
    double E_prev_eV, last_dE, last_dEdchi, last_euler;
};

struct OptParams {
    double n_elec, ntol, lr, tol_grad, tol_change, dV;
    int n_conv, method, n_maxiter, conv_target, history, max_iter, max_eval;
};

__device__ __forceinline__ double bits_to_double(unsigned long long b) { return __longlong_as_double((long long)b); }

// ------------------------------------------------------------------------------------------------
//  closure kernels
// ------------------------------------------------------------------------------------------------
__global__ void k_reset_max(OptState* st) {
    st->max_dEdchi_bits = 0ull;
    st->max_euler_bits = 0ull;
}

// one-CTA reduction of per-block partials (nterms rows of PAD_MAX_BLOCKS)
__device__ void reduce_partials(const double* __restrict__ partials, int nblocks, int nterms, int row_stride,
                                double* out /*shared, nterms*/) {
    __shared__ double sm[PAD_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int t = 0; t < nterms; ++t) {
        double v = 0.0;
        for (int b = threadIdx.x; b < nblocks; b += PAD_THREADS) v += partials[(size_t)t * row_stride + b];
        v = warp_sum(v);
        if (lane == 0) sm[warp] = v;
        __syncthreads();
        if (warp == 0) {
            double w = lane < PAD_THREADS / 32 ? sm[lane] : 0.0;
            w = warp_sum(w);
            if (lane == 0) out[t] = w;
        }
        __syncthreads();
    }
}

// the sums a transition kernel needs: reduced here from the per-block partials (single GPU), or already reduced
// and all-reduced over the ranks in `totals` (slab plans, see slab_reduce below)
__device__ void gather_sums(const double* __restrict__ partials, int nblocks, int nterms, const double* __restrict__ totals,
                            double* out /*shared, nterms*/) {
    if (totals) {
        if ((int)threadIdx.x < nterms) out[threadIdx.x] = totals[threadIdx.x];
        __syncthreads();
    } else {
        reduce_partials(partials, nblocks, nterms, PAD_MAX_BLOCKS, out);
    }
}

__global__ void __launch_bounds__(PAD_THREADS) k_reduce_to(const double* __restrict__ partials, int nblocks, int nterms,
                                                         double* __restrict__ out) {
    __shared__ double sums[OPT_NACC];
    reduce_partials(partials, nblocks, nterms, PAD_MAX_BLOCKS, sums);
    if ((int)threadIdx.x < nterms) out[threadIdx.x] = sums[threadIdx.x];
}

// stop rule of System.optimize_density (system.py:869-901), run at the end of every optimiser step
__device__ void end_step(OptState& st, const OptParams& P, double* trace) {
    st.outer_iter++;
    const double E_eV = st.E * kEvPerHa;
    const double dE = E_eV - st.E_prev_eV;
    st.E_prev_eV = E_eV;
    const double dEdchi = bits_to_double(st.max_dEdchi_bits), euler = bits_to_double(st.max_euler_bits);
    st.last_dE = dE; st.last_dEdchi = dEdchi; st.last_euler = euler;
    if (trace) {
        double* row = trace + 4 * (size_t)(st.outer_iter - 1);
        row[0] = E_eV; row[1] = dE; row[2] = dEdchi; row[3] = euler;
    }
    const double stop = P.conv_target == 0 ? fabs(dE) : (P.conv_target == 1 ? dEdchi : euler);
    if (st.outer_iter > 5) st.conv_count = (stop < P.ntol) ? st.conv_count + 1 : 0;
    if (st.conv_count == P.n_conv) { st.done = 1; st.converged = 1; }
    else if (st.outer_iter >= P.n_maxiter) { st.done = 1; }
}

// after the closure: finish the gradient reductions, then the L-BFGS / TPGD state machine
__global__ void __launch_bounds__(PAD_THREADS) k_after_closure(OptState* stp, OptParams P, const double* __restrict__ partials,
                                                             int nblocks, const double* __restrict__ totals, double* trace) {
    __shared__ double sums[2];
    gather_sums(partials, nblocks, 2, totals, sums);
    if (threadIdx.x != 0) return;
    OptState& st = *stp;
    if (st.done) { st.do_move = 0; st.do_pass1 = 0; return; }
    st.g_l1 = sums[0];
    st.gg = sums[1];
    st.closures++;
    st.do_move = 0;
    st.do_pass1 = 0;
    const double g_l1 = st.g_l1;
    if (P.method == 1) {                       // ---- TPGD: every closure is one optimiser step
        st.do_move = 1;
        st.do_pass1 = 1;
        return;
    }
    if (st.phase == 1) {                       // closure that followed the move of inner iteration `it`
        st.loss = st.E;
        bool brk = isnan(g_l1);
        if (!brk) {
            st.evals++;
            brk = (st.evals >= P.max_eval) || (g_l1 <= P.tol_grad) || (st.gtd > -P.tol_change) ||
                  (fabs(st.t) * st.d_l1 <= P.tol_change) || (fabs(st.loss - st.prev_loss) < P.tol_change);
        }
        if (brk) {
            end_step(st, P, trace);
            st.phase = 0;
            if (st.done) return;
            // the reference would now re-evaluate the closure at the same chi (first line of the next
            // step()); E and g are already known, so fall through and start that step directly
        }
    }
    if (st.phase == 0) {                       // first closure of a step
        st.loss = st.E;
        st.evals = 1;
        st.it = 0;
        if (g_l1 <= P.tol_grad || isnan(st.gg)) {      // step() returns at once (lbfgsnew.py:548, :568)
            end_step(st, P, trace);
            return;
        }
        st.phase = 1;
    }
    st.it++;
    st.n_iter_total++;
    st.do_move = 1;
    st.do_pass1 = st.n_iter_total > 1;
}

// ------------------------------------------------------------------------------------------------
//  L-BFGS pass 1: s = t d, y = g - g_prev into the free slot, and every inner product needed
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(PAD_THREADS) k_lbfgs_pass1(size_t n, const OptState* __restrict__ stp, const double* __restrict__ g,
                                                           const double* __restrict__ prev_g, const double* __restrict__ d,
                                                           double* __restrict__ Sh, double* __restrict__ Yh,
                                                           double* __restrict__ partials) {
    if (!stp->do_pass1) return;
    const int k = stp->k, fs = stp->free_slot;
    const double t = stp->t;
    bool used[OPT_SLOTS];
#pragma unroll
    for (int a = 0; a < OPT_SLOTS; ++a) used[a] = false;
    for (int i = 0; i < k; ++i) {
        const int a = stp->order[i];
#pragma unroll
        for (int b = 0; b < OPT_SLOTS; ++b) if (b == a) used[b] = true;
    }
    double acc[OPT_NACC];
#pragma unroll
    for (int j = 0; j < OPT_NACC; ++j) acc[j] = 0.0;
    double* __restrict__ s_new = Sh + (size_t)fs * n;
    double* __restrict__ y_new = Yh + (size_t)fs * n;
    const size_t stride = (size_t)gridDim.x * PAD_THREADS;
    for (size_t i = (size_t)blockIdx.x * PAD_THREADS + threadIdx.x; i < n; i += stride) {
        // every load of the iteration is issued before the first use (predicated loads, no branches): with up to
        // 2 k + 3 vectors to stream the pass is bound by the bytes a thread keeps in flight
        const double gi = g[i], pg = prev_g[i], di = d[i];
        double sa[OPT_SLOTS], ya[OPT_SLOTS];
#pragma unroll
        for (int a = 0; a < OPT_SLOTS; ++a) {
            sa[a] = used[a] ? Sh[(size_t)a * n + i] : 0.0;
            ya[a] = used[a] ? Yh[(size_t)a * n + i] : 0.0;
        }
        const double y = gi - pg;
        const double s = t * di;
        s_new[i] = s;
        y_new[i] = y;
        acc[0] += s * y; acc[1] += y * y; acc[2] += s * s; acc[3] += s * gi; acc[4] += y * gi;
#pragma unroll
        for (int a = 0; a < OPT_SLOTS; ++a) {
            acc[5 + 5 * a + 0] += sa[a] * y;      // s_a . y_new
            acc[5 + 5 * a + 1] += s * ya[a];      // s_new . y_a
            acc[5 + 5 * a + 2] += ya[a] * y;      // y_a . y_new
            acc[5 + 5 * a + 3] += sa[a] * gi;     // s_a . g
            acc[5 + 5 * a + 4] += ya[a] * gi;     // y_a . g
        }
    }
    // block reduction of OPT_NACC sums
    __shared__ double sm[PAD_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < OPT_NACC; ++j) {
        double v = warp_sum(acc[j]);
        if (lane == 0) sm[warp] = v;
        __syncthreads();
        if (warp == 0) {
            double w = lane < PAD_THREADS / 32 ? sm[lane] : 0.0;
            w = warp_sum(w);
            if (lane == 0) partials[(size_t)j * PAD_MAX_BLOCKS + blockIdx.x] = w;
        }
        __syncthreads();
    }
}

// scalar part: curvature test, history update, two-loop recursion in coefficient space
__global__ void __launch_bounds__(PAD_THREADS) k_lbfgs_direction(OptState* stp, OptParams P, const double* __restrict__ partials,
                                                               int nblocks, const double* __restrict__ totals) {
    __shared__ double sums[OPT_NACC];
    OptState& st = *stp;
    if (!st.do_move) return;
    if (st.do_pass1) gather_sums(partials, nblocks, OPT_NACC, totals, sums);
    if (threadIdx.x != 0) return;
    if (st.n_iter_total == 1) {
        st.k = 0;
        st.free_slot = 0;
        st.H = 1.0;
    } else {
        const int f = st.free_slot;
        const double ys = sums[0], yy = sums[1], ss = sums[2];
        for (int i = 0; i < st.k; ++i) {
            const int a = st.order[i];
            st.Sg[a] = sums[5 + 5 * a + 3];
            st.Yg[a] = sums[5 + 5 * a + 4];
        }
        if (ys > 1e-10 * ss) {                         // lbfgsnew.py:622
            int released = -1;
            if (st.k == P.history) {                   // drop the oldest pair
                released = st.order[0];
                for (int i = 1; i < st.k; ++i) st.order[i - 1] = st.order[i];
                st.k--;
            }
            for (int i = 0; i < st.k; ++i) {
                const int a = st.order[i];
                st.SY[a][f] = sums[5 + 5 * a + 0];
                st.SY[f][a] = sums[5 + 5 * a + 1];
                st.YY[a][f] = st.YY[f][a] = sums[5 + 5 * a + 2];
            }
            st.SY[f][f] = ys;
            st.YY[f][f] = yy;
            st.Sg[f] = sums[3];
            st.Yg[f] = sums[4];
            st.order[st.k++] = f;
            st.H = ys / yy;                             // lbfgsnew.py:634
            if (released >= 0) st.free_slot = released;
            else {
                bool taken[OPT_SLOTS];
                for (int b = 0; b < OPT_SLOTS; ++b) taken[b] = false;
                for (int i = 0; i < st.k; ++i) taken[st.order[i]] = true;
                for (int b = 0; b < OPT_SLOTS; ++b) if (!taken[b]) { st.free_slot = b; break; }
            }
        }
    }
    // two-loop recursion (lbfgsnew.py:641-663) on coefficients of {s_a, y_a, g}
    double al[OPT_SLOTS];
    for (int b = 0; b < OPT_SLOTS; ++b) { st.cS[b] = 0.0; st.cY[b] = 0.0; al[b] = 0.0; }
    st.cg = -1.0;
    for (int i = st.k - 1; i >= 0; --i) {
        const int a = st.order[i];
        double sq = st.cg * st.Sg[a];
        for (int j = 0; j < st.k; ++j) { const int b = st.order[j]; sq += st.cY[b] * st.SY[a][b]; }
        al[a] = sq / st.SY[a][a];
        st.cY[a] -= al[a];
    }
    st.cg *= st.H;
    for (int j = 0; j < st.k; ++j) st.cY[st.order[j]] *= st.H;
    for (int i = 0; i < st.k; ++i) {
        const int a = st.order[i];
        double yr = st.cg * st.Yg[a];
        for (int j = 0; j < st.k; ++j) {
            const int b = st.order[j];
            yr += st.cY[b] * st.YY[a][b] + st.cS[b] * st.SY[b][a];
        }
        st.cS[a] += al[a] - yr / st.SY[a][a];
    }
    double gtd = st.cg * st.gg;
    for (int j = 0; j < st.k; ++j) { const int b = st.order[j]; gtd += st.cY[b] * st.Yg[b] + st.cS[b] * st.Sg[b]; }
    st.gtd = gtd;
    st.prev_loss = st.loss;
    st.t = (st.n_iter_total == 1) ? fmin(1.0, 1.0 / st.g_l1) * P.lr : P.lr;     // lbfgsnew.py:677-680
}

// pass 2: d = sum of basis vectors, g_prev <- g, chi += t d, |d|_1
__global__ void __launch_bounds__(PAD_THREADS) k_lbfgs_pass2(size_t n, const OptState* __restrict__ stp, const double* __restrict__ g,
                                                           double* __restrict__ prev_g, double* __restrict__ d,
                                                           double* __restrict__ chi, const double* __restrict__ Sh,
                                                           const double* __restrict__ Yh, double* __restrict__ partials) {
    if (!stp->do_move) return;
    const int k = stp->k;
    const double t = stp->t, cg = stp->cg;
    double cS[OPT_SLOTS], cY[OPT_SLOTS];
    bool used[OPT_SLOTS];
#pragma unroll
    for (int a = 0; a < OPT_SLOTS; ++a) { cS[a] = stp->cS[a]; cY[a] = stp->cY[a]; used[a] = false; }
    for (int i = 0; i < k; ++i) {
        const int a = stp->order[i];
#pragma unroll
        for (int b = 0; b < OPT_SLOTS; ++b) if (b == a) used[b] = true;
    }
    double acc[1] = {0.0};
    const size_t stride = (size_t)gridDim.x * PAD_THREADS;
    for (size_t i = (size_t)blockIdx.x * PAD_THREADS + threadIdx.x; i < n; i += stride) {
        const double gi = g[i], xi = chi[i];
        double sa[OPT_SLOTS], ya[OPT_SLOTS];
#pragma unroll
        for (int a = 0; a < OPT_SLOTS; ++a) {      // all loads first (see pass 1)
            sa[a] = used[a] ? Sh[(size_t)a * n + i] : 0.0;
            ya[a] = used[a] ? Yh[(size_t)a * n + i] : 0.0;
        }
        double di = cg * gi;
#pragma unroll
        for (int a = 0; a < OPT_SLOTS; ++a)
            if (used[a]) di += cS[a] * sa[a] + cY[a] * ya[a];
        d[i] = di;
        prev_g[i] = gi;
        chi[i] = xi + t * di;
        acc[0] += fabs(di);
    }
    block_reduce_store<1>(acc, partials);
}

__global__ void __launch_bounds__(PAD_THREADS) k_lbfgs_after_move(OptState* stp, OptParams P, const double* __restrict__ partials,
                                                                int nblocks, const double* __restrict__ totals, double* trace) {
    __shared__ double sums[1];
    if (!stp->do_move) return;
    gather_sums(partials, nblocks, 1, totals, sums);
    if (threadIdx.x != 0) return;
    OptState& st = *stp;
    st.d_l1 = sums[0];
    if (st.it == P.max_iter) {            // last inner iteration: no re-evaluation (lbfgsnew.py:716, :735)
        end_step(st, P, trace);
        st.phase = 0;
    }
}

// ------------------------------------------------------------------------------------------------
//  TPGD (two_point_gradient_descent.py:36-61)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(PAD_THREADS) k_tpgd_dots(size_t n, const OptState* __restrict__ stp, const double* __restrict__ chi,
                                                         const double* __restrict__ g, double* __restrict__ x_prev,
                                                         double* __restrict__ g_prev, double* __restrict__ partials) {
    if (!stp->do_move) return;
    const bool first = stp->tp_iter == 0;
    double acc[2] = {0.0, 0.0};
    const size_t stride = (size_t)gridDim.x * PAD_THREADS;
    for (size_t i = (size_t)blockIdx.x * PAD_THREADS + threadIdx.x; i < n; i += stride) {
        const double x = chi[i], gi = g[i];
        if (!first) {
            const double dx = x - x_prev[i], dg = gi - g_prev[i];
            acc[0] += dx * dx;
            acc[1] += dx * dg;
        }
        x_prev[i] = x;
        g_prev[i] = gi;
    }
    block_reduce_store<2>(acc, partials);
}

__global__ void __launch_bounds__(PAD_THREADS) k_tpgd_alpha(OptState* stp, OptParams P, const double* __restrict__ partials,
                                                          int nblocks, const double* __restrict__ totals, double* trace) {
    __shared__ double sums[2];
    if (!stp->do_move) return;
    gather_sums(partials, nblocks, 2, totals, sums);
    if (threadIdx.x != 0) return;
    OptState& st = *stp;
    double alpha = P.lr;
    if (st.tp_iter != 0 && sums[1] != 0.0) {
        const double bb = sums[0] / sums[1];
        if (bb > 0.0) alpha = bb;
    }
    st.tp_alpha = alpha;
    st.tp_iter++;
    end_step(st, P, trace);        // the step is taken even on the iteration that converges (as in the reference)
}

__global__ void __launch_bounds__(PAD_THREADS) k_tpgd_update(size_t n, const OptState* __restrict__ stp, double* __restrict__ chi,
                                                           const double* __restrict__ g) {
    if (!stp->do_move) return;
    const double a = stp->tp_alpha;
    const size_t stride = (size_t)gridDim.x * PAD_THREADS;
    for (size_t i = (size_t)blockIdx.x * PAD_THREADS + threadIdx.x; i < n; i += stride) chi[i] -= a * g[i];
}

__global__ void k_set_Eprev(OptState* st, const double* E) { st->E_prev_eV = E[0] * kEvPerHa; }

}  // namespace

// =================================================================================================
//  fused evaluation of a term list
// =================================================================================================
extern "C" int pad_eval_total(pad_plan* p, const pad_terms* T, const double* den, const double* v_ext, double* E_out,
                              double* v_out, void* stream) {
    if (!p || !T || !den) { pad_set_error("pad_eval_total: null argument"); return PAD_ERR_ARG; }
    int acc = 0;
    if (T->kinetic == 2 && v_out && g_pad_fast_fft && g_pad_fuse_terms && pad_wgc99_total_supported(p) && !(T->local_mask & PAD_LOCAL_TF) &&
        (T->local_mask || T->hartree)) {
        // ONE pass over the grid for the whole list: the local terms ride on the WGC99 mid pass, the Hartree term is a
        // fourth field of its second transform batch (csrc/fftz.cu)
        if ((T->local_mask & PAD_LOCAL_IONEL) && !v_ext) { pad_set_error("pad_eval_total: IonElectron needs v_ext"); return PAD_ERR_ARG; }
        pad_wgc_extras ex{T->local_mask, v_ext, T->hartree};
        PAD_TRY(pad_eval_wgc99_ex(p, den, T->alpha, T->beta, T->gamma, T->kappa, E_out, v_out, 0, stream, &ex));
        if (T->pbe) PAD_TRY(pad_eval_pbe(p, den, T->pbe, E_out, v_out, 1, stream));
        return PAD_OK;
    }
    if (T->local_mask) {
        PAD_TRY(pad_eval_local(p, den, v_ext, T->local_mask, E_out, v_out, acc, stream));
        acc = 1;
    }
    if (T->hartree) {
        PAD_TRY(pad_eval_hartree(p, den, E_out, v_out, acc, stream));
        acc = 1;
    }
    if (T->kinetic == 1) {
        PAD_TRY(pad_eval_wt(p, den, T->alpha, T->beta, T->kinetic_parts, E_out, v_out, acc, stream));
        acc = 1;
    } else if (T->kinetic == 2) {
        PAD_TRY(pad_eval_wgc99(p, den, T->alpha, T->beta, T->gamma, T->kappa, E_out, v_out, acc, stream));
        acc = 1;
    } else if (T->kinetic == 3) {
        // pad_eval_hc adds into v_out, so the potential must exist before it is called
        if (!acc && v_out) PAD_CUDA(cudaMemsetAsync(v_out, 0, sizeof(double) * p->N, (cudaStream_t)stream));
        if (!acc && E_out) PAD_CUDA(cudaMemsetAsync(E_out, 0, sizeof(double), (cudaStream_t)stream));
        PAD_TRY(pad_eval_hc(p, den, T->hc_variant, T->hc_p0, T->hc_p1, T->beta, T->kappa, T->hc_geometric, T->hc_table_dev,
                            T->hc_n_eta, E_out, v_out, 1, nullptr, stream));
        acc = 1;
    } else if (T->kinetic == 4) {
        // PBE rides along: one gradient / divergence round trip carries both energy densities and both w fields
        const pad_semilocal_args P{T->sl_variant, T->sl_p0, T->sl_p1, T->pbe};
        PAD_TRY(pad_eval_semilocal_ex(p, den, P, E_out, v_out, acc, stream));
        acc = 1;
    }
    if (T->pbe && T->kinetic != 4) {
        PAD_TRY(pad_eval_pbe(p, den, T->pbe, E_out, v_out, acc, stream));
        acc = 1;
    }
    if (!acc) { pad_set_error("pad_eval_total: empty term list"); return PAD_ERR_ARG; }
    return PAD_OK;
}

// =================================================================================================
//  chi-parametrisation
// =================================================================================================
template <int NRED, class F>
static void launch_ew_opt(pad_plan* p, cudaStream_t s, F f) {
    ew_kernel<NRED, F><<<pad_grid_for(p->N), PAD_THREADS, 0, s>>>(p->N, f, p->partials);
    ++g_pad_launches;
}

static void finalize_sums(pad_plan* p, cudaStream_t s, int nterms, double* sums_out) {
    FinalizeArgs a;
    a.nblocks = pad_grid_for(p->N);
    a.nterms = nterms;
    a.accumulate = 0;
    for (int t = 0; t < PAD_MAX_RED; ++t) a.coef[t] = 0.0;
    a.sums_out = sums_out;
    a.E_out = nullptr;
    pad_launch_finalize(p, a, s);
}

extern "C" int pad_chi_to_density(pad_plan* p, const double* chi, double n_elec, double* den_out, void* stream) {
    if (!p || !chi || !den_out) { pad_set_error("pad_chi_to_density: null argument"); return PAD_ERR_ARG; }
    PAD_CUDA(cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    double* scal = p->scal;
    const double dV = p->dV;
    launch_ew_opt<1>(p, s, [=] __device__(size_t i, double(&acc)[1]) { const double c = chi[i]; acc[0] += c * c; });
    finalize_sums(p, s, 1, scal + S_TMP0 + 4);
    launch_ew_opt<0>(p, s, [=] __device__(size_t i, double(&)[1]) {
        const double c = chi[i];
        den_out[i] = (n_elec / (scal[S_TMP0 + 4] * dV)) * c * c;
    });
    PAD_CUDA(cudaGetLastError());
    return PAD_OK;
}

// projected gradient (system.py:850-853) + its reductions: |g|_1, g.g (sums) and max|dE/dchi|, max|mu - v|
__global__ void __launch_bounds__(PAD_THREADS) k_chi_project(size_t n, const double* __restrict__ chi, const double* __restrict__ v,
                                                           double n_elec, double dV, const double* __restrict__ sum_chi2,
                                                           const double* __restrict__ sum_vrho, double* __restrict__ grad_out,
                                                           unsigned long long* max_bits, const int* done_flag,
                                                           double* __restrict__ partials) {
    const double scale = n_elec / (sum_chi2[0] * dV);
    const double mu = sum_vrho[0] * dV / n_elec;
    const bool write = !done_flag || !*done_flag;
    double acc[2] = {0.0, 0.0};
    double m_g = 0.0, m_e = 0.0;
    const size_t stride = (size_t)gridDim.x * PAD_THREADS;
    for (size_t i = (size_t)blockIdx.x * PAD_THREADS + threadIdx.x; i < n; i += stride) {
        const double dv = v[i] - mu;
        const double gd = scale * 2.0 * chi[i] * dv;          // delta E / delta chi
        const double gi = gd * dV;                            // dE / d chi_ijk
        if (write) grad_out[i] = gi;
        acc[0] += fabs(gi);
        acc[1] += gi * gi;
        m_g = fmax(m_g, fabs(gd));
        m_e = fmax(m_e, fabs(dv));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        m_g = fmax(m_g, __shfl_xor_sync(0xffffffffu, m_g, o));
        m_e = fmax(m_e, __shfl_xor_sync(0xffffffffu, m_e, o));
    }
    if ((threadIdx.x & 31) == 0) {
        // non-negative doubles order like their bit patterns
        atomicMax(&max_bits[0], (unsigned long long)__double_as_longlong(m_g));
        atomicMax(&max_bits[1], (unsigned long long)__double_as_longlong(m_e));
    }
    block_reduce_store<2>(acc, partials);
}

// shared by the public entry point and the optimiser: needs sum chi^2 in *sum_chi2
static int chi_project_impl(pad_plan* p, cudaStream_t s, const double* chi, const double* den, const double* v,
                            double n_elec, const double* sum_chi2, double* sum_vrho, double* grad_out,
                            unsigned long long* max_bits /*2*/, const int* done_flag) {
    launch_ew_opt<1>(p, s, [=] __device__(size_t i, double(&acc)[1]) { acc[0] += v[i] * den[i]; });
    finalize_sums(p, s, 1, sum_vrho);
    k_chi_project<<<pad_grid_for(p->N), PAD_THREADS, 0, s>>>(p->N, chi, v, n_elec, p->dV, sum_chi2, sum_vrho, grad_out,
                                                            max_bits, done_flag, p->partials);
    ++g_pad_launches;
    PAD_CUDA(cudaGetLastError());
    return PAD_OK;
}

__global__ void k_pack_stats(const double* partials_sums, const unsigned long long* bits, double* out) {
    out[0] = partials_sums[0];
    out[1] = partials_sums[1];
    out[2] = bits_to_double(bits[0]);
    out[3] = bits_to_double(bits[1]);
}

extern "C" int pad_chi_project(pad_plan* p, const double* chi, const double* den, const double* v, double n_elec,
                               double* grad_out, double* stats_out, void* stream) {
    if (!p || !chi || !den || !v || !grad_out) { pad_set_error("pad_chi_project: null argument"); return PAD_ERR_ARG; }
    PAD_CUDA(cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    double* scal = p->scal;
    launch_ew_opt<1>(p, s, [=] __device__(size_t i, double(&acc)[1]) { const double c = chi[i]; acc[0] += c * c; });
    finalize_sums(p, s, 1, scal + S_TMP0 + 4);
    unsigned long long* bits = reinterpret_cast<unsigned long long*>(scal + S_TMP0 + 6);
    PAD_CUDA(cudaMemsetAsync(bits, 0, 2 * sizeof(unsigned long long), s));
    PAD_TRY(chi_project_impl(p, s, chi, den, v, n_elec, scal + S_TMP0 + 4, scal + S_TMP0 + 5, grad_out, bits, nullptr));
    if (stats_out) {
        PAD_TRY(pad_allreduce_max_bits(p, bits, 2, s));
        finalize_sums(p, s, 2, scal + S_E_PARTS);
        k_pack_stats<<<1, 1, 0, s>>>(scal + S_E_PARTS, bits, stats_out);
        ++g_pad_launches;
    }
    PAD_CUDA(cudaGetLastError());
    return PAD_OK;
}

// =================================================================================================
//  device-resident optimiser
// =================================================================================================
struct pad_denopt {
    pad_plan* plan;
    pad_terms terms;
    OptParams P;
    OptState* st;            // device
    OptState* host_ring;     // pinned, OPT_RING entries
    cudaEvent_t ev[OPT_RING];
    double *chi, *g, *prev_g, *d, *den, *v, *Sh, *Yh, *x_prev;
    double* partials;        // OPT_NACC * PAD_MAX_BLOCKS
    double* trace;           // device, 4 * n_maxiter
    double* E_dev;
    size_t bytes;
};

extern "C" int pad_denopt_create(pad_denopt** out, pad_plan* plan, const pad_terms* terms, const pad_denopt_params* prm) {
    if (!out || !plan || !terms || !prm) { pad_set_error("pad_denopt_create: null argument"); return PAD_ERR_ARG; }
    if (prm->method != 0 && prm->method != 1) { pad_set_error("pad_denopt_create: method must be 0 (LBFGS) or 1 (TPGD)"); return PAD_ERR_ARG; }
    if (prm->history < 1 || prm->history > OPT_M) { pad_set_error("pad_denopt_create: history must be in 1..%d", OPT_M); return PAD_ERR_ARG; }
    if (prm->conv_target < 0 || prm->conv_target > 2) { pad_set_error("pad_denopt_create: bad conv_target"); return PAD_ERR_ARG; }
    PAD_CUDA(cudaSetDevice(plan->device));
    pad_denopt* o = new pad_denopt();
    memset(o, 0, sizeof(*o));
    o->plan = plan;
    o->terms = *terms;
    OptParams& P = o->P;
    P.n_elec = prm->n_elec; P.ntol = prm->ntol; P.lr = prm->step_size; P.tol_grad = prm->tolerance_grad;
    P.tol_change = prm->tolerance_change; P.dV = plan->dV; P.n_conv = prm->n_conv_cond_count; P.method = prm->method;
    P.n_maxiter = prm->n_maxiter; P.conv_target = prm->conv_target; P.history = prm->history;
    P.max_iter = prm->max_iter; P.max_eval = prm->max_iter * 5 / 4;
    const size_t N = plan->N, vb = sizeof(double) * N;
    const int nvec = 6 + (P.method == 0 ? 2 * OPT_SLOTS : 1);
    double* pool = nullptr;
    const size_t Np = (N + 31) & ~(size_t)31;      // 256-byte aligned vectors: den / v are cuFFT operands
    PAD_CUDA(cudaMalloc(&pool, vb * nvec + sizeof(double) * 32 * 8));
    o->bytes = vb * nvec;
    o->chi = pool; o->g = pool + Np; o->prev_g = pool + 2 * Np; o->d = pool + 3 * Np; o->den = pool + 4 * Np; o->v = pool + 5 * Np;
    if (P.method == 0) { o->Sh = pool + 6 * Np; o->Yh = o->Sh + (size_t)OPT_SLOTS * N; o->x_prev = nullptr; }
    else { o->x_prev = pool + 6 * Np; }
    PAD_CUDA(cudaMalloc(&o->partials, sizeof(double) * OPT_NACC * PAD_MAX_BLOCKS));
    PAD_CUDA(cudaMalloc(&o->st, sizeof(OptState)));
    PAD_CUDA(cudaMalloc(&o->trace, sizeof(double) * 4 * (size_t)(prm->n_maxiter > 0 ? prm->n_maxiter : 1)));
    PAD_CUDA(cudaMalloc(&o->E_dev, sizeof(double)));
    PAD_CUDA(cudaMallocHost(&o->host_ring, sizeof(OptState) * OPT_RING));
    for (int i = 0; i < OPT_RING; ++i) PAD_CUDA(cudaEventCreateWithFlags(&o->ev[i], cudaEventDisableTiming));
    *out = o;
    return PAD_OK;
}

extern "C" int pad_denopt_destroy(pad_denopt* o) {
    if (!o) return PAD_OK;
    cudaSetDevice(o->plan->device);
    cudaFree(o->chi);
    cudaFree(o->partials);
    cudaFree(o->st);
    cudaFree(o->trace);
    cudaFree(o->E_dev);
    cudaFreeHost(o->host_ring);
    for (int i = 0; i < OPT_RING; ++i) cudaEventDestroy(o->ev[i]);
    delete o;
    return PAD_OK;
}

// slab plans: per-block partials -> `nterms` totals in the plan's communication scratch -> ONE all-reduce over the
// ranks; returns the pointer the following transition kernel reads its sums from (nullptr on single-GPU plans, where
// that kernel reduces the partials itself).  The all-reduce is enqueued unconditionally -- every rank takes the same
// branches because every scalar the state machine sees has been all-reduced.
static int slab_reduce(pad_plan* p, const double* partials, int nterms, cudaStream_t s, const double** totals) {
    *totals = nullptr;
    if (!p->dist) return PAD_OK;
    k_reduce_to<<<1, PAD_THREADS, 0, s>>>(partials, pad_grid_for(p->N), nterms, p->comm_scratch);
    ++g_pad_launches;
    PAD_TRY(pad_slab_comm(p, PAD_COMM_ALL_REDUCE, nterms, s));
    *totals = p->comm_scratch;
    return PAD_OK;
}

// one closure: chi -> n -> E, v -> projected gradient (+ its reductions, left in o->partials rows 0,1)
static int enqueue_closure(pad_denopt* o, const double* v_ext, cudaStream_t s) {
    pad_plan* p = o->plan;
    OptState* st = o->st;
    const double n_elec = o->P.n_elec, dV = p->dV;
    const double* chi = o->chi;
    double* den = o->den;
    launch_ew_opt<1>(p, s, [=] __device__(size_t i, double(&acc)[1]) { const double c = chi[i]; acc[0] += c * c; });
    finalize_sums(p, s, 1, &st->sum_chi2);
    launch_ew_opt<0>(p, s, [=] __device__(size_t i, double(&)[1]) {
        if (st->done) return;                                   // keep the density of the last real closure
        const double c = chi[i];
        den[i] = (n_elec / (st->sum_chi2 * dV)) * c * c;
    });
    PAD_TRY(pad_eval_total(p, &o->terms, den, v_ext, &st->E, o->v, (void*)s));
    k_reset_max<<<1, 1, 0, s>>>(st);
    ++g_pad_launches;
    PAD_TRY(chi_project_impl(p, s, chi, den, o->v, n_elec, &st->sum_chi2, &st->sum_vrho, o->g, &st->max_dEdchi_bits, &st->done));
    PAD_TRY(pad_allreduce_max_bits(p, &st->max_dEdchi_bits, 2, s));       // max_dEdchi_bits, max_euler_bits are adjacent
    return PAD_OK;
}

extern "C" int pad_denopt_run(pad_denopt* o, double* den_inout, const double* v_ext, pad_denopt_result* res,
                              double* trace_host, void* stream) {
    if (!o || !den_inout || !res) { pad_set_error("pad_denopt_run: null argument"); return PAD_ERR_ARG; }
    pad_plan* p = o->plan;
    PAD_CUDA(cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    o->P.dV = p->dV;
    const OptParams P = o->P;
    const size_t N = p->N;
    const int grid = pad_grid_for(N);
    OptState* st = o->st;
    PAD_CUDA(cudaMemsetAsync(st, 0, sizeof(OptState), s));
    // E_prev = energy of the starting density (system.py:856); chi = sqrt(n) (system.py:820)
    PAD_TRY(pad_eval_total(p, &o->terms, den_inout, v_ext, o->E_dev, nullptr, stream));
    k_set_Eprev<<<1, 1, 0, s>>>(st, o->E_dev);
    double* chi = o->chi;
    launch_ew_opt<0>(p, s, [=] __device__(size_t i, double(&)[1]) { chi[i] = sqrt(den_inout[i]); });
    PAD_CUDA(cudaGetLastError());

    const bool debug = getenv("PAD_DENOPT_DEBUG") != nullptr;       // per-tick state dump on stderr
    const long long max_ticks = (long long)P.n_maxiter * (P.method == 0 ? P.max_iter : 1) + OPT_LOOKAHEAD + 2;
    long long tick = 0;
    bool done = false;
    for (; tick < max_ticks && !done; ++tick) {
        if (tick >= OPT_LOOKAHEAD) {
            const long long j = tick - OPT_LOOKAHEAD;
            PAD_CUDA(cudaEventSynchronize(o->ev[j % OPT_RING]));
            if (debug) {
                const OptState& h = o->host_ring[j % OPT_RING];
                fprintf(stderr, "[denopt] tick %lld closures %d outer %d it %d phase %d E %.12f |g|1 %.6e gg %.6e k %d H %.6e t %.3e gtd %.6e |d|1 %.6e\n",
                        j, h.closures, h.outer_iter, h.it, h.phase, h.E, h.g_l1, h.gg, h.k, h.H, h.t, h.gtd, h.d_l1);
            }
            if (o->host_ring[j % OPT_RING].done) { done = true; break; }
        }
        const double* tot = nullptr;
        PAD_TRY(enqueue_closure(o, v_ext, s));
        PAD_TRY(slab_reduce(p, p->partials, 2, s, &tot));
        k_after_closure<<<1, PAD_THREADS, 0, s>>>(st, P, p->partials, grid, tot, o->trace);
        if (P.method == 0) {
            k_lbfgs_pass1<<<grid, PAD_THREADS, 0, s>>>(N, st, o->g, o->prev_g, o->d, o->Sh, o->Yh, o->partials);
            PAD_TRY(slab_reduce(p, o->partials, OPT_NACC, s, &tot));       // all 5k+5 inner products in one all-reduce
            k_lbfgs_direction<<<1, PAD_THREADS, 0, s>>>(st, P, o->partials, grid, tot);
            k_lbfgs_pass2<<<grid, PAD_THREADS, 0, s>>>(N, st, o->g, o->prev_g, o->d, o->chi, o->Sh, o->Yh, p->partials);
            PAD_TRY(slab_reduce(p, p->partials, 1, s, &tot));
            k_lbfgs_after_move<<<1, PAD_THREADS, 0, s>>>(st, P, p->partials, grid, tot, o->trace);
            g_pad_launches += 5;
        } else {
            k_tpgd_dots<<<grid, PAD_THREADS, 0, s>>>(N, st, o->chi, o->g, o->x_prev, o->prev_g, p->partials);
            PAD_TRY(slab_reduce(p, p->partials, 2, s, &tot));
            k_tpgd_alpha<<<1, PAD_THREADS, 0, s>>>(st, P, p->partials, grid, tot, o->trace);
            k_tpgd_update<<<grid, PAD_THREADS, 0, s>>>(N, st, o->chi, o->g);
            g_pad_launches += 4;
        }
        PAD_CUDA(cudaGetLastError());
        PAD_CUDA(cudaMemcpyAsync(&o->host_ring[tick % OPT_RING], st, sizeof(OptState), cudaMemcpyDeviceToHost, s));
        PAD_CUDA(cudaEventRecord(o->ev[tick % OPT_RING], s));
    }
    PAD_CUDA(cudaStreamSynchronize(s));
    OptState fin;
    PAD_CUDA(cudaMemcpy(&fin, st, sizeof(OptState), cudaMemcpyDeviceToHost));
    PAD_CUDA(cudaMemcpyAsync(den_inout, o->den, sizeof(double) * N, cudaMemcpyDeviceToDevice, s));
    if (trace_host && fin.outer_iter > 0)
        PAD_CUDA(cudaMemcpyAsync(trace_host, o->trace, sizeof(double) * 4 * (size_t)fin.outer_iter, cudaMemcpyDeviceToHost, s));
    PAD_CUDA(cudaStreamSynchronize(s));
    res->iterations = fin.outer_iter;
    res->converged = fin.converged;
    res->closures = fin.closures;
    res->energy = fin.E;
    res->last_dE_eV = fin.last_dE;
    res->last_dEdchi = fin.last_dEdchi;
    res->last_euler = fin.last_euler;
    if (!fin.done) { pad_set_error("pad_denopt_run: tick budget exhausted before the stop rule fired"); return PAD_ERR_ARG; }
    return PAD_OK;
}
