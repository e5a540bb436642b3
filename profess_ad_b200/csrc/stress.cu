// Analytic stress of the native functionals:  sigma_ij = (1/vol) dE/d eps_ij  at fixed electron number (the density
// scales as 1/vol) -- what get_stress / System.__compute_stress obtain by autograd through box_vecs
// (functional_tools.py:73-100, system.py:927-935).  Formulas: tests/tools_for_tests.py:212-472 of the reference,
// restated over the half spectrum with weights w (1 on the self-conjugate planes, 2 elsewhere) and the plain
// "Nyquist made positive" wave vectors: for even multipliers the Hermitian symmetrisation drops out of the energy, for
// the gradient terms the strain acts on the real-space gradient as g -> (1 - eps) g exactly (tests/analytic_model.py
// checks every formula against autograd through box_vecs to 1e-14 on even, odd and skewed grids).
//
//   local (TF, LDA-x, PZ-c) : delta_ij (E - int v n) / vol
//   Hartree                 : sum_k w 4 pi |c_k|^2 k_i k_j / k^4  -  delta_ij E_H / vol
//   Weizsaecker             : - sum_k w |chi_k|^2 k_i k_j
//   Wang-Teter family NL    : pref sum_k w Re(a_k conj b_k) aux3(eta) (k_i k_j / k^2 - delta_ij / 3) - (2/3) delta_ij T_NL / vol
//   PBE                     : delta_ij mean(f - n f_n - 2 sigma f_sigma) - 2 mean(f_sigma g_i g_j)
//   semilocal kinetic (LKT, PG): delta_ij mean(e - n e_n - 2 sigma e_sigma - L e_L) - 2 mean(e_sigma g_i g_j)
//                             - 2 mean(e_L d_i d_j n),  the last as  2 sum_k w Re(conj(l_k) c_k) k_i k_j
//                             (l_k: coefficients of e_L; the strain derivative of -k^2 is 2 k_i k_j with the same k)
// (c_k, chi_k, a_k, b_k: Fourier coefficients, norm = 'forward', of n, sqrt n, n^alpha, n^beta.)
//   WangGovindCarter99 NL   : pad_stress_wgc99_nl (functionals.cu): same structure with the eta-derivatives of the four kernels;
//                             the derivative with the kernel regenerated for the strained cell (the reference's autograd
//                             with a fresh kernel; with a kernel cached at the same cell the reference silently drops the
//                             kernel's own eta-dependence, functionals.py:961-966)
//   HuangCarter / RevisedHuangCarter NL : pad_stress_hc_nl (hc.cu)
#include "common.cuh"
#include "xc.cuh"

namespace {

constexpr double k3Pi2 = 29.608813203268074;

__global__ void k_stress_add(const double* __restrict__ sums, double c_iso, double c_t, double* __restrict__ sig) {
    const double iso = c_iso * sums[0];
    sig[0] += c_t * sums[1] + iso;
    sig[4] += c_t * sums[2] + iso;
    sig[8] += c_t * sums[3] + iso;
    sig[1] += c_t * sums[4]; sig[3] += c_t * sums[4];
    sig[2] += c_t * sums[5]; sig[6] += c_t * sums[5];
    sig[5] += c_t * sums[6]; sig[7] += c_t * sums[6];
}

__device__ __forceinline__ void add_tensor(double (&acc)[7], double t, double kx, double ky, double kz) {
    acc[1] += t * kx * kx; acc[2] += t * ky * ky; acc[3] += t * kz * kz;
    acc[4] += t * kx * ky; acc[5] += t * kx * kz; acc[6] += t * ky * kz;
}

template <class F>
void launch_n(pad_plan* p, cudaStream_t s, F f) {
    ew_kernel<7, F><<<pad_grid_for(p->N), PAD_THREADS, 0, s>>>(p->N, f, p->partials);
    ++g_pad_launches;
}

template <class F>
void launch_k(pad_plan* p, cudaStream_t s, F f) {
    ew_kernel<7, F><<<pad_grid_for(p->Nk), PAD_THREADS, 0, s>>>(p->Nk, f, p->partials);
    ++g_pad_launches;
}

}  // namespace

int pad_stress_accumulate(pad_plan* p, cudaStream_t s, int nblocks, double c_iso, double c_t, double* sig) {
    FinalizeArgs a;
    a.nblocks = nblocks;
    a.nterms = 7;
    a.accumulate = 0;
    for (int t = 0; t < PAD_MAX_RED; ++t) a.coef[t] = 0.0;
    a.sums_out = p->scal + S_E_PARTS;
    a.E_out = nullptr;
    pad_launch_finalize(p, a, s);
    k_stress_add<<<1, 1, 0, s>>>(p->scal + S_E_PARTS, c_iso, c_t, sig);
    ++g_pad_launches;
    PAD_CUDA(cudaGetLastError());
    return PAD_OK;
}

extern "C" int pad_stress_terms(pad_plan* p, const pad_terms* T, const double* den, double* stress_out, void* stream) {
    if (!p || !T || !den || !stress_out) { pad_set_error("pad_stress_terms: null argument"); return PAD_ERR_ARG; }
    PAD_CUDA(cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    const KGeom geom = p->geom;
    const double inv_n = geom.inv_n;
    const int gN = pad_grid_for(p->N), gK = pad_grid_for(p->Nk);
    PAD_CUDA(cudaMemsetAsync(stress_out, 0, sizeof(double) * 9, s));
    cufftDoubleComplex* C[3];
    double* R[4];
    for (int i = 0; i < 3; ++i) PAD_TRY(pad_get_cbuf(p, i, &C[i]));

    // ---- local terms (IonElectron is handled by pad_ion_stress) ------------------------------------------
    // WangGovindCarter99 = TF + vW + its own non-local term (functionals.py:983-985)
    // HuangCarter / RevisedHuangCarter = TF + vW + their non-local term too (functionals.py:1267-1269)
    int parts = T->kinetic == 1 ? T->kinetic_parts : (T->kinetic == 2 || T->kinetic == 3 ? (PAD_PART_TF | PAD_PART_VW) : 0);
    // ThomasFermi can appear as a term of its own and inside a Wang-Teter style functional: count both
    const double tfc = ((T->local_mask & PAD_LOCAL_TF) ? 1.0 : 0.0) + ((parts & PAD_PART_TF) ? 1.0 : 0.0);
    const bool tf = tfc != 0.0;
    const bool ldax = T->local_mask & PAD_LOCAL_LDAX, pzc = T->local_mask & PAD_LOCAL_PZC;
    if (tf || ldax || pzc) {
        launch_n(p, s, [=] __device__(size_t i, double(&acc)[7]) {
            const double n = den[i], c = cbrt(n);
            double e = 0.0, v = 0.0;
            if (tf) { e += tfc * kCTF * n * c * c; v += tfc * (5.0 / 3.0) * kCTF * c * c; }
            if (ldax) { e += kCX * n * c; v += (4.0 / 3.0) * kCX * c; }
            if (pzc) { PZ r = pz_correlation(n, c); e += r.e; v += r.v; }
            acc[0] += e - v * n;
        });
        PAD_TRY(pad_stress_accumulate(p, s, gN, inv_n, 0.0, stress_out));
    }

    // ---- Hartree ------------------------------------------------------------------------------------------
    if (T->hartree) {
        PAD_TRY(pad_fft_forward(p, den, C[0], s));
        const cufftDoubleComplex* Rh = C[0];
        launch_k(p, s, [=] __device__(size_t i, double(&acc)[7]) {
            const KPoint k = make_kpoint(geom, (uint32_t)i);
            const double k2 = k.kx * k.kx + k.ky * k.ky + k.kz * k.kz;
            if (k2 == 0.0) return;
            const cufftDoubleComplex r = Rh[i];
            const bool edge = k.j2 == 0 || (geom.e2 && k.j2 == geom.n2 / 2);
            const double a = (edge ? 1.0 : 2.0) * 4.0 * kPi * (r.x * r.x + r.y * r.y) * inv_n * inv_n / k2;
            acc[0] -= 0.5 * a;
            add_tensor(acc, a / k2, k.kx, k.ky, k.kz);
        });
        PAD_TRY(pad_stress_accumulate(p, s, gK, 1.0, 1.0, stress_out));
    }

    // ---- Weizsaecker ----------------------------------------------------------------------------------------
    if (parts & PAD_PART_VW) {
        PAD_TRY(pad_get_rbuf(p, 0, &R[0]));
        double* chi = R[0];
        ew_kernel<0><<<gN, PAD_THREADS, 0, s>>>(p->N, [=] __device__(size_t i, double(&)[1]) { chi[i] = sqrt(den[i]); }, p->partials);
        ++g_pad_launches;
        PAD_TRY(pad_fft_forward(p, chi, C[0], s));
        const cufftDoubleComplex* X = C[0];
        launch_k(p, s, [=] __device__(size_t i, double(&acc)[7]) {
            const KPoint k = make_kpoint(geom, (uint32_t)i);
            const cufftDoubleComplex r = X[i];
            const bool edge = k.j2 == 0 || (geom.e2 && k.j2 == geom.n2 / 2);
            add_tensor(acc, -(edge ? 1.0 : 2.0) * (r.x * r.x + r.y * r.y) * inv_n * inv_n, k.kx, k.ky, k.kz);
        });
        PAD_TRY(pad_stress_accumulate(p, s, gK, 0.0, 1.0, stress_out));
    }

    // ---- non-local term of the Wang-Teter family ---------------------------------------------------------------
    if (T->kinetic == 2) PAD_TRY(pad_stress_wgc99_nl(p, den, T->alpha, T->beta, T->gamma, T->kappa, stress_out, s));
    if (T->kinetic == 3)
        PAD_TRY(pad_stress_hc_nl(p, den, T->hc_variant, T->hc_p0, T->hc_p1, T->beta, T->kappa, T->hc_geometric, T->hc_table_dev, T->hc_n_eta,
                                 stress_out, s));
    if (parts & PAD_PART_NL) {
        const double alpha = T->alpha, beta = T->beta;
        PAD_TRY(pad_get_rbuf(p, 0, &R[0]));
        double* pw = R[0];
        double* scal = p->scal;
        {   // n0 = N_elec / vol from the density itself (functionals.py:646-647)
            ew_kernel<1><<<gN, PAD_THREADS, 0, s>>>(p->N, [=] __device__(size_t i, double(&acc)[1]) { acc[0] += den[i]; }, p->partials);
            ++g_pad_launches;
            FinalizeArgs a;
            a.nblocks = gN; a.nterms = 1; a.accumulate = 0;
            for (int t = 0; t < PAD_MAX_RED; ++t) a.coef[t] = 0.0;
            a.sums_out = scal + S_SUM_RHO; a.E_out = nullptr;
            pad_launch_finalize(p, a, s);
        }
        ew_kernel<0><<<gN, PAD_THREADS, 0, s>>>(p->N, [=] __device__(size_t i, double(&)[1]) { pw[i] = exp(alpha * log(den[i])); }, p->partials);
        PAD_TRY(pad_fft_forward(p, pw, C[1], s));
        const cufftDoubleComplex *A = C[1], *B = C[1];
        if (alpha != beta) {
            ew_kernel<0><<<gN, PAD_THREADS, 0, s>>>(p->N, [=] __device__(size_t i, double(&)[1]) { pw[i] = exp(beta * log(den[i])); }, p->partials);
            PAD_TRY(pad_fft_forward(p, pw, C[2], s));
            B = C[2];
            ++g_pad_launches;
        }
        ++g_pad_launches;
        launch_k(p, s, [=] __device__(size_t i, double(&acc)[7]) {
            const KPoint k = make_kpoint(geom, (uint32_t)i);
            const double k2 = k.kx * k.kx + k.ky * k.ky + k.kz * k.kz;
            if (k2 == 0.0) return;
            const double n0 = scal[S_SUM_RHO] * inv_n;
            const double kF = cbrt(k3Pi2 * n0);
            const double pref = 0.5 * kPi * kPi / (alpha * beta) / exp((alpha + beta - 2.0) * log(n0)) / kF;
            const double kpref = kCTF * 5.0 / (9.0 * alpha * beta * exp((alpha + beta - 5.0 / 3.0) * log(n0)));
            const cufftDoubleComplex a = A[i], b = B[i];
            const bool edge = k.j2 == 0 || (geom.e2 && k.j2 == geom.n2 / 2);
            const double ab = (edge ? 1.0 : 2.0) * (a.x * b.x + a.y * b.y) * inv_n * inv_n;
            const double eta = sqrt(k2) / (2.0 * kF);
            double lind, aux3;
            if (eta == 1.0) {          // the reference pins G^{-1}(1) = 1/2 by assignment: no derivative through it
                lind = 0.5;
                aux3 = 6.0;
            } else {
                const double lg = log(fabs((1.0 + eta) / (1.0 - eta)));
                lind = 0.5 + (1.0 - eta * eta) / (4.0 * eta) * lg;
                aux3 = eta / (lind * lind) * (0.5 / eta - 0.25 * (1.0 + 1.0 / (eta * eta)) * lg) + 6.0 * eta * eta;
            }
            const double t = pref * ab * aux3;
            acc[0] -= t / 3.0 + (2.0 / 3.0) * kpref * (1.0 / lind - 3.0 * eta * eta - 1.0) * ab;
            add_tensor(acc, t / k2, k.kx, k.ky, k.kz);
        });
        PAD_TRY(pad_stress_accumulate(p, s, gK, 1.0, 1.0, stress_out));
    }

    // ---- PBE -------------------------------------------------------------------------------------------------------
    if (T->pbe) {
        for (int i = 0; i < 3; ++i) PAD_TRY(pad_get_rbuf(p, i, &R[i]));
        PAD_TRY(pad_gradient(p, den, R[0], R[1], R[2], stream));
        const double *Gx = R[0], *Gy = R[1], *Gz = R[2];
        const bool do_x = T->pbe & 1, do_c = T->pbe & 2;
        launch_n(p, s, [=] __device__(size_t i, double(&acc)[7]) {
            const double n = den[i], gx = Gx[i], gy = Gy[i], gz = Gz[i];
            const double sig = gx * gx + gy * gy + gz * gz;
            double f, f_rho, f_sig;
            pbe_point(n, sig, cbrt(n), do_x, do_c, f, f_rho, f_sig);
            acc[0] += f - n * f_rho - 2.0 * sig * f_sig;
            add_tensor(acc, -2.0 * f_sig, gx, gy, gz);
        });
        PAD_TRY(pad_stress_accumulate(p, s, gN, inv_n, inv_n, stress_out));
    }

    // ---- semilocal kinetic functionals -------------------------------------------------------------------------------
    if (T->kinetic == 4) {
        const bool lap = T->sl_variant == PAD_SEMILOCAL_PG;
        for (int i = 0; i < 4; ++i) PAD_TRY(pad_get_rbuf(p, i, &R[i]));
        PAD_TRY(pad_gradient(p, den, R[0], R[1], R[2], stream));
        if (lap) PAD_TRY(pad_laplacian(p, den, R[3], stream));
        const double *Gx = R[0], *Gy = R[1], *Gz = R[2];
        double* L = R[3];
        const int variant = T->sl_variant;
        const double p0 = T->sl_p0, p1 = T->sl_p1;
        launch_n(p, s, [=] __device__(size_t i, double(&acc)[7]) {
            const double n = den[i], gx = Gx[i], gy = Gy[i], gz = Gz[i];
            const double sig = gx * gx + gy * gy + gz * gz, l = lap ? L[i] : 0.0;
            double e, e_n, e_s, e_l;
            semilocal_kinetic_point(n, sig, l, variant, p0, p1, e, e_n, e_s, e_l);
            acc[0] += e - n * e_n - 2.0 * sig * e_s - l * e_l;
            add_tensor(acc, -2.0 * e_s, gx, gy, gz);
            if (lap) L[i] = e_l;
        });
        PAD_TRY(pad_stress_accumulate(p, s, gN, inv_n, inv_n, stress_out));
        if (lap) {
            PAD_TRY(pad_fft_forward(p, L, C[0], s));
            PAD_TRY(pad_fft_forward(p, den, C[1], s));
            const cufftDoubleComplex *El = C[0], *Nk = C[1];
            launch_k(p, s, [=] __device__(size_t i, double(&acc)[7]) {
                const KPoint k = make_kpoint(geom, (uint32_t)i);
                const cufftDoubleComplex a = El[i], b = Nk[i];
                const bool edge = k.j2 == 0 || (geom.e2 && k.j2 == geom.n2 / 2);
                add_tensor(acc, 2.0 * (edge ? 1.0 : 2.0) * (a.x * b.x + a.y * b.y) * inv_n * inv_n, k.kx, k.ky, k.kz);
            });
            PAD_TRY(pad_stress_accumulate(p, s, gK, 0.0, 1.0, stress_out));
        }
    }
    PAD_CUDA(cudaGetLastError());
    return PAD_OK;
}
