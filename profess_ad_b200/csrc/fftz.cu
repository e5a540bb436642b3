// Hand-written z-axis (contiguous axis) real<->half-complex FFT passes with the real-space
// elementwise work fused in, for power-of-two n2 in {128, 256, 512}.  The (x, y) axes are transformed by the
// strided passes of fft_strided.cuh (n0, n1 in {64, 128, 256, 512}; the reciprocal-space multiply fused into the x
// pass, the slab transposition carried by the y / x passes) -- or, for other (n0, n1) on single-GPU plans, by one
// batched 2-D cuFFT Z2Z plan -- over the padded half-spectrum layout
//      spec[x][y][nzp],  nzp = n2/2 + 8 (multiple of 8 complex = 128 B rows),  nzh = n2/2 + 1 used.
// This translation unit also holds everything that needs the table log / exp of fastmath.cuh: the WGC99 / Wang-Teter /
// Hartree / PBE pipelines, the fast local-term and PBE point kernels.
//
// Why: in the plain cuFFT pipeline every real-space pre/post kernel is a separate HBM round trip and
// the r2c/c2r pass runs at ~3.7 TB/s.  Here a warp owns 32/TPL lines; TPL lanes share one line:
// they load the line ONCE, generate every field that has to be transformed from it (e.g. n^beta,
// n^beta theta, n^beta theta^2/2, sqrt(n) for WGC99), run the M = n2/2 point packed complex FFT in
// registers (one warp-synchronous shared-memory exchange), do the real post-processing and write
// the half-spectrum lines.  The inverse pass mirrors it and ends in the real-space post-op (energy
// densities, potential assembly) without the fields ever touching HBM.
//
// Conventions match cuFFT: forward and inverse are unnormalised (the 1/N lives in the multipliers).
#include "common.cuh"
#include "fft_core.cuh"
#include "fft_strided.cuh"
#include "zy_pipe.cuh"
#include "fastmath.cuh"
#include "xc.cuh"

namespace {

constexpr double k3Pi2 = 29.608813203268074;

// ------------------------------------------------------------------------------------------------
//  twiddle table
// ------------------------------------------------------------------------------------------------
bool g_tw_ready[64] = {false};

int ensure_twiddles(int device) {
    if (g_tw_ready[device & 63]) return PAD_OK;
    static double2 host[FFT_TW_N];
    for (int j = 0; j < FFT_TW_N; ++j) {
        // exact symmetries first, so that the table is bit-symmetric
        const double a = -2.0 * kPi * (double)j / (double)FFT_TW_N;
        host[j].x = cos(a);
        host[j].y = sin(a);
    }
    host[0] = {1.0, 0.0};
    host[FFT_TW_N / 4] = {0.0, -1.0};
    host[FFT_TW_N / 2] = {-1.0, 0.0};
    host[3 * FFT_TW_N / 4] = {0.0, 1.0};
    PAD_CUDA(cudaMemcpyToSymbol(g_fft_tw, host, sizeof(host)));
    // fastmath.cuh tables, evaluated in long double
    static double2 hlog[128];
    static double hexp[64];
    for (int i = 0; i < 128; ++i) {
        const long double c = 1.0L + ((long double)i + 0.5L) / 128.0L;
        const double inv = (double)(1.0L / c);
        hlog[i].x = inv;
        hlog[i].y = (double)(-logl((long double)inv));
    }
    for (int j = 0; j < 64; ++j) hexp[j] = (double)exp2l((long double)j / 64.0L);
    PAD_CUDA(cudaMemcpyToSymbol(g_fm_log, hlog, sizeof(hlog)));
    PAD_CUDA(cudaMemcpyToSymbol(g_fm_exp, hexp, sizeof(hexp)));
    g_tw_ready[device & 63] = true;
    return PAD_OK;
}

// ------------------------------------------------------------------------------------------------
//  z-pass kernels.  TPL lanes share a line; each lane owns the 8 packed-complex points
//  n = t + TPL j (j < 8) of the line -- as FFT input AND as FFT output (line_fft8), so everything
//  that is per real-space point (staged inputs, the NF inverse results) lives in registers.
//
//  Every line slot (32 / TPL per warp) has its own shared-memory landing zone; the global inputs of the
//  slot's NEXT line are copied into it with cp.async as soon as the current line has consumed the
//  corresponding part, so the HBM latency is off the critical path although only 8 warps fit on an SM.
//  Steady state: G groups in flight per thread, the oldest one is the item needed next => wait_group<G-1>.
//
//  Shared memory per block: [ tw1: M cd | tw2: M cd ] + per line slot [ FFT scratch | landing zone ].
// ------------------------------------------------------------------------------------------------
template <int M, int TPL>
struct ZLayout {
    static constexpr int kTwBytes = 2 * M * 16;
    static constexpr int kScratch = 8 * (TPL + 1);                    // cd, line_fft8 exchange
    static constexpr int kSpecLine = M + 2;                           // cd per staged half-spectrum line (M + 1 used)
    static constexpr int kLinesPerWarp = 32 / TPL;
    __host__ __device__ static constexpr int inv_line_bytes(int nf, int nreal) { return (kScratch + nf * kSpecLine) * 16 + nreal * 2 * M * 8; }
    // streamed inverse pass: scratch | two spectral landing buffers (ring) | one density line
    __host__ __device__ static constexpr int stream_line_bytes(bool kden) { return (kScratch + 2 * kSpecLine) * 16 + (kden ? 2 * M * 8 : 0); }
    __host__ __device__ static constexpr int fwd_line_bytes(int nin) { return (kScratch > M + 1 ? kScratch : M + 2) * 16 + nin * 2 * M * 8; }
};

// tw1[e] = exp(-2 pi i e / M), tw2[e] = exp(-2 pi i e / (2 M)), e < M
template <int M>
__device__ __forceinline__ void load_twiddles(cd* tw1, cd* tw2) {
    for (int e = threadIdx.x; e < M; e += blockDim.x) {
        const double2 w = g_fft_tw[e * (FFT_TW_N / M)];
        tw1[e] = cd{w.x, w.y};
        const double2 w2 = g_fft_tw[e * (FFT_TW_N / (2 * M))];
        tw2[e] = cd{w2.x, w2.y};
    }
    fm_load_tables();          // log / exp tables of fastmath.cuh (ends with __syncthreads)
}

// forward: field F generated from the staged values, packed FFT, real post-processing, store
template <int M, int TPL, int F, class Gen>
__device__ __forceinline__ void zfwd_field(const Gen& gen, const double (&sa)[Gen::NST][8], const double (&sb)[Gen::NST][8],
                                           cd* S, const cd* tw1, const cd* tw2, int t, cd* __restrict__ out, bool live) {
    constexpr int NST = Gen::NST;
    cd v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        double a[NST], b[NST];
#pragma unroll
        for (int s = 0; s < NST; ++s) { a[s] = sa[s][j]; b[s] = sb[s][j]; }
        v[j] = cd{gen.template field<F>(a), gen.template field<F>(b)};
    }
    line_fft8<M, TPL, -1>(v, S, t, tw1);
#pragma unroll
    for (int r = 0; r < 8; ++r) S[t + TPL * fft_nat<8>(r)] = v[r];      // natural order
    __syncwarp();
    // X[k] = Ev + w^k Od, X[M-k] = conj(Ev - w^k Od);  Ev = (Z[k] + conj Z[M-k])/2, Od = -i (Z[k] - conj Z[M-k])/2
#pragma unroll
    for (int i = 0; i < (M / 2 + TPL) / TPL; ++i) {
        const int k = t + TPL * i;
        if (k <= M / 2) {
            const cd A = S[k], B = cconj(S[(M - k) & (M - 1)]);
            const cd Ev = cscale(A + B, 0.5);
            const cd D = A - B;
            const cd Od = cd{0.5 * D.y, -0.5 * D.x};
            const cd T = cmul(Od, tw2[k]);
            if (live) {
                if (k == 0) {
                    out[0] = cd{A.x + A.y, 0.0};
                    out[M] = cd{A.x - A.y, 0.0};
                } else {
                    out[k] = Ev + T;
                    out[M - k] = cconj(Ev - T);
                }
            }
        }
    }
    __syncwarp();
}

//   Gen::NST, Gen::NIN              staged doubles per point; real input fields (<= 2) read per point
//   gen.stage(in[NIN] (double2 each: the points g, g + 1), a[NST], b[NST])
//   gen.field<F>(st[NST])           value of field F at a point
struct ZIn {
    const double* f[4];
};

template <int M, int TPL, int NF, class Gen>
__global__ void __launch_bounds__(128, 4) zfwd_kernel(Gen gen, ZIn in, cd* __restrict__ o0, cd* __restrict__ o1, cd* __restrict__ o2,
                                                  cd* __restrict__ o3, int nlines, int nzp) {
    using L = ZLayout<M, TPL>;
    constexpr int LPW = L::kLinesPerWarp, NST = Gen::NST, NIN = Gen::NIN;
    constexpr int kLineBytes = L::fwd_line_bytes(NIN);
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cd* tw1 = reinterpret_cast<cd*>(smem_raw);
    cd* tw2 = tw1 + M;
    load_twiddles<M>(tw1, tw2);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const int sub = lane / TPL, t = lane % TPL;
    unsigned char* slot = smem_raw + L::kTwBytes + (size_t)(warp * LPW + sub) * kLineBytes;
    cd* S = reinterpret_cast<cd*>(slot);
    double2* land = reinterpret_cast<double2*>(slot + (L::kScratch > M + 1 ? L::kScratch : M + 2) * 16);   // [NIN][M] pairs
    const int stride = gridDim.x * wpb * LPW;

    // chunk t + TPL j of a line is copied AND read by lane t: no cross-lane hazard on the landing zone
    auto issue = [&](int line) {
        if (line < nlines) {
#pragma unroll
            for (int q = 0; q < NIN; ++q) {
                const double2* src = reinterpret_cast<const double2*>(in.f[q] + (size_t)line * (2 * M)) + t;
#pragma unroll
                for (int j = 0; j < 8; ++j) cp_async16(land + q * M + t + TPL * j, src + TPL * j);
            }
        }
        cp_async_commit();
    };
    int line0 = (blockIdx.x * wpb + warp) * LPW;
    issue(line0 + sub);
    for (; line0 < nlines; line0 += stride) {
        const int line = line0 + sub;
        const bool live = line < nlines;
        cp_async_wait<0>();
        double sa[NST][8], sb[NST][8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            double2 pin[NIN];
#pragma unroll
            for (int q = 0; q < NIN; ++q) pin[q] = live ? land[q * M + t + TPL * j] : make_double2(1.0, 1.0);
            double a[NST], b[NST];
            gen.stage(pin, a, b);
#pragma unroll
            for (int s = 0; s < NST; ++s) { sa[s][j] = a[s]; sb[s][j] = b[s]; }
        }
        issue(line + stride);
        const size_t orow = (size_t)(live ? line : 0) * nzp;
        zfwd_field<M, TPL, 0>(gen, sa, sb, S, tw1, tw2, t, o0 + orow, live);
        if constexpr (NF > 1) zfwd_field<M, TPL, 1>(gen, sa, sb, S, tw1, tw2, t, o1 + orow, live);
        if constexpr (NF > 2) zfwd_field<M, TPL, 2>(gen, sa, sb, S, tw1, tw2, t, o2 + orow, live);
        if constexpr (NF > 3) zfwd_field<M, TPL, 3>(gen, sa, sb, S, tw1, tw2, t, o3 + orow, live);
    }
    cp_async_wait<0>();
}

// inverse of one field from its staged half-spectrum line X[0..M]: packed complex Z, inverse FFT; slot r of
// `res` then holds the real pair (f[2n], f[2n+1]) for n = t + TPL fft_nat<8>(r), scaled like an unnormalised
// c2r of length 2M.   Z[k] = (X[k] + conj X[M-k]) + i conj(w^k) (X[k] - conj X[M-k]),  w = exp(-i pi / M);
// every lane builds the 8 inputs of its own FFT directly (no exchange); Im X[0], Im X[M] are ignored (c2r).
template <int M, int TPL>
__device__ __forceinline__ void zinv_field(const cd* X, cd* res, cd* S, const cd* tw1, const cd* tw2, int t) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int k = t + TPL * j;
        cd Xa = X[k], Xb = X[M - k];
        if (k == 0) { Xa.y = 0.0; Xb.y = 0.0; }
        const cd B = cconj(Xb);
        const cd Ev = Xa + B;
        const cd Od = cmul(Xa - B, cconj(tw2[k]));
        res[j] = cd{Ev.x - Od.y, Ev.y + Od.x};
    }
    line_fft8<M, TPL, +1>(res, S, t, tw1);
}

struct ZSpec {
    const cd* f[4];
};

// forward z work of a CTA: the lines line_begin + warp LPW + k stride < line_end (global line index = x n1 + y)
template <int M, int TPL, int NF, class Gen>
__device__ __forceinline__ void zfwd_item(const Gen& gen, const ZIn& in, const SPassFields& out, int line_begin, int line_end, int stride,
                                          int nzp, unsigned char* zarea, const cd* tw1, const cd* tw2) {
    using L = ZLayout<M, TPL>;
    constexpr int LPW = L::kLinesPerWarp, NST = Gen::NST, NIN = Gen::NIN;
    constexpr int kLineBytes = L::fwd_line_bytes(NIN);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane / TPL, t = lane % TPL;
    unsigned char* slot = zarea + (size_t)(warp * LPW + sub) * kLineBytes;
    cd* S = reinterpret_cast<cd*>(slot);
    double2* land = reinterpret_cast<double2*>(slot + (L::kScratch > M + 1 ? L::kScratch : M + 2) * 16);   // [NIN][M] pairs
    auto issue = [&](int line) {
        if (line < line_end) {
#pragma unroll
            for (int q = 0; q < NIN; ++q) {
                const double2* src = reinterpret_cast<const double2*>(in.f[q] + (size_t)line * (2 * M)) + t;
#pragma unroll
                for (int j = 0; j < 8; ++j) cp_async16(land + q * M + t + TPL * j, src + TPL * j);
            }
        }
        cp_async_commit();
    };
    int line0 = line_begin + warp * LPW;
    issue(line0 + sub);
    for (; line0 < line_end; line0 += stride) {
        const int line = line0 + sub;
        const bool live = line < line_end;
        cp_async_wait<0>();
        double sa[NST][8], sb[NST][8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            double2 pin[NIN];
#pragma unroll
            for (int q = 0; q < NIN; ++q) pin[q] = live ? land[q * M + t + TPL * j] : make_double2(1.0, 1.0);
            double a[NST], b[NST];
            gen.stage(pin, a, b);
#pragma unroll
            for (int s = 0; s < NST; ++s) { sa[s][j] = a[s]; sb[s][j] = b[s]; }
        }
        issue(line + stride);
        const size_t orow = (size_t)(live ? line : line_begin) * nzp;
        zfwd_field<M, TPL, 0>(gen, sa, sb, S, tw1, tw2, t, out.f[0] + orow, live);
        if constexpr (NF > 1) zfwd_field<M, TPL, 1>(gen, sa, sb, S, tw1, tw2, t, out.f[1] + orow, live);
        if constexpr (NF > 2) zfwd_field<M, TPL, 2>(gen, sa, sb, S, tw1, tw2, t, out.f[2] + orow, live);
        if constexpr (NF > 3) zfwd_field<M, TPL, 3>(gen, sa, sb, S, tw1, tw2, t, out.f[3] + orow, live);
    }
    cp_async_wait<0>();
}

// inverse z item: NF half-spectrum lines -> NF real lines in registers -> post-op; if NFW > 0 the post-op hands
// Post::NST staged values per point to GenF and NFW fields generated from them are transformed forward again and
// written over the lines of spec.f[0..NFW-1] (the inputs of the line are in shared memory by then).
//   post.apply(g, n, vold, u0[NF], u1[NF], acc, sta[NST], stb[NST])
template <int M, int TPL, int NF, int NRED, class Post, int NFW, class GenF>
__device__ __forceinline__ void zinv_item(const Post& post, const GenF& genf, const SPassFields& spec, const double* __restrict__ den,
                                          const double* __restrict__ vin, int line_begin, int line_end, int stride, int nzp,
                                          unsigned char* zarea, const cd* tw1, const cd* tw2, double* acc) {
    using L = ZLayout<M, TPL>;
    constexpr int LPW = L::kLinesPerWarp;
    constexpr int NREAL = (Post::kDen ? 1 : 0) + (Post::kVin ? 1 : 0);
    constexpr int G = NF + NREAL;
    constexpr int kLineBytes = L::inv_line_bytes(NF, NREAL);
    constexpr int NST = Post::NST > 0 ? Post::NST : 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane / TPL, t = lane % TPL;
    unsigned char* slot = zarea + (size_t)(warp * LPW + sub) * kLineBytes;
    cd* S = reinterpret_cast<cd*>(slot);
    cd* sp = S + L::kScratch;                                  // [NF][kSpecLine]
    double2* rland = reinterpret_cast<double2*>(sp + NF * L::kSpecLine);   // [NREAL][M] pairs

    auto issue_spec = [&](int f, int line) {
        if (line < line_end) {
            const cd* src = spec.f[f] + (size_t)line * nzp + t;
            cd* dst = sp + f * L::kSpecLine + t;
#pragma unroll
            for (int i = 0; i < (M + TPL) / TPL; ++i)
                if (t + TPL * i <= M) cp_async16(dst + TPL * i, src + TPL * i);
        }
        cp_async_commit();
    };
    auto issue_real = [&](int q, const double* base, int line) {
        if (line < line_end) {
            const double2* src = reinterpret_cast<const double2*>(base + (size_t)line * (2 * M)) + t;
#pragma unroll
            for (int j = 0; j < 8; ++j) cp_async16(rland + q * M + t + TPL * j, src + TPL * j);
        }
        cp_async_commit();
    };
    int line0 = line_begin + warp * LPW;
    {
        const int line = line0 + sub;
#pragma unroll
        for (int f = 0; f < NF; ++f) issue_spec(f, line);
        if constexpr (Post::kDen) issue_real(0, den, line);
        if constexpr (Post::kVin) issue_real(Post::kDen ? 1 : 0, vin, line);
    }
    for (; line0 < line_end; line0 += stride) {
        const int line = line0 + sub;
        const bool live = line < line_end;
        const int next = line + stride;
        const size_t base = (size_t)line * (2 * M);
        cd res[NF][8];
#pragma unroll
        for (int f = 0; f < NF; ++f) {
            cp_async_wait<G - 1>();
            __syncwarp();
            zinv_field<M, TPL>(sp + f * L::kSpecLine, res[f], S, tw1, tw2, t);
            issue_spec(f, next);
        }
        double2 nn[8], vv[8];
        if constexpr (Post::kDen) {
            cp_async_wait<G - 1>();
#pragma unroll
            for (int r = 0; r < 8; ++r) nn[r] = rland[t + TPL * fft_nat<8>(r)];
            issue_real(0, den, next);
        }
        if constexpr (Post::kVin) {
            cp_async_wait<G - 1>();
#pragma unroll
            for (int r = 0; r < 8; ++r) vv[r] = rland[(Post::kDen ? M : 0) + t + TPL * fft_nat<8>(r)];
            issue_real(Post::kDen ? 1 : 0, vin, next);
        }
        double sa[NST][8], sb[NST][8];
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            double u0[NF], u1[NF];
#pragma unroll
            for (int f = 0; f < NF; ++f) { u0[f] = res[f][r].x; u1[f] = res[f][r].y; }
            double a[NST], b[NST];
#pragma unroll
            for (int s = 0; s < NST; ++s) { a[s] = 1.0; b[s] = 1.0; }
            if (live)
                post.apply(base + 2 * (t + TPL * fft_nat<8>(r)), Post::kDen ? nn[r] : make_double2(0.0, 0.0),
                           Post::kVin ? vv[r] : make_double2(0.0, 0.0), u0, u1, acc, a, b);
#pragma unroll
            for (int s = 0; s < NST; ++s) { sa[s][fft_nat<8>(r)] = a[s]; sb[s][fft_nat<8>(r)] = b[s]; }
        }
        if constexpr (NFW > 0) {
            __syncwarp();
            const size_t orow = (size_t)(live ? line : line_begin) * nzp;
            zfwd_field<M, TPL, 0>(genf, sa, sb, S, tw1, tw2, t, spec.f[0] + orow, live);
            if constexpr (NFW > 1) zfwd_field<M, TPL, 1>(genf, sa, sb, S, tw1, tw2, t, spec.f[1] + orow, live);
            if constexpr (NFW > 2) zfwd_field<M, TPL, 2>(genf, sa, sb, S, tw1, tw2, t, spec.f[2] + orow, live);
            if constexpr (NFW > 3) zfwd_field<M, TPL, 3>(genf, sa, sb, S, tw1, tw2, t, spec.f[3] + orow, live);
        }
    }
    cp_async_wait<0>();
}

// Streamed inverse z work: like zinv_item, but the NF spectral lines of a real-space line pass through a ring of TWO
// landing buffers and every inverse result is FOLDED into Post::NACC per-point accumulators as soon as it exists
// (WGC99: conv = u1 + th u2 + th^2 u3 / 2 and w = u2 + th u3 instead of u1, u2, u3), the last field goes to the post-op
// directly.  A thread then holds 2 NACC + 4 doubles per point instead of 2 NF + 2, and a line slot 8.4 KB of shared
// memory instead of 12.5 KB: three CTAs (12 warps) per SM instead of two -- the pass is bound by dependent-issue latency,
// so resident warps are what it needs.
//   Ctx  post.begin()                                   per-thread constants
//   post.fold<F>(ctx, n, u, acc[NACC])                  field F < NF - 1 at one real point with density n
//   post.finish(ctx, g, n2, accA, accB, uA, uB, red, sta, stb)   points g, g + 1: accumulators, last field, sums, staged values
template <int M, int TPL, int NF, int NRED, class Post, int NFW, class GenF>
__device__ __forceinline__ void zinv_item_stream(const Post& post, const GenF& genf, const SPassFields& spec, const double* __restrict__ den,
                                                 int line_begin, int line_end, int stride, int nzp, unsigned char* zarea,
                                                 const cd* tw1, const cd* tw2, double* acc) {
    using L = ZLayout<M, TPL>;
    constexpr int LPW = L::kLinesPerWarp;
    constexpr int kLineBytes = L::stream_line_bytes(Post::kDen);
    constexpr int NACC = Post::NACC > 0 ? Post::NACC : 1;
    constexpr int NST = Post::NST > 0 ? Post::NST : 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane / TPL, t = lane % TPL;
    unsigned char* slot = zarea + (size_t)(warp * LPW + sub) * kLineBytes;
    cd* S = reinterpret_cast<cd*>(slot);
    cd* sp = S + L::kScratch;                                  // [2][kSpecLine]
    double2* rland = reinterpret_cast<double2*>(sp + 2 * L::kSpecLine);
    const typename Post::Ctx ctx = post.begin();

    auto issue_spec = [&](int f, int line, int buf) {
        if (line < line_end) {
            const cd* src = spec.f[f] + (size_t)line * nzp + t;
            cd* dst = sp + buf * L::kSpecLine + t;
#pragma unroll
            for (int i = 0; i < (M + TPL) / TPL; ++i)
                if (t + TPL * i <= M) cp_async16(dst + TPL * i, src + TPL * i);
        }
        cp_async_commit();
    };
    auto issue_real = [&](int line) {
        if (Post::kDen && line < line_end) {
            const double2* src = reinterpret_cast<const double2*>(den + (size_t)line * (2 * M)) + t;
#pragma unroll
            for (int j = 0; j < 8; ++j) cp_async16(rland + t + TPL * j, src + TPL * j);
        }
        cp_async_commit();
    };
    // commit order (oldest first) at the top of every line: S0, R, S1  (NF = 1: S0, R)
    int line0 = line_begin + warp * LPW;
    issue_spec(0, line0 + sub, 0);
    issue_real(line0 + sub);
    if constexpr (NF > 1) issue_spec(1, line0 + sub, 1);
    int par = 0;          // ring position of the line's first field (flips from line to line when NF is odd)
    for (; line0 < line_end; line0 += stride) {
        const int line = line0 + sub;
        const bool live = line < line_end;
        const int next = line + stride;
        const size_t base = (size_t)line * (2 * M);
        double aA[NACC][8], aB[NACC][8];
        double2 nn[8];
        cd res[8];
#pragma unroll
        for (int f = 0; f < NF; ++f) {
            if constexpr (NF == 1) cp_async_wait<0>();
            else if (f == NF - 1) cp_async_wait<2>();
            else cp_async_wait<1>();
            __syncwarp();
            const int buf = NF == 1 ? 0 : ((par + f) & 1);
            zinv_field<M, TPL>(sp + buf * L::kSpecLine, res, S, tw1, tw2, t);      // ends with __syncwarp: the buffer is free
            if constexpr (NF == 1) {
                issue_spec(0, next, 0);
                issue_real(next);
            } else {
                if (f + 2 < NF) issue_spec(f + 2, line, buf);
                else issue_spec(f + 2 - NF, next, buf);
            }
            if (f < NF - 1) {
#pragma unroll
                for (int r = 0; r < 8; ++r) {
                    const double2 n2 = Post::kDen ? rland[t + TPL * fft_nat<8>(r)] : make_double2(0.0, 0.0);
                    double a[NACC], b[NACC];
#pragma unroll
                    for (int q = 0; q < NACC; ++q) { a[q] = aA[q][r]; b[q] = aB[q][r]; }
                    if (f == 0) post.template fold<0>(ctx, n2.x, res[r].x, a), post.template fold<0>(ctx, n2.y, res[r].y, b);
                    else if (f == 1) post.template fold<1>(ctx, n2.x, res[r].x, a), post.template fold<1>(ctx, n2.y, res[r].y, b);
                    else post.template fold<2>(ctx, n2.x, res[r].x, a), post.template fold<2>(ctx, n2.y, res[r].y, b);
#pragma unroll
                    for (int q = 0; q < NACC; ++q) { aA[q][r] = a[q]; aB[q][r] = b[q]; }
                }
            }
            if (NF > 1 && f == NF - 2) {
                // the density line moves to registers for the post-op, its landing zone takes the next line's
#pragma unroll
                for (int r = 0; r < 8; ++r) nn[r] = Post::kDen ? rland[t + TPL * fft_nat<8>(r)] : make_double2(0.0, 0.0);
                issue_real(next);
            }
        }
        if constexpr (NF == 1) {
#pragma unroll
            for (int r = 0; r < 8; ++r) nn[r] = make_double2(0.0, 0.0);
        }
        double sa[NST][8], sb[NST][8];
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            double a[NACC], b[NACC], st0[NST], st1[NST];
#pragma unroll
            for (int q = 0; q < NACC; ++q) { a[q] = aA[q][r]; b[q] = aB[q][r]; }
#pragma unroll
            for (int q = 0; q < NST; ++q) { st0[q] = 1.0; st1[q] = 1.0; }
            if (live) post.finish(ctx, base + 2 * (t + TPL * fft_nat<8>(r)), nn[r], a, b, res[r].x, res[r].y, acc, st0, st1);
#pragma unroll
            for (int q = 0; q < NST; ++q) { sa[q][fft_nat<8>(r)] = st0[q]; sb[q][fft_nat<8>(r)] = st1[q]; }
        }
        if constexpr (NFW > 0) {
            __syncwarp();
            const size_t orow = (size_t)(live ? line : line_begin) * nzp;
            zfwd_field<M, TPL, 0>(genf, sa, sb, S, tw1, tw2, t, spec.f[0] + orow, live);
            if constexpr (NFW > 1) zfwd_field<M, TPL, 1>(genf, sa, sb, S, tw1, tw2, t, spec.f[1] + orow, live);
            if constexpr (NFW > 2) zfwd_field<M, TPL, 2>(genf, sa, sb, S, tw1, tw2, t, spec.f[2] + orow, live);
            if constexpr (NFW > 3) zfwd_field<M, TPL, 3>(genf, sa, sb, S, tw1, tw2, t, spec.f[3] + orow, live);
        }
        if constexpr (NF > 1) par = (par + NF) & 1;
    }
    cp_async_wait<0>();
}

struct GenNone {                       // placeholder GenF of inverse kernels without a forward part
    static constexpr int NST = 1, NIN = 1;
    __device__ void stage(const double2*, double*, double*) const {}
    template <int F>
    __device__ double field(const double* s) const { return s[0]; }
};

//   Post::kDen / Post::kVin          the post-op reads the density / the previous potential at its points
//   post.apply(g, n, vold, u0[NF], u1[NF], acc, sta[NST], stb[NST])   for the points g and g + 1 (n, vold: double2)
// NFW > 0: NFW fields generated by GenF from the post-op's staged values are transformed forward again and written over
// the lines of spec.f[0..NFW-1] (WGC99: the mid pass and the forward z pass of the second batch in one kernel -- P never
// travels through HBM)
// STREAM: zinv_item_stream (spectral lines through a two-buffer ring, results folded as they arrive; 3 CTAs per SM) instead
// of zinv_item (all NF lines landed and transformed before the post-op; 2 CTAs per SM)
template <int M, int TPL, int NF, int NRED, class Post, int NFW, class GenF, bool STREAM>
__global__ void __launch_bounds__(128, STREAM ? 3 : 2) zinv_kernel(Post post, GenF genf, SPassFields spec, const double* __restrict__ den,
                                                                  const double* __restrict__ vin, int nlines, int nzp,
                                                                  double* __restrict__ partials) {
    using L = ZLayout<M, TPL>;
    constexpr int LPW = L::kLinesPerWarp;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cd* tw1 = reinterpret_cast<cd*>(smem_raw);
    cd* tw2 = tw1 + M;
    load_twiddles<M>(tw1, tw2);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    double acc[NRED > 0 ? NRED : 1];
#pragma unroll
    for (int r = 0; r < (NRED > 0 ? NRED : 1); ++r) acc[r] = 0.0;
    if constexpr (STREAM)
        zinv_item_stream<M, TPL, NF, NRED, Post, NFW, GenF>(post, genf, spec, den, blockIdx.x * wpb * LPW, nlines, gridDim.x * wpb * LPW,
                                                            nzp, smem_raw + L::kTwBytes, tw1, tw2, acc);
    else
        zinv_item<M, TPL, NF, NRED, Post, NFW, GenF>(post, genf, spec, den, vin, blockIdx.x * wpb * LPW, nlines, gridDim.x * wpb * LPW, nzp,
                                                     smem_raw + L::kTwBytes, tw1, tw2, acc);
    if constexpr (NRED > 0) {
        __shared__ double red[NRED][4];
#pragma unroll
        for (int r = 0; r < NRED; ++r) {
            const double w = warp_sum(acc[r]);
            if (lane == 0) red[r][warp] = w;
        }
        __syncthreads();
        if (threadIdx.x < NRED) {
            double s = 0.0;
            for (int w = 0; w < wpb; ++w) s += red[threadIdx.x][w];
            partials[(size_t)threadIdx.x * PAD_MAX_BLOCKS + blockIdx.x] = s;
        }
    }
}

inline int zgrid(int nlines, int lines_per_block, int blocks_per_sm) {
    int b = (nlines + lines_per_block - 1) / lines_per_block;
    const int cap = 148 * blocks_per_sm;
    if (b > cap) b = cap;
    if (b > PAD_MAX_BLOCKS) b = PAD_MAX_BLOCKS;
    return b < 1 ? 1 : b;
}

// z lines of the plan's real-space block: slab plans hold n0_loc x-planes
inline int z_lines(const pad_plan* p) { return (p->dist ? p->n0_loc : p->n0) * p->n1; }

template <int M, int TPL, int NF, class Gen>
int launch_zfwd(pad_plan* p, cudaStream_t s, Gen gen, const double* in0, const double* in1, cd* o0, cd* o1, cd* o2, cd* o3,
                const double* in2 = nullptr, const double* in3 = nullptr) {
    constexpr int warps = 4;
    using L = ZLayout<M, TPL>;
    constexpr int smem = L::kTwBytes + warps * L::kLinesPerWarp * L::fwd_line_bytes(Gen::NIN);
    auto kern = zfwd_kernel<M, TPL, NF, Gen>;
    static bool attr_done[64] = {false};
    if (!attr_done[p->device & 63]) {
        PAD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr_done[p->device & 63] = true;
    }
    const int nlines = z_lines(p);
    ZIn in{{in0, in1, in2, in3}};
    kern<<<zgrid(nlines, warps * (32 / TPL), 4), warps * 32, smem, s>>>(gen, in, o0, o1, o2, o3, nlines, p->nzp);
    ++g_pad_launches;
    PAD_CUDA(cudaGetLastError());
    return PAD_OK;
}

template <int M, int TPL, int NF, int NRED, class Post, int NFW, class GenF, bool STREAM>
int launch_zinv_impl(pad_plan* p, cudaStream_t s, Post post, const cd* i0, const cd* i1, const cd* i2, const cd* i3,
                     const double* den, const double* vin, int* grid_out, GenF genf) {
    constexpr int warps = 4;
    using L = ZLayout<M, TPL>;
    constexpr int NREAL = (Post::kDen ? 1 : 0) + (Post::kVin ? 1 : 0);
    constexpr int line_bytes = STREAM ? L::stream_line_bytes(Post::kDen) : L::inv_line_bytes(NF, NREAL);
    constexpr int smem = L::kTwBytes + warps * L::kLinesPerWarp * line_bytes;
    auto kern = zinv_kernel<M, TPL, NF, NRED, Post, NFW, GenF, STREAM>;
    static bool attr_done[64] = {false};
    if (!attr_done[p->device & 63]) {
        PAD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr_done[p->device & 63] = true;
    }
    const int nlines = z_lines(p);
    constexpr int by_smem = (227 * 1024) / (smem + 1024);
    constexpr int want = STREAM ? 3 : 2;
    const int grid = zgrid(nlines, warps * (32 / TPL), by_smem < want ? by_smem : want);
    SPassFields in;
    in.f[0] = const_cast<cd*>(i0); in.f[1] = const_cast<cd*>(i1); in.f[2] = const_cast<cd*>(i2); in.f[3] = const_cast<cd*>(i3);
    kern<<<grid, warps * 32, smem, s>>>(post, genf, in, den, vin, nlines, p->nzp, p->partials);
    ++g_pad_launches;
    if (grid_out) *grid_out = grid;
    PAD_CUDA(cudaGetLastError());
    return PAD_OK;
}

template <int M, int TPL, int NF, int NRED, class Post, int NFW = 0, class GenF = GenNone>
int launch_zinv(pad_plan* p, cudaStream_t s, Post post, const cd* i0, const cd* i1, const cd* i2, const cd* i3,
                const double* den, const double* vin, int* grid_out, GenF genf = GenF{}) {
#ifdef PAD_BUILD_ZINV_STREAM      // measured 7-13 % slower than the batch form at 256^3 (DESIGN.md section 4.1): not built by default
    if (g_pad_zinv_stream)
        return launch_zinv_impl<M, TPL, NF, NRED, Post, NFW, GenF, true>(p, s, post, i0, i1, i2, i3, den, vin, grid_out, genf);
#endif
    return launch_zinv_impl<M, TPL, NF, NRED, Post, NFW, GenF, false>(p, s, post, i0, i1, i2, i3, den, vin, grid_out, genf);
}

// ------------------------------------------------------------------------------------------------
//  software-pipelined (z, y) kernels (zy_pipe.cuh): the z passes above as ITEMS over a group of lines of one
//  x-plane, next to the y items of that plane
// ------------------------------------------------------------------------------------------------

template <int M, int LY>
__device__ __forceinline__ cd* pipe_tables(unsigned char* smem_raw, cd*& tw1, cd*& tw2, cd*& twy) {
    tw1 = reinterpret_cast<cd*>(smem_raw);
    tw2 = tw1 + M;
    twy = tw2 + M;
    load_twiddles<M>(tw1, tw2);
    spass_load_twiddles<LY>(twy);
    return twy + LY;
}

// forward: stage 0 = [gen + z r2c] of a line group, stage 1 = in-place y FFT of a group of tiles
template <int M, int TPL, int NF, class Gen, int LY>
__global__ void __launch_bounds__(128, 4) zy_fwd_kernel(Gen gen, ZIn in, SPassFields out, PipeCtl* ctl, PipeShape sh, ZYGeom g) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int sm_item[4];
    cd *tw1, *tw2, *twy;
    cd* work = pipe_tables<M, LY>(smem_raw, tw1, tw2, twy);
    const int ntiles = NF * g.chunks + 1;
    PipeSched ps;
    pipe_begin<2>(ctl, ps);
    for (;;) {
        const PipeItem it = pipe_next<2>(ctl, sh, sm_item, ps);
        if (it.stage < 0) break;
        if (it.stage == 0) {
            const int l0 = it.plane * g.n1 + it.sub * g.lpi;
            zfwd_item<M, TPL, NF>(gen, in, out, l0, l0 + g.lpi, 4 * (32 / TPL), g.nzp, reinterpret_cast<unsigned char*>(work), tw1, tw2);
        } else {
            const int w0 = it.sub * g.tpi;
            ytile_item_direct<LY, -1, true>(out, NF, g, it.plane, w0, min(w0 + g.tpi, ntiles), ntiles, work, twy);
        }
        pipe_done(ctl, sh, it);
    }
    pipe_exit(ctl, sh, sm_item);
}

// inverse: stage 0 = in-place inverse y FFT of a group of tiles (NF fields), stage 1 = [z c2r + post-op (+ gen + z r2c of
// NFW fields)] of a line group, stage 2 (NFW > 0) = in-place forward y FFT of the NFW new fields.
// part: per-item partial sums [NRED][nplanes * items[1]] (deterministic whatever CTA ran the item)
template <int M, int TPL, int NF, int NRED, class Post, int NFW, class GenF, int LY>
__global__ void __launch_bounds__(128, 2) yz_inv_kernel(Post post, GenF genf, SPassFields spec, const double* __restrict__ den,
                                                       const double* __restrict__ vin, PipeCtl* ctl, PipeShape sh, ZYGeom g,
                                                       double* __restrict__ part) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int sm_item[4];
    __shared__ double red[NRED > 0 ? NRED : 1][4];
    cd *tw1, *tw2, *twy;
    cd* work = pipe_tables<M, LY>(smem_raw, tw1, tw2, twy);
    const int nt_in = NF * g.chunks + 1, nt_out = NFW * g.chunks + 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int NSTAGE = NFW > 0 ? 3 : 2;
    PipeSched ps;
    pipe_begin<NSTAGE>(ctl, ps);
    for (;;) {
        const PipeItem it = pipe_next<NSTAGE>(ctl, sh, sm_item, ps);
        if (it.stage < 0) break;
        if (it.stage == 0) {
            const int w0 = it.sub * g.tpi;
            ytile_item_async<LY, +1, false>(spec, NF, g, it.plane, w0, min(w0 + g.tpi, nt_in), nt_in, work, twy);
        } else if (it.stage == 1) {
            double acc[NRED > 0 ? NRED : 1];
#pragma unroll
            for (int r = 0; r < (NRED > 0 ? NRED : 1); ++r) acc[r] = 0.0;
            const int l0 = it.plane * g.n1 + it.sub * g.lpi;
            zinv_item<M, TPL, NF, NRED, Post, NFW, GenF>(post, genf, spec, den, vin, l0, l0 + g.lpi, 4 * (32 / TPL), g.nzp,
                                                         reinterpret_cast<unsigned char*>(work), tw1, tw2, acc);
            if constexpr (NRED > 0) {
#pragma unroll
                for (int r = 0; r < NRED; ++r) {
                    const double w = warp_sum(acc[r]);
                    if (lane == 0) red[r][warp] = w;
                }
                __syncthreads();
                if (threadIdx.x < NRED) {
                    const double s = (red[threadIdx.x][0] + red[threadIdx.x][1]) + (red[threadIdx.x][2] + red[threadIdx.x][3]);
                    part[(size_t)threadIdx.x * ((size_t)sh.nplanes * sh.items[1]) + (size_t)it.plane * sh.items[1] + it.sub] = s;
                }
            }
        } else {
            const int w0 = it.sub * g.tpi;
            ytile_item_async<LY, -1, true>(spec, NFW, g, it.plane, w0, min(w0 + g.tpi, nt_out), nt_out, work, twy);
        }
        pipe_done(ctl, sh, it);
    }
    pipe_exit(ctl, sh, sm_item);
}

// sum of the per-item partials in a fixed order
__global__ void __launch_bounds__(PAD_THREADS) pipe_finalize_kernel(const double* __restrict__ part, int nitems, FinalizeArgs a) {
    __shared__ double sm[PAD_THREADS / 32];
    __shared__ double total[PAD_MAX_RED];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int t = 0; t < a.nterms; ++t) {
        double v = 0.0;
        for (int b = threadIdx.x; b < nitems; b += PAD_THREADS) v += part[(size_t)t * nitems + b];
        v = warp_sum(v);
        if (lane == 0) sm[warp] = v;
        __syncthreads();
        if (warp == 0) {
            double w = lane < PAD_THREADS / 32 ? sm[lane] : 0.0;
            w = warp_sum(w);
            if (lane == 0) total[t] = w;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        double e = 0.0;
        for (int t = 0; t < a.nterms; ++t) {
            if (a.sums_out) a.sums_out[t] = total[t];
            e += a.coef[t] * total[t];
        }
        if (a.E_out) a.E_out[0] = (a.accumulate ? a.E_out[0] : 0.0) + e;
    }
}

inline bool spass_len_ok(int n) { return n == 64 || n == 128 || n == 256 || n == 512; }
inline bool pipe_len_ok(int n) { return n == 128 || n == 256; }
bool pipe_shape(const pad_plan* p) {
    return g_pad_pipe && g_pad_own_xy && !p->dist && (p->n2 == 128 || p->n2 == 256 || p->n2 == 512) && pipe_len_ok(p->n1) &&
           spass_len_ok(p->n0) && p->n0 <= PIPE_MAX_PLANES;
}

int pipe_prepare(pad_plan* p, int lines_per_iter, ZYGeom* g) {
    if (!p->pipe_ctl) {
        PAD_CUDA(cudaMalloc(&p->pipe_ctl, sizeof(PipeCtl)));
        PAD_CUDA(cudaMemset(p->pipe_ctl, 0, sizeof(PipeCtl)));
        p->bytes_allocated += sizeof(PipeCtl);
    }
    g->n1 = p->n1; g->nzp = p->nzp; g->nzh = p->nzh; g->chunks = p->nzh / 8;
    g->plane = (long long)p->n1 * p->nzp;
    int lpi = g_pad_pipe_lpi > 0 ? g_pad_pipe_lpi : 2 * lines_per_iter;
    lpi = (lpi / lines_per_iter) * lines_per_iter;
    if (lpi < lines_per_iter) lpi = lines_per_iter;
    while (lpi > lines_per_iter && p->n1 % lpi) lpi -= lines_per_iter;
    if (p->n1 % lpi) { pad_set_error("pipelined (z, y) pass: n1 = %d is not a multiple of %d lines", p->n1, lpi); return PAD_ERR_ARG; }
    g->lpi = lpi;
    g->tpi = g_pad_pipe_tpi > 0 ? g_pad_pipe_tpi : 4;
    return PAD_OK;
}

template <int M, int TPL, int NF, class Gen, int LY>
int launch_zy_fwd_L(pad_plan* p, cudaStream_t s, Gen gen, const double* in0, const double* in1, cd* const* out) {
    using L = ZLayout<M, TPL>;
    using P = SPass<LY>;
    constexpr int warps = 4;
    constexpr int zbytes = warps * L::kLinesPerWarp * L::fwd_line_bytes(Gen::NIN);
    constexpr int ybytes = P::TPC * P::TILE_CD * 16;
    constexpr int smem = (2 * M + LY) * 16 + (zbytes > ybytes ? zbytes : ybytes);
    auto kern = zy_fwd_kernel<M, TPL, NF, Gen, LY>;
    static bool attr_done[64] = {false};
    if (!attr_done[p->device & 63]) {
        PAD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr_done[p->device & 63] = true;
    }
    ZYGeom g;
    PAD_TRY(pipe_prepare(p, warps * L::kLinesPerWarp, &g));
    PipeShape sh;
    sh.nstage = 2; sh.nplanes = p->n0;
    sh.items[0] = p->n1 / g.lpi;
    sh.items[1] = (NF * g.chunks + 1 + g.tpi - 1) / g.tpi;
    sh.items[2] = 0;
    constexpr int by_smem = (227 * 1024) / (smem + 1024);
    const int grid = 148 * (by_smem < 4 ? by_smem : 4);
    ZIn in{{in0, in1, nullptr, nullptr}};
    SPassFields o;
    for (int i = 0; i < 4; ++i) o.f[i] = i < NF ? out[i] : nullptr;
    kern<<<grid, warps * 32, smem, s>>>(gen, in, o, reinterpret_cast<PipeCtl*>(p->pipe_ctl), sh, g);
    ++g_pad_launches;
    PAD_CUDA(cudaGetLastError());
    return PAD_OK;
}

template <int M, int TPL, int NF, class Gen>
int launch_zy_fwd(pad_plan* p, cudaStream_t s, Gen gen, const double* in0, const double* in1, cd* const* out) {
    if (p->n1 == 256) return launch_zy_fwd_L<M, TPL, NF, Gen, 256>(p, s, gen, in0, in1, out);
    return launch_zy_fwd_L<M, TPL, NF, Gen, 128>(p, s, gen, in0, in1, out);
}

template <int M, int TPL, int NF, int NRED, class Post, int NFW, class GenF, int LY>
int launch_yz_inv_L(pad_plan* p, cudaStream_t s, Post post, GenF genf, cd* const* spec, const double* den, const double* vin,
                    const FinalizeArgs* fin) {
    using L = ZLayout<M, TPL>;
    using P = SPass<LY>;
    constexpr int warps = 4;
    constexpr int NREAL = (Post::kDen ? 1 : 0) + (Post::kVin ? 1 : 0);
    constexpr int zbytes = warps * L::kLinesPerWarp * L::inv_line_bytes(NF, NREAL);
    constexpr int ybytes = 2 * P::TPC * P::TILE_CD * 16;
    constexpr int smem = (2 * M + LY) * 16 + (zbytes > ybytes ? zbytes : ybytes);
    auto kern = yz_inv_kernel<M, TPL, NF, NRED, Post, NFW, GenF, LY>;
    static bool attr_done[64] = {false};
    if (!attr_done[p->device & 63]) {
        PAD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr_done[p->device & 63] = true;
    }
    ZYGeom g;
    PAD_TRY(pipe_prepare(p, warps * L::kLinesPerWarp, &g));
    PipeShape sh;
    sh.nstage = NFW > 0 ? 3 : 2; sh.nplanes = p->n0;
    sh.items[0] = (NF * g.chunks + 1 + g.tpi - 1) / g.tpi;
    sh.items[1] = p->n1 / g.lpi;
    sh.items[2] = NFW > 0 ? (NFW * g.chunks + 1 + g.tpi - 1) / g.tpi : 0;
    const size_t nitems = (size_t)sh.nplanes * sh.items[1];
    if (NRED > 0 && p->pipe_part_n < nitems * NRED) {
        if (p->pipe_part) PAD_CUDA(cudaFree(p->pipe_part));
        p->pipe_part = nullptr;
        PAD_CUDA(cudaMalloc(&p->pipe_part, sizeof(double) * nitems * NRED));
        p->pipe_part_n = nitems * NRED;
        p->bytes_allocated += sizeof(double) * nitems * NRED;
    }
    constexpr int by_smem = (227 * 1024) / (smem + 1024);
    static_assert(by_smem >= 1, "pipelined inverse pass: line slots do not fit in shared memory");
    const int grid = 148 * (by_smem < 2 ? by_smem : 2);
    SPassFields f;
    for (int i = 0; i < 4; ++i) f.f[i] = i < NF ? spec[i] : nullptr;
    kern<<<grid, warps * 32, smem, s>>>(post, genf, f, den, vin, reinterpret_cast<PipeCtl*>(p->pipe_ctl), sh, g, p->pipe_part);
    ++g_pad_launches;
    PAD_CUDA(cudaGetLastError());
    if (NRED > 0 && fin) {
        pipe_finalize_kernel<<<1, PAD_THREADS, 0, s>>>(p->pipe_part, (int)nitems, *fin);
        ++g_pad_launches;
        PAD_CUDA(cudaGetLastError());
    }
    return PAD_OK;
}

template <int M, int TPL, int NF, int NRED, class Post, int NFW, class GenF>
int launch_yz_inv(pad_plan* p, cudaStream_t s, Post post, GenF genf, cd* const* spec, const double* den, const double* vin,
                  const FinalizeArgs* fin) {
    if (p->n1 == 256) return launch_yz_inv_L<M, TPL, NF, NRED, Post, NFW, GenF, 256>(p, s, post, genf, spec, den, vin, fin);
    return launch_yz_inv_L<M, TPL, NF, NRED, Post, NFW, GenF, 128>(p, s, post, genf, spec, den, vin, fin);
}

// ------------------------------------------------------------------------------------------------
//  batched 2-D (x, y) transform over the padded layout, in place
// ------------------------------------------------------------------------------------------------
int ensure_xy(pad_plan* p, cudaStream_t s) {
    if (!p->xy_ready) {
        p->nzp = p->n2 / 2 + 8;
        int n[2] = {p->n0, p->n1};
        size_t w = 0;
        PAD_CUFFT(cufftCreate(&p->xy));
        PAD_CUFFT(cufftSetAutoAllocation(p->xy, 0));
        PAD_CUFFT(cufftMakePlanMany(p->xy, 2, n, n, p->nzp, 1, n, p->nzp, 1, CUFFT_Z2Z, p->nzh, &w));
        if (w > 0) {
            PAD_CUDA(cudaMalloc(&p->xy_work, w));
            p->bytes_allocated += w;
        }
        PAD_CUFFT(cufftSetWorkArea(p->xy, p->xy_work));
        p->xy_stream = (cudaStream_t)(-1);
        p->xy_ready = true;
    }
    if (p->xy_stream != s) {
        PAD_CUFFT(cufftSetStream(p->xy, s));
        p->xy_stream = s;
    }
    return PAD_OK;
}

int xy_exec(pad_plan* p, cudaStream_t s, cd* spec, int dir) {
    PAD_TRY(ensure_xy(p, s));
    PAD_CUFFT(cufftExecZ2Z(p->xy, reinterpret_cast<cufftDoubleComplex*>(spec), reinterpret_cast<cufftDoubleComplex*>(spec),
                           dir < 0 ? CUFFT_FORWARD : CUFFT_INVERSE));
    ++g_pad_fft_execs;
    return PAD_OK;
}

int get_zbuf(pad_plan* p, int i, cd** out) {
    if (i < 0 || i >= 4) { pad_set_error("zbuf index %d", i); return PAD_ERR_ARG; }
    if (p->dist) {          // slab plans: caller-owned buffers (the exchange callback has to know them)
        if (!p->slab_fast[i]) { pad_set_error("slab plan: pad_plan_set_slab_fast_buffers has not been called"); return PAD_ERR_ARG; }
        *out = reinterpret_cast<cd*>(p->slab_fast[i]);
        return PAD_OK;
    }
    const size_t bytes = sizeof(cd) * (size_t)p->n0 * p->n1 * p->nzp;
    if (!p->zbuf[i]) {
        PAD_CUDA(cudaMalloc(&p->zbuf[i], bytes));
        PAD_CUDA(cudaMemset(p->zbuf[i], 0, bytes));       // padding columns stay zero forever
        p->bytes_allocated += bytes;
    }
    *out = reinterpret_cast<cd*>(p->zbuf[i]);
    return PAD_OK;
}


// ------------------------------------------------------------------------------------------------
//  own strided passes (fft_strided.cuh): launchers
// ------------------------------------------------------------------------------------------------
bool own_xy_shape(const pad_plan* p) { return spass_len_ok(p->n0) && spass_len_ok(p->n1); }

SPassGeom spass_geom(const pad_plan* p, int axis) {
    SPassGeom g;
    // slab plans: the y pass sees the local layout (n0_loc, n1, nzp), the x pass the transposed one (n0, n1_loc, nzp)
    const long long row = p->nzp, plane = (long long)(p->dist && axis == 0 ? p->n1_loc : p->n1) * p->nzp;
    g.axis_stride = axis == 0 ? plane : row;
    g.outer_stride = axis == 0 ? row : plane;
    g.n_outer = axis == 0 ? (p->dist ? p->n1_loc : p->n1) : (p->dist ? p->n0_loc : p->n0);
    g.nzh = p->nzh;
    return g;
}

template <int L, int DIR, bool WIDE = false>
int launch_spass_L(pad_plan* p, cudaStream_t s, const SPassFields& f, int nf, const SPassGeom& g) {
    if constexpr (L == 256 && !WIDE) {
        if (g_pad_ywide) return launch_spass_L<L, DIR, true>(p, s, f, nf, g);
    }
    auto kern = spass_kernel<L, DIR, WIDE>;
    using P = SPass<L, WIDE>;
    constexpr int smem = spass_smem_bytes<L, WIDE>(1);
    static bool attr_done[64] = {false};
    if (!attr_done[p->device & 63]) {
        PAD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr_done[p->device & 63] = true;
    }
    const long long tiles = (long long)nf * spass_tiles(g);
    long long grid = (tiles + P::TPC - 1) / P::TPC;
    if (grid > (1 << 20)) grid = 1 << 20;
    kern<<<(unsigned)grid, P::THREADS, smem, s>>>(f, nf, g);
    ++g_pad_launches;
    PAD_CUDA(cudaGetLastError());
    return PAD_OK;
}

template <int L, int DIR, int BLK>
int launch_spass_blocked_L(pad_plan* p, cudaStream_t s, const cd* src, cd* dst, const SPassGeom& g, const SPassBlocked& bl,
                           const SPassPeers& peers = SPassPeers{}) {
    auto kern = spass_blocked_kernel<L, DIR, BLK>;
    constexpr int smem = spass_smem_bytes<L>(1);
    static bool attr_done[64] = {false};
    if (!attr_done[p->device & 63]) {
        PAD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr_done[p->device & 63] = true;
    }
    const long long tiles = spass_tiles(g);
    long long grid = (tiles + SPass<L>::TPC - 1) / SPass<L>::TPC;
    if (grid > (1 << 20)) grid = 1 << 20;
    kern<<<(unsigned)grid, 128, smem, s>>>(src, dst, g, bl, peers);
    ++g_pad_launches;
    PAD_CUDA(cudaGetLastError());
    return PAD_OK;
}

int launch_spass_blocked(pad_plan* p, cudaStream_t s, int dir, const cd* src, cd* dst) {
    const SPassGeom g = spass_geom(p, 1);
    const SPassBlocked bl{p->n1_loc, (long long)p->n0_loc * p->n1_loc * p->nzp, (long long)p->n1_loc * p->nzp};
#define SPASS_BLK_CASE(LL)                                                                                   \
    case LL:                                                                                                 \
        return dir < 0 ? launch_spass_blocked_L<LL, -1, 1>(p, s, src, dst, g, bl) : launch_spass_blocked_L<LL, +1, 2>(p, s, src, dst, g, bl);
    switch (p->n1) {
        SPASS_BLK_CASE(64)
        SPASS_BLK_CASE(128)
        SPASS_BLK_CASE(256)
        SPASS_BLK_CASE(512)
    }
#undef SPASS_BLK_CASE
    pad_set_error("strided FFT pass: length %d not supported", p->n1);
    return PAD_ERR_ARG;
}

// index of a registered slab spectrum buffer (0..3), or -1
int slab_field_index(const pad_plan* p, const cd* ptr) {
    for (int i = 0; i < 4; ++i)
        if (ptr == reinterpret_cast<const cd*>(p->slab_fast[i])) return i;
    return -1;
}

// forward y pass of field `fi` with its result rows pushed into the owner ranks' transposed buffers
int launch_spass_push(pad_plan* p, cudaStream_t s, int fi) {
    const SPassGeom g = spass_geom(p, 1);
    const SPassBlocked bl{p->n1_loc, (long long)p->n0_loc * p->n1_loc * p->nzp, (long long)p->n1_loc * p->nzp};
    SPassPeers peers;
    for (int r = 0; r < 8; ++r) peers.p[r] = r < p->world ? reinterpret_cast<cd*>(p->peer_T[fi][r]) : nullptr;
    peers.my_rank = p->rank;
    const cd* src = reinterpret_cast<const cd*>(p->peer_B[fi][p->rank]);
    switch (p->n1) {
        case 64: return launch_spass_blocked_L<64, -1, 3>(p, s, src, nullptr, g, bl, peers);
        case 128: return launch_spass_blocked_L<128, -1, 3>(p, s, src, nullptr, g, bl, peers);
        case 256: return launch_spass_blocked_L<256, -1, 3>(p, s, src, nullptr, g, bl, peers);
        case 512: return launch_spass_blocked_L<512, -1, 3>(p, s, src, nullptr, g, bl, peers);
    }
    pad_set_error("strided FFT pass: length %d not supported", p->n1);
    return PAD_ERR_ARG;
}

int launch_spass_local(pad_plan* p, cudaStream_t s, int axis, int dir, cd* const* fields, int nf);

// Slab plans, y axis: the pass and the transposition of a batch of fields, software-pipelined over the two stagings.
//   forward:  fields[f] (local layout) --y pass, rows blocked by rank--> staging b --all-to-all--> fields[f] (transposed layout)
//   inverse:  fields[f] (transposed)   --all-to-all--> staging b --y pass from blocked rows--> fields[f] (local layout)
// The exchange of field f runs on the plan's communication stream while the pass of field f + 1 (forward) or f - 1 (inverse)
// runs on `s`; fields[] must be slab_fast buffers 0..3 in order (the callback names them by index).
int slab_ypass_exchange(pad_plan* p, cudaStream_t s, int dir, cd* const* fields, int nf) {
    if (p->slab_push) {
        // peer pointers: forward = y pass with pushed rows, then a barrier (every rank's rows have arrived before the x pass
        // reads the transposed buffers); inverse = barrier (every rank's x pass has pushed its planes), then the plain local pass
        if (dir < 0) {
            for (int f = 0; f < nf; ++f) {
                const int fi = slab_field_index(p, fields[f]);
                if (fi < 0) { pad_set_error("slab y pass: field %d is not a registered slab buffer", f); return PAD_ERR_ARG; }
                PAD_TRY(launch_spass_push(p, s, fi));
            }
            return pad_slab_comm(p, PAD_COMM_BARRIER, 0, s);
        }
        PAD_TRY(pad_slab_comm(p, PAD_COMM_BARRIER, 0, s));
        return launch_spass_local(p, s, 1, +1, fields, nf);
    }
    PAD_TRY(pad_ensure_comm_stream(p));
    int idx[4];
    for (int f = 0; f < nf; ++f) {
        idx[f] = -1;
        for (int i = 0; i < 4; ++i)
            if (fields[f] == reinterpret_cast<cd*>(p->slab_fast[i])) idx[f] = i;
        if (idx[f] < 0) { pad_set_error("slab y pass: field %d is not a registered slab_fast buffer", f); return PAD_ERR_ARG; }
    }
    cd* stg[2] = {reinterpret_cast<cd*>(p->slab_fast[4]), reinterpret_cast<cd*>(p->slab_fast[5])};
    const long long count = (long long)p->n0_loc * p->n1_loc * p->nzp;
    auto a2a = [&](int dst, int src) -> int {
        return pad_slab_comm(p, PAD_COMM_ALL_TO_ALL_FAST + 8 * dst + src, count, p->comm_stream);
    };
    if (dir < 0) {
        for (int f = 0; f < nf; ++f) {
            const int b = f & 1;
            if (f >= 2) PAD_CUDA(cudaStreamWaitEvent(s, p->ev_a2a[b], 0));               // exchange f - 2 has left staging b
            PAD_TRY(launch_spass_blocked(p, s, -1, fields[f], stg[b]));
            PAD_CUDA(cudaEventRecord(p->ev_ready[b], s));
            PAD_CUDA(cudaStreamWaitEvent(p->comm_stream, p->ev_ready[b], 0));
            PAD_TRY(a2a(idx[f], 4 + b));
            PAD_CUDA(cudaEventRecord(p->ev_a2a[b], p->comm_stream));
        }
        PAD_CUDA(cudaStreamWaitEvent(s, p->ev_a2a[0], 0));
        if (nf > 1) PAD_CUDA(cudaStreamWaitEvent(s, p->ev_a2a[1], 0));
        return PAD_OK;
    }
    // inverse: everything queued on `s` so far (the x pass) precedes the first exchange
    PAD_CUDA(cudaEventRecord(p->ev_ready[0], s));
    PAD_CUDA(cudaStreamWaitEvent(p->comm_stream, p->ev_ready[0], 0));
    auto exchange = [&](int f) -> int {
        const int b = f & 1;
        if (f >= 2) PAD_CUDA(cudaStreamWaitEvent(p->comm_stream, p->ev_free[b], 0));    // the pass of field f - 2 has read staging b
        PAD_TRY(a2a(4 + b, idx[f]));
        PAD_CUDA(cudaEventRecord(p->ev_a2a[b], p->comm_stream));
        return PAD_OK;
    };
    PAD_TRY(exchange(0));
    for (int f = 0; f < nf; ++f) {
        const int b = f & 1;
        if (f + 1 < nf) PAD_TRY(exchange(f + 1));
        PAD_CUDA(cudaStreamWaitEvent(s, p->ev_a2a[b], 0));
        PAD_TRY(launch_spass_blocked(p, s, +1, stg[b], fields[f]));
        PAD_CUDA(cudaEventRecord(p->ev_free[b], s));
    }
    return PAD_OK;
}

// in-place FFT of nf padded half-spectra along axis 0 (x) or 1 (y)
int launch_spass(pad_plan* p, cudaStream_t s, int axis, int dir, cd* const* fields, int nf) {
    if (p->dist && axis == 1) return slab_ypass_exchange(p, s, dir, fields, nf);
    if (p->dist && p->slab_push) { pad_set_error("slab plan with peer buffers: a bare x pass is not part of the pipeline"); return PAD_ERR_ARG; }
    return launch_spass_local(p, s, axis, dir, fields, nf);
}
int launch_spass_local(pad_plan* p, cudaStream_t s, int axis, int dir, cd* const* fields, int nf) {
    SPassFields f;
    for (int i = 0; i < 4; ++i) f.f[i] = i < nf ? fields[i] : nullptr;
    const SPassGeom g = spass_geom(p, axis);
    const int L = axis == 0 ? p->n0 : p->n1;
#define SPASS_CASE(LL)                                                        \
    case LL:                                                                  \
        return dir < 0 ? launch_spass_L<LL, -1>(p, s, f, nf, g) : launch_spass_L<LL, +1>(p, s, f, nf, g);
    switch (L) {
        SPASS_CASE(64)
        SPASS_CASE(128)
        SPASS_CASE(256)
        SPASS_CASE(512)
    }
#undef SPASS_CASE
    pad_set_error("strided FFT pass: length %d not supported", L);
    return PAD_ERR_ARG;
}

template <int L, int NF, class Mix, bool PUSH = false, int NIN = NF, int NOUT = NF>
int launch_xmix_L(pad_plan* p, cudaStream_t s, const SPassFields& f, const SPassGeom& g, Mix mix, const XmixPush& push = XmixPush{}) {
    auto kern = xmix_kernel<L, NF, Mix, PUSH, NIN, NOUT>;
    using P = SPass<L, kXmixWide<L>>;
    constexpr int smem = spass_smem_bytes<L, kXmixWide<L>>(NF);
    static bool attr_done[64] = {false};
    if (!attr_done[p->device & 63]) {
        PAD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr_done[p->device & 63] = true;
    }
    // persistent CTAs: the kernel prefetches its next tile while it finishes the current one
    constexpr int by_smem = (227 * 1024) / (smem + 1024);
    constexpr int want_sm = xmix_ctas_per_sm<L, NF>();
    constexpr int per_sm = by_smem < want_sm ? by_smem : want_sm;
    static_assert(per_sm >= 1, "fused x pass: tile buffers do not fit in shared memory");
    const long long tiles = spass_tiles(g);
    long long grid = (tiles + P::TPC - 1) / P::TPC;
    if (grid > 148 * per_sm) grid = 148 * per_sm;
    kern<<<(unsigned)grid, P::THREADS, smem, s>>>(f, g, p->geom, mix, push);
    ++g_pad_launches;
    PAD_CUDA(cudaGetLastError());
    return PAD_OK;
}

// gradient (NIN = 1: one spectrum in, NF out) and divergence (NOUT = 1: NF in, one out) forms of the fused x pass;
// NF = 3: grad / div, NF = 4 (n0 <= 256): grad and Laplacian / div and Laplacian (semilocal functionals of lap n)
template <int NIN, int NOUT, class Mix, int NF = 3>
int launch_xmix3_io(pad_plan* p, cudaStream_t s, cd* const* fields, Mix mix) {
    if (p->dist) { pad_set_error("fused x pass (gradient / divergence form): single-GPU plans only"); return PAD_ERR_ARG; }
    SPassFields f;
    for (int i = 0; i < 4; ++i) f.f[i] = i < NF ? fields[i] : nullptr;
    const SPassGeom g = spass_geom(p, 0);
    switch (p->n0) {
        case 64: return launch_xmix_L<64, NF, Mix, false, NIN, NOUT>(p, s, f, g, mix);
        case 128: return launch_xmix_L<128, NF, Mix, false, NIN, NOUT>(p, s, f, g, mix);
        case 256: return launch_xmix_L<256, NF, Mix, false, NIN, NOUT>(p, s, f, g, mix);
        case 512:
            if constexpr (NF <= 3) return launch_xmix_L<512, NF, Mix, false, NIN, NOUT>(p, s, f, g, mix);
            break;              // four 512-point tiles do not fit in shared memory: the caller takes the cuFFT route
    }
    pad_set_error("fused x pass: length %d not supported", p->n0);
    return PAD_ERR_ARG;
}

template <int L, class Mix>
int launch_xone_L(pad_plan* p, cudaStream_t s, cd* field, const SPassGeom& g, Mix mix) {
    auto kern = xone_kernel<L, Mix>;
    constexpr int smem = spass_smem_bytes<L>(1);
    static bool attr_done[64] = {false};
    if (!attr_done[p->device & 63]) {
        PAD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr_done[p->device & 63] = true;
    }
    const long long tiles = spass_tiles(g);
    long long grid = (tiles + SPass<L>::TPC - 1) / SPass<L>::TPC;
    if (grid > (1 << 20)) grid = 1 << 20;
    kern<<<(unsigned)grid, 128, smem, s>>>(field, g, p->geom, mix);
    ++g_pad_launches;
    PAD_CUDA(cudaGetLastError());
    return PAD_OK;
}

// spec_f <- IFFT_x( mix( FFT_x(spec_0..NF-1) ) )
template <int NF, class Mix>
int launch_xmix(pad_plan* p, cudaStream_t s, cd* const* fields, Mix mix) {
    if constexpr (NF == 1 && Mix::kRing == 1) {
        // one field, computed multiplier: the two-transform plain pass (single-GPU plans, L <= 256)
        if (g_pad_xone && !p->dist && p->n0 <= 256) {
            const SPassGeom g1 = spass_geom(p, 0);
            switch (p->n0) {
                case 64: return launch_xone_L<64>(p, s, fields[0], g1, mix);
                case 128: return launch_xone_L<128>(p, s, fields[0], g1, mix);
                case 256: return launch_xone_L<256>(p, s, fields[0], g1, mix);
            }
        }
    }
    SPassFields f;
    for (int i = 0; i < 4; ++i) f.f[i] = i < NF ? fields[i] : nullptr;
    const SPassGeom g = spass_geom(p, 0);
    if (p->dist && p->slab_push) {
        // the fields live in the transposed buffers (the forward y passes pushed them there); results go to the owners' local buffers
        XmixPush push;
        for (int i = 0; i < NF; ++i) {
            const int fi = slab_field_index(p, fields[i]);
            if (fi < 0) { pad_set_error("fused x pass: field %d is not a registered slab buffer", i); return PAD_ERR_ARG; }
            f.f[i] = reinterpret_cast<cd*>(p->peer_T[fi][p->rank]);
            for (int r = 0; r < 8; ++r) push.peer[i][r] = r < p->world ? reinterpret_cast<cd*>(p->peer_B[fi][r]) : nullptr;
        }
        int lg = 0;
        while ((1 << lg) < p->n0_loc) ++lg;
        if ((1 << lg) != p->n0_loc) { pad_set_error("fused x pass on slabs: n0 / world = %d must be a power of two", p->n0_loc); return PAD_ERR_ARG; }
        push.n0_loc_log2 = lg; push.n1 = p->n1; push.y0 = p->rank * p->n1_loc;
        switch (p->n0) {
            case 64: return launch_xmix_L<64, NF, Mix, true>(p, s, f, g, mix, push);
            case 128: return launch_xmix_L<128, NF, Mix, true>(p, s, f, g, mix, push);
            case 256: return launch_xmix_L<256, NF, Mix, true>(p, s, f, g, mix, push);
            case 512: return launch_xmix_L<512, NF, Mix, true>(p, s, f, g, mix, push);
        }
        pad_set_error("fused x pass: length %d not supported", p->n0);
        return PAD_ERR_ARG;
    }
    switch (p->n0) {
        case 64: return launch_xmix_L<64, NF>(p, s, f, g, mix);
        case 128: return launch_xmix_L<128, NF>(p, s, f, g, mix);
        case 256: return launch_xmix_L<256, NF>(p, s, f, g, mix);
        case 512: return launch_xmix_L<512, NF>(p, s, f, g, mix);
    }
    pad_set_error("fused x pass: length %d not supported", p->n0);
    return PAD_ERR_ARG;
}

// reciprocal-space multipliers for the fused x pass (Mix concept: fft_strided.cuh)
struct MixWgc {                        // WGC99 3x3 kernel mix (functionals.py:968-981), kernels pre-scaled by 1/N
    static constexpr int kRing = 8;
    const double2* K4;                 // [(kx n1 + ky) nzp + z][2]: (W0, K1), (K2, K3)
    int fold;                          // orthorhombic cell: K(kx, ky, kz) = K(|kx|, |ky|, kz) bit for bit, so only the quarter
                                       // kx <= n0/2, ky <= n1/2 of the table is ever read (72 of 285 MB at 256^3: L2 sized)
    struct Coef { double2 a, b; };
    struct Line { size_t prow, kxs; int n0; };
    __device__ __forceinline__ Line line(const KGeom& g, int ky, int z) const {
        const int fy = ky <= g.n1 - ky ? ky : g.n1 - ky;
        return Line{(size_t)fy * g.nzp_pad + z, (size_t)g.n1_loc * g.nzp_pad, g.n0};
    }
    __device__ __forceinline__ Coef fetch(const Line& l, int kx, size_t pidx, bool live) const {
        Coef c;
        c.a = c.b = make_double2(0.0, 0.0);
        if (live) {
            if (fold) {
                const int fx = kx <= l.n0 - kx ? kx : l.n0 - kx;
                pidx = l.prow + (size_t)fx * l.kxs;
                c.a = __ldg(K4 + 2 * pidx); c.b = __ldg(K4 + 2 * pidx + 1);
            } else {
                c.a = __ldcs(K4 + 2 * pidx); c.b = __ldcs(K4 + 2 * pidx + 1);
            }
        }
        return c;
    }
    __device__ __forceinline__ void apply(const Coef& k, cd* q) const {
        const double w0 = k.a.x, k1 = k.a.y, k2 = k.b.x, k3 = k.b.y;
        const cd A = q[0], B = q[1], C = q[2];
        q[0] = cd{w0 * A.x + k1 * B.x + k2 * C.x, w0 * A.y + k1 * B.y + k2 * C.y};
        q[1] = cd{k1 * A.x + k3 * B.x, k1 * A.y + k3 * B.y};
        q[2] = cd{k2 * A.x, k2 * A.y};
    }
};
struct MixLaplace {                    // -k^2 / N   (functional_tools.py:209-227)
    static constexpr int kRing = 1;
    double inv_n;
    typedef double Coef;
    typedef KLine Line;
    __device__ __forceinline__ Line line(const KGeom& g, int ky, int z) const { return make_kline(g, ky, z); }
    __device__ __forceinline__ Coef fetch(const Line& l, int kx, size_t, bool live) const {
        if (!live) return 0.0;
        return -inv_n * kline_sym_even(l, kx, [](double k2) { return k2; });
    }
    __device__ __forceinline__ void apply(const Coef& m, cd* q) const { q[0] = cd{q[0].x * m, q[0].y * m}; }
};
struct MixCoulomb {                    // 4 pi / (k^2 N), 0 at k = 0   (functionals.py:49-72)
    static constexpr int kRing = 1;
    double inv_n;
    typedef double Coef;
    typedef KLine Line;
    __device__ __forceinline__ Line line(const KGeom& g, int ky, int z) const { return make_kline(g, ky, z); }
    __device__ __forceinline__ Coef fetch(const Line& l, int kx, size_t, bool live) const {
        if (!live) return 0.0;
        // k = 0 is the only point with k2 == 0 exactly (f0 = 0 and C = 0); anything else is > 0
        return inv_n * kline_sym_even(l, kx, [](double k2) { return k2 > 0.0 ? 4.0 * kPi / k2 : 0.0; });
    }
    __device__ __forceinline__ void apply(const Coef& m, cd* q) const { q[0] = cd{q[0].x * m, q[0].y * m}; }
};
struct MixScale {                      // plain 1/N (round-trip tests)
    static constexpr int kRing = 1;
    double m;
    typedef double Coef;
    struct Line {};
    __device__ __forceinline__ Line line(const KGeom&, int, int) const { return Line{}; }
    __device__ __forceinline__ Coef fetch(const Line&, int, size_t, bool) const { return m; }
    __device__ __forceinline__ void apply(const Coef& c, cd* q) const { q[0] = cd{q[0].x * c, q[0].y * c}; }
};

// single-GPU plans: any (n0, n1) (cuFFT does the (x, y) transform where the own strided passes do not cover the lengths);
// slab plans: only with the own passes and registered buffers (the y pass carries the transposition)
bool fast_shape(const pad_plan* p) {
    if (!(p->n2 == 128 || p->n2 == 256 || p->n2 == 512)) return false;
    if (!p->dist) return true;
    return g_pad_own_xy && spass_len_ok(p->n0) && spass_len_ok(p->n1) && p->slab_fast[0] != nullptr;
}

// dispatch on n2: M = n2/2; (M, TPL) in {(64, 8), (128, 16), (256, 32)}
#define ZDISPATCH(p, CALL)                                                  \
    do {                                                                    \
        if ((p)->n2 == 512) { constexpr int M = 256, TPL = 32; CALL; }      \
        else if ((p)->n2 == 256) { constexpr int M = 128, TPL = 16; CALL; } \
        else { constexpr int M = 64, TPL = 8; CALL; }                       \
    } while (0)

// ------------------------------------------------------------------------------------------------
//  functors
// ------------------------------------------------------------------------------------------------
struct GenCopy {                       // plain r2c of one real field
    static constexpr int NST = 1, NIN = 1;
    __device__ void stage(const double2* in, double* a, double* b) const { a[0] = in[0].x; b[0] = in[0].y; }
    template <int F>
    __device__ double field(const double* s) const { return s[0]; }
};

struct PostStore {                     // plain c2r of one real field
    static constexpr bool kDen = false, kVin = false;
    static constexpr int NST = 0;
    double* out;
    __device__ void apply(size_t g, double2, double2, const double* u0, const double* u1, double*, double*, double*) const {
        *reinterpret_cast<double2*>(out + g) = make_double2(u0[0], u1[0]);
    }
    // streamed kernel
    static constexpr int NACC = 0;
    typedef int Ctx;
    __device__ Ctx begin() const { return 0; }
    template <int F>
    __device__ void fold(const Ctx&, double, double, double*) const {}
    __device__ void finish(const Ctx&, size_t g, double2, const double*, const double*, double uA, double uB, double*, double*, double*) const {
        *reinterpret_cast<double2*>(out + g) = make_double2(uA, uB);
    }
};

// n^e for the first forward pass
// the same for the two points of a packed pair in ONE call: the two dependent chains (log polynomial, exp polynomial)
// are independent of each other, so the scheduler interleaves them -- the out-of-line per-point functions of round 1 were
// half of the inverse z kernel's instructions and mostly stalled on their own results (ncu: 'wait' on DFMA chains)
__device__ __noinline__ double2 pow_pos_pair(double2 n, double e) {
    if (fm_ok(n.x) && fm_ok(n.y)) {
        const double lx = fm_log(n.x), ly = fm_log(n.y);
        return make_double2(fm_exp(e * lx), fm_exp(e * ly));
    }
    return make_double2(exp(e * log(n.x)), exp(e * log(n.y)));
}
// two exponents, one log per point
__device__ __noinline__ void pow2_pos_pair(double2 n, double e1, double e2, double2& p1, double2& p2) {
    if (fm_ok(n.x) && fm_ok(n.y)) {
        const double lx = fm_log(n.x), ly = fm_log(n.y);
        p1 = make_double2(fm_exp(e1 * lx), fm_exp(e1 * ly));
        p2 = make_double2(fm_exp(e2 * lx), fm_exp(e2 * ly));
        return;
    }
    const double lx = log(n.x), ly = log(n.y);
    p1 = make_double2(exp(e1 * lx), exp(e1 * ly));
    p2 = make_double2(exp(e2 * lx), exp(e2 * ly));
}

__device__ __noinline__ double pow_pos_ool(double n, double e) {
    if (fm_ok(n)) return fm_exp(e * fm_log(n));
    return exp(e * log(n));
}

// WGC99, first forward pass: a = n^beta, a theta, a theta^2 / 2, chi = sqrt(n)   (functionals.py:974-981, :242-243)
struct GenWgcA {
    static constexpr int NST = 2, NIN = 1;      // staged: n, n^beta;  input: density
    const double* scal;
    double beta;
    __device__ void stage(const double2* in, double* a, double* b) const {
        const double2 pw = pow_pos_pair(in[0], beta);
        a[0] = in[0].x; a[1] = pw.x;
        b[0] = in[0].y; b[1] = pw.y;
    }
    template <int F>
    __device__ double field(const double* s) const {
        if constexpr (F == 0) return s[1];
        else if constexpr (F == 3) {
            if (fm_ok(s[0])) return fm_sqrt_from_rsqrt(s[0], fm_rsqrt(s[0]));
            return s[0] != 0.0 ? sqrt(s[0]) : 0.0;
        } else {
            const double th = s[0] - scal[S_NREF];
            return F == 1 ? s[1] * th : 0.5 * s[1] * th * th;
        }
    }
};

// WGC99, second forward pass: P = n^alpha (stored by the mid pass), P theta, P theta^2 / 2
struct GenWgcP {
    static constexpr int NST = 2, NIN = 2;      // staged: n, P;  inputs: density, P
    const double* scal;
    __device__ void stage(const double2* in, double* a, double* b) const {
        a[0] = in[0].x; a[1] = in[1].x;
        b[0] = in[0].y; b[1] = in[1].y;
    }
    template <int F>
    __device__ double field(const double* s) const {
        if constexpr (F == 0) return s[1];
        else {
            const double th = s[0] - scal[S_NREF];
            return F == 1 ? s[1] * th : 0.5 * s[1] * th * th;
        }
    }
};

// second forward batch of the fused term list: P, P theta, P theta^2 / 2 and the density itself (for the Hartree term)
struct GenWgcP4 {
    static constexpr int NST = 2, NIN = 2;
    const double* scal;
    __device__ void stage(const double2* in, double* a, double* b) const {
        a[0] = in[0].x; a[1] = in[1].x;
        b[0] = in[0].y; b[1] = in[1].y;
    }
    template <int F>
    __device__ double field(const double* s) const {
        if constexpr (F == 0) return s[1];
        else if constexpr (F == 3) return s[0];
        else {
            const double th = s[0] - scal[S_NREF];
            return F == 1 ? s[1] * th : 0.5 * s[1] * th * th;
        }
    }
};

// WGC99 mid pass: u1, u2, u3, lap(chi) -> energy densities, first half of the potential, P
struct MidOut {
    double v, P, e_tf, e_vw, e_nl;
};
// kept out of line: inlined 16 times per line the transcendental code alone overflows the instruction cache
__device__ __noinline__ MidOut wgc_mid_point(double n, double n_ref, double alpha, double u1, double u2, double u3, double lap) {
    MidOut o;
    const double th = n - n_ref;
    const double conv = u1 + th * (u2 + 0.5 * th * u3);
    if (fm_ok(n)) {
        // one log, two table exps and one rsqrt give n^alpha, n^(2/3), sqrt(n), 1/sqrt(n), 1/n
        const double l = fm_log(n);
        o.P = fm_exp(alpha * l);
        const double c2 = fm_exp((2.0 / 3.0) * l);
        const double y = fm_rsqrt(n);
        const double chi = fm_sqrt_from_rsqrt(n, y);
        o.e_tf = kCTF * n * c2;
        o.e_vw = chi * lap;
        o.e_nl = o.P * conv;
        o.v = (5.0 / 3.0) * kCTF * c2 - 0.5 * lap * y + kCTF * (alpha * o.P * (y * y) * conv + o.P * (u2 + th * u3));
        return o;
    }
    o.P = exp(alpha * log(n));
    const double c = cbrt(n);
    const double chi = n != 0.0 ? sqrt(n) : 0.0;
    o.e_tf = kCTF * n * c * c;
    o.e_vw = chi * lap;
    o.e_nl = o.P * conv;
    double v = (5.0 / 3.0) * kCTF * c * c;
    if (n != 0.0) v += -0.5 * lap / chi;
    v += kCTF * (alpha * o.P / n * conv + o.P * (u2 + th * u3));
    o.v = v;
    return o;
}

// streamed kernels: the three convolution fields are folded as they arrive into  conv = u1 + th u2 + th^2 u3 / 2  and
// w = u2 + th u3  (th = n - n_ref); both the mid and the final pass need exactly these two combinations
struct WgcCtx {
    double n_ref;
};
template <int F>
__device__ __forceinline__ void wgc_fold(const WgcCtx& c, double n, double u, double* a) {
    const double th = n - c.n_ref;
    if constexpr (F == 0) { a[0] = u; a[1] = 0.0; }
    else if constexpr (F == 1) { a[0] = fma(th, u, a[0]); a[1] = u; }
    else { a[0] = fma(0.5 * th * th, u, a[0]); a[1] = fma(th, u, a[1]); }
}
__device__ __noinline__ MidOut wgc_mid_point_cw(double n, double alpha, double conv, double w, double lap) {
    MidOut o;
    if (fm_ok(n)) {
        const double l = fm_log(n);
        o.P = fm_exp(alpha * l);
        const double c2 = fm_exp((2.0 / 3.0) * l);
        const double y = fm_rsqrt(n);
        const double chi = fm_sqrt_from_rsqrt(n, y);
        o.e_tf = kCTF * n * c2;
        o.e_vw = chi * lap;
        o.e_nl = o.P * conv;
        o.v = (5.0 / 3.0) * kCTF * c2 - 0.5 * lap * y + kCTF * (alpha * o.P * (y * y) * conv + o.P * w);
        return o;
    }
    o.P = exp(alpha * log(n));
    const double c = cbrt(n);
    const double chi = n != 0.0 ? sqrt(n) : 0.0;
    o.e_tf = kCTF * n * c * c;
    o.e_vw = chi * lap;
    o.e_nl = o.P * conv;
    double v = (5.0 / 3.0) * kCTF * c * c;
    if (n != 0.0) v += -0.5 * lap / chi;
    v += kCTF * (alpha * o.P / n * conv + o.P * w);
    o.v = v;
    return o;
}

// both points of a packed pair in one call (see pow_pos_pair); energy densities summed over the pair
struct MidOut2 {
    double2 v, P;
    double e_tf, e_vw, e_nl;
};
__device__ __noinline__ MidOut2 wgc_mid_pair(double2 n, double n_ref, double alpha, double2 u1, double2 u2, double2 u3, double2 lap) {
    MidOut2 o;
    if (fm_ok(n.x) && fm_ok(n.y)) {
        const double thx = n.x - n_ref, thy = n.y - n_ref;
        const double wx = u2.x + thx * u3.x, wy = u2.y + thy * u3.y;
        const double cvx = u1.x + thx * (u2.x + 0.5 * thx * u3.x), cvy = u1.y + thy * (u2.y + 0.5 * thy * u3.y);
        const double lx = fm_log(n.x), ly = fm_log(n.y);
        const double Px = fm_exp(alpha * lx), Py = fm_exp(alpha * ly);
        const double c2x = fm_exp((2.0 / 3.0) * lx), c2y = fm_exp((2.0 / 3.0) * ly);
        const double yx = fm_rsqrt(n.x), yy = fm_rsqrt(n.y);
        const double chx = fm_sqrt_from_rsqrt(n.x, yx), chy = fm_sqrt_from_rsqrt(n.y, yy);
        o.P = make_double2(Px, Py);
        o.e_tf = kCTF * (n.x * c2x + n.y * c2y);
        o.e_vw = chx * lap.x + chy * lap.y;
        o.e_nl = Px * cvx + Py * cvy;
        o.v.x = (5.0 / 3.0) * kCTF * c2x - 0.5 * lap.x * yx + kCTF * (alpha * Px * (yx * yx) * cvx + Px * wx);
        o.v.y = (5.0 / 3.0) * kCTF * c2y - 0.5 * lap.y * yy + kCTF * (alpha * Py * (yy * yy) * cvy + Py * wy);
        return o;
    }
    const MidOut a = wgc_mid_point(n.x, n_ref, alpha, u1.x, u2.x, u3.x, lap.x);
    const MidOut b = wgc_mid_point(n.y, n_ref, alpha, u1.y, u2.y, u3.y, lap.y);
    o.v = make_double2(a.v, b.v);
    o.P = make_double2(a.P, b.P);
    o.e_tf = a.e_tf + b.e_tf; o.e_vw = a.e_vw + b.e_vw; o.e_nl = a.e_nl + b.e_nl;
    return o;
}

struct PostWgcMid {
    static constexpr bool kDen = true, kVin = false;
    static constexpr int NST = 2;              // staged for the second forward batch (GenWgcP): n, P = n^alpha
    const double* scal;
    double* v_out;
    double* P_out;                             // null: P stays on chip (pipelined kernel with the forward part fused)
    double alpha;
    int accumulate, want_v;
    __device__ void apply(size_t g, double2 n, double2, const double* u0, const double* u1, double* acc, double* sta, double* stb) const {
        double2 vo = make_double2(0.0, 0.0);
        if (want_v && accumulate) vo = *reinterpret_cast<const double2*>(v_out + g);
        const double n_ref = scal[S_NREF];
        const MidOut2 o = wgc_mid_pair(n, n_ref, alpha, make_double2(u0[0], u1[0]), make_double2(u0[1], u1[1]), make_double2(u0[2], u1[2]),
                                       make_double2(u0[3], u1[3]));
        acc[0] += o.e_tf; acc[1] += o.e_vw; acc[2] += o.e_nl;
        sta[0] = n.x; sta[1] = o.P.x;
        stb[0] = n.y; stb[1] = o.P.y;
        if (want_v) {
            *reinterpret_cast<double2*>(v_out + g) = make_double2(vo.x + o.v.x, vo.y + o.v.y);
            if (P_out) *reinterpret_cast<double2*>(P_out + g) = o.P;
        }
    }
    // streamed kernel: fields u1, u2, u3 folded, lap(chi) last
    static constexpr int NACC = 2;
    typedef WgcCtx Ctx;
    __device__ Ctx begin() const { return WgcCtx{scal[S_NREF]}; }
    template <int F>
    __device__ void fold(const Ctx& c, double n, double u, double* a) const { wgc_fold<F>(c, n, u, a); }
    __device__ void finish(const Ctx&, size_t g, double2 n, const double* aA, const double* aB, double lapA, double lapB, double* acc,
                           double* sta, double* stb) const {
        double2 vo = make_double2(0.0, 0.0);
        if (want_v && accumulate) vo = *reinterpret_cast<const double2*>(v_out + g);
        const MidOut a = wgc_mid_point_cw(n.x, alpha, aA[0], aA[1], lapA);
        const MidOut b = wgc_mid_point_cw(n.y, alpha, aB[0], aB[1], lapB);
        acc[0] += a.e_tf; acc[1] += a.e_vw; acc[2] += a.e_nl;
        acc[0] += b.e_tf; acc[1] += b.e_vw; acc[2] += b.e_nl;
        sta[0] = n.x; sta[1] = a.P;
        stb[0] = n.y; stb[1] = b.P;
        if (want_v) {
            *reinterpret_cast<double2*>(v_out + g) = make_double2(vo.x + a.v, vo.y + b.v);
            if (P_out) *reinterpret_cast<double2*>(P_out + g) = make_double2(a.P, b.P);
        }
    }
};

// ---- fused term list (system.py:759-772 with WGC99 as the kinetic term): the local terms LDA exchange, Perdew-Zunger
//      correlation and IonElectron ride on the mid pass (they need n, n^(1/3), log n: all there), the Hartree term
//      is a fourth field of the second batch (n -> 4 pi / k^2 -> v_H, E_H = 1/2 sum n v_H) -----------------------------
struct MidOutT {
    double v, P, e_tf, e_vw, e_nl, e_loc;
};
__device__ __noinline__ MidOutT wgc_mid_point_total_cw(double n, double alpha, double conv, double wsum, double lap, int mask,
                                                      double vext) {
    MidOutT o;
    double e_loc = 0.0, v_loc = 0.0;
    if (fm_ok(n)) {
        const double l = fm_log(n);
        o.P = fm_exp(alpha * l);
        const double c2 = fm_exp((2.0 / 3.0) * l);
        const double y = fm_rsqrt(n);
        const double chi = fm_sqrt_from_rsqrt(n, y);
        const double inv_n = y * y;
        o.e_tf = kCTF * n * c2;
        o.e_vw = chi * lap;
        o.e_nl = o.P * conv;
        o.v = (5.0 / 3.0) * kCTF * c2 - 0.5 * lap * y + kCTF * (alpha * o.P * inv_n * conv + o.P * wsum);
        if (mask & (PAD_LOCAL_LDAX | PAD_LOCAL_PZC)) {
            const double c13 = c2 * c2 * inv_n;                       // n^(1/3)
            if (mask & PAD_LOCAL_LDAX) { e_loc += kCX * n * c13; v_loc += (4.0 / 3.0) * kCX * c13; }
            if (mask & PAD_LOCAL_PZC) {
                // pz_correlation (xc.cuh, functionals.py:1515-1521) with rs = kRS13 n^(-1/3) and log rs from the log above
                const double A = 0.0311, B = -0.048, C = 0.002, D = -0.0116;
                const double ga = -0.1423, b1 = 1.0529, b2 = 0.3334;
                const double rs = kRS13 * c2 * inv_n;
                if (rs < 1.0) {
                    const double lr = -0.47747065276706023 - (1.0 / 3.0) * l;
                    e_loc += n * (A * lr + B + C * rs * lr + D * rs);
                    v_loc += lr * (A + (2.0 / 3.0) * C * rs) + (B - A / 3.0) + rs / 3.0 * (2.0 * D - C);
                } else {
                    const double sr = sqrt(rs);
                    const double dn = 1.0 + b1 * sr + b2 * rs;
                    const double idn = 1.0 / dn;
                    e_loc += n * ga * idn;
                    v_loc += ga * (1.0 + (7.0 / 6.0) * b1 * sr + (4.0 / 3.0) * b2 * rs) * (idn * idn);
                }
            }
        }
    } else {
        o.P = exp(alpha * log(n));
        const double c = cbrt(n);
        const double chi = n != 0.0 ? sqrt(n) : 0.0;
        o.e_tf = kCTF * n * c * c;
        o.e_vw = chi * lap;
        o.e_nl = o.P * conv;
        double v = (5.0 / 3.0) * kCTF * c * c;
        if (n != 0.0) v += -0.5 * lap / chi;
        v += kCTF * (alpha * o.P / n * conv + o.P * wsum);
        o.v = v;
        if (mask & PAD_LOCAL_LDAX) { e_loc += kCX * n * c; v_loc += (4.0 / 3.0) * kCX * c; }
        if (mask & PAD_LOCAL_PZC) { const PZ r = pz_correlation(n, c); e_loc += r.e; v_loc += r.v; }
    }
    if (mask & PAD_LOCAL_IONEL) { e_loc += n * vext; v_loc += vext; }
    o.e_loc = e_loc;
    o.v += v_loc;
    return o;
}

__device__ __forceinline__ MidOutT wgc_mid_point_total(double n, double n_ref, double alpha, double u1, double u2, double u3,
                                                      double lap, int mask, double vext) {
    const double th = n - n_ref;
    return wgc_mid_point_total_cw(n, alpha, u1 + th * (u2 + 0.5 * th * u3), u2 + th * u3, lap, mask, vext);
}

struct PostWgcMidT {                           // NRED = 4: TF, vW, non-local, local terms
    static constexpr bool kDen = true, kVin = false;
    static constexpr int NST = 2;
    const double* scal;
    double* v_out;
    const double* v_ext;                       // IonElectron (may be null when the bit is not set)
    double* P_out;                             // null: P stays on chip (forward part fused)
    double alpha;
    int accumulate, mask;
    __device__ void apply(size_t g, double2 n, double2, const double* u0, const double* u1, double* acc, double* sta, double* stb) const {
        double2 vo = make_double2(0.0, 0.0), ve = make_double2(0.0, 0.0);
        if (accumulate) vo = *reinterpret_cast<const double2*>(v_out + g);
        if (mask & PAD_LOCAL_IONEL) ve = *reinterpret_cast<const double2*>(v_ext + g);
        const double n_ref = scal[S_NREF];
        const MidOutT a = wgc_mid_point_total(n.x, n_ref, alpha, u0[0], u0[1], u0[2], u0[3], mask, ve.x);
        const MidOutT b = wgc_mid_point_total(n.y, n_ref, alpha, u1[0], u1[1], u1[2], u1[3], mask, ve.y);
        acc[0] += a.e_tf; acc[1] += a.e_vw; acc[2] += a.e_nl; acc[3] += a.e_loc;
        acc[0] += b.e_tf; acc[1] += b.e_vw; acc[2] += b.e_nl; acc[3] += b.e_loc;
        sta[0] = n.x; sta[1] = a.P;
        stb[0] = n.y; stb[1] = b.P;
        *reinterpret_cast<double2*>(v_out + g) = make_double2(vo.x + a.v, vo.y + b.v);
        if (P_out) *reinterpret_cast<double2*>(P_out + g) = make_double2(a.P, b.P);
    }
    static constexpr int NACC = 2;
    typedef WgcCtx Ctx;
    __device__ Ctx begin() const { return WgcCtx{scal[S_NREF]}; }
    template <int F>
    __device__ void fold(const Ctx& c, double n, double u, double* a) const { wgc_fold<F>(c, n, u, a); }
    __device__ void finish(const Ctx&, size_t g, double2 n, const double* aA, const double* aB, double lapA, double lapB, double* acc,
                           double* sta, double* stb) const {
        double2 vo = make_double2(0.0, 0.0), ve = make_double2(0.0, 0.0);
        if (accumulate) vo = *reinterpret_cast<const double2*>(v_out + g);
        if (mask & PAD_LOCAL_IONEL) ve = *reinterpret_cast<const double2*>(v_ext + g);
        const MidOutT a = wgc_mid_point_total_cw(n.x, alpha, aA[0], aA[1], lapA, mask, ve.x);
        const MidOutT b = wgc_mid_point_total_cw(n.y, alpha, aB[0], aB[1], lapB, mask, ve.y);
        acc[0] += a.e_tf; acc[1] += a.e_vw; acc[2] += a.e_nl; acc[3] += a.e_loc;
        acc[0] += b.e_tf; acc[1] += b.e_vw; acc[2] += b.e_nl; acc[3] += b.e_loc;
        sta[0] = n.x; sta[1] = a.P;
        stb[0] = n.y; stb[1] = b.P;
        *reinterpret_cast<double2*>(v_out + g) = make_double2(vo.x + a.v, vo.y + b.v);
        if (P_out) *reinterpret_cast<double2*>(P_out + g) = make_double2(a.P, b.P);
    }
};

// WGC99 final pass: g1, g2, g3 -> second half of the potential
__device__ __noinline__ double wgc_fin_point(double n, double n_ref, double beta, double g1, double g2, double g3) {
    const double th = n - n_ref;
    double a, da;
    if (fm_ok(n)) {
        const double l = fm_log(n);
        a = fm_exp(beta * l);
        da = beta * fm_exp((beta - 1.0) * l);
    } else {
        a = exp(beta * log(n));
        da = beta * a / n;
    }
    return kCTF * (da * g1 + (da * th + a) * g2 + (0.5 * da * th * th + a * th) * g3);
}

__device__ __noinline__ double wgc_fin_point_cw(double n, double beta, double s1, double s2) {
    double a, da;
    if (fm_ok(n)) {
        const double l = fm_log(n);
        a = fm_exp(beta * l);
        da = beta * fm_exp((beta - 1.0) * l);
    } else {
        a = exp(beta * log(n));
        da = beta * a / n;
    }
    return kCTF * (da * s1 + a * s2);
}

__device__ __noinline__ double2 wgc_fin_pair(double2 n, double n_ref, double beta, double2 g1, double2 g2, double2 g3) {
    if (fm_ok(n.x) && fm_ok(n.y)) {
        const double thx = n.x - n_ref, thy = n.y - n_ref;
        const double lx = fm_log(n.x), ly = fm_log(n.y);
        const double ax = fm_exp(beta * lx), ay = fm_exp(beta * ly);
        const double dax = beta * fm_exp((beta - 1.0) * lx), day = beta * fm_exp((beta - 1.0) * ly);
        return make_double2(kCTF * (dax * g1.x + (dax * thx + ax) * g2.x + (0.5 * dax * thx * thx + ax * thx) * g3.x),
                            kCTF * (day * g1.y + (day * thy + ay) * g2.y + (0.5 * day * thy * thy + ay * thy) * g3.y));
    }
    return make_double2(wgc_fin_point(n.x, n_ref, beta, g1.x, g2.x, g3.x), wgc_fin_point(n.y, n_ref, beta, g1.y, g2.y, g3.y));
}

struct PostWgcFin {
    static constexpr bool kDen = true, kVin = true;
    static constexpr int NST = 0;
    const double* scal;
    double* v_out;
    double beta;
    __device__ void apply(size_t g, double2 n, double2 v, const double* u0, const double* u1, double*, double*, double*) const {
        const double n_ref = scal[S_NREF];
        const double2 f = wgc_fin_pair(n, n_ref, beta, make_double2(u0[0], u1[0]), make_double2(u0[1], u1[1]), make_double2(u0[2], u1[2]));
        v.x += f.x;
        v.y += f.y;
        *reinterpret_cast<double2*>(v_out + g) = v;
    }
    // streamed kernel: g1, g2 folded, g3 last; the first half of the potential is read from v_out itself
    static constexpr int NACC = 2;
    typedef WgcCtx Ctx;
    __device__ Ctx begin() const { return WgcCtx{scal[S_NREF]}; }
    template <int F>
    __device__ void fold(const Ctx& c, double n, double u, double* a) const { wgc_fold<F>(c, n, u, a); }
    __device__ void finish(const Ctx& c, size_t g, double2 n, const double* aA, const double* aB, double g3A, double g3B, double*,
                           double*, double*) const {
        double2 v = *reinterpret_cast<const double2*>(v_out + g);
        double a[2] = {aA[0], aA[1]}, b[2] = {aB[0], aB[1]};
        wgc_fold<2>(c, n.x, g3A, a);
        wgc_fold<2>(c, n.y, g3B, b);
        v.x += wgc_fin_point_cw(n.x, beta, a[0], a[1]);
        v.y += wgc_fin_point_cw(n.y, beta, b[0], b[1]);
        *reinterpret_cast<double2*>(v_out + g) = v;
    }
};

// Tail of the fused term list: c2r of the Hartree potential (4 pi n / k^2, the fourth field of the second batch) with the local
// terms of the list -- LDA exchange, Perdew-Zunger correlation, IonElectron -- evaluated on the same sweep.  A one-field inverse
// pass has the fp64 issue slots to spare that the mid pass (four fields, 255 registers, 8 warps / SM) does not: with the local
// terms inside the mid pass that kernel took 534 instead of 264 us at 256^3, and the four-field final pass 437 instead of
// 199 us.  NRED = 2: sum n v_H, sum of the local energy densities.
struct LocalOut {
    double e, v;
};
__device__ __noinline__ LocalOut local_terms_point(double n, int mask, double vext) {
    LocalOut o{0.0, 0.0};
    if (mask & (PAD_LOCAL_TF | PAD_LOCAL_LDAX | PAD_LOCAL_PZC)) {
        const double c = cbrt(n);
        if (mask & PAD_LOCAL_TF) { o.e += kCTF * n * c * c; o.v += (5.0 / 3.0) * kCTF * c * c; }
        if (mask & PAD_LOCAL_LDAX) { o.e += kCX * n * c; o.v += (4.0 / 3.0) * kCX * c; }
        if (mask & PAD_LOCAL_PZC) { const PZ r = pz_correlation(n, c); o.e += r.e; o.v += r.v; }
    }
    if (mask & PAD_LOCAL_IONEL) { o.e += n * vext; o.v += vext; }
    return o;
}
// the same terms from one table log per point (fastmath.cuh): n^(1/3), rs, sqrt(rs), log rs all come from log n
__device__ __forceinline__ LocalOut local_terms_fast(double n, int mask, double vext) {
    if (!fm_ok(n)) return local_terms_point(n, mask, vext);
    LocalOut o{0.0, 0.0};
    if (mask & (PAD_LOCAL_TF | PAD_LOCAL_LDAX | PAD_LOCAL_PZC)) {
        const double l = fm_log(n);
        const double c13 = fm_exp((1.0 / 3.0) * l);                    // n^(1/3)
        if (mask & PAD_LOCAL_TF) { o.e += kCTF * n * c13 * c13; o.v += (5.0 / 3.0) * kCTF * c13 * c13; }
        if (mask & PAD_LOCAL_LDAX) { o.e += kCX * n * c13; o.v += (4.0 / 3.0) * kCX * c13; }
        if (mask & PAD_LOCAL_PZC) {
            // pz_correlation (xc.cuh, functionals.py:1515-1521) with rs = kRS13 n^(-1/3)
            const double A = 0.0311, B = -0.048, C = 0.002, D = -0.0116;
            const double ga = -0.1423, b1 = 1.0529, b2 = 0.3334;
            const double y3 = fm_rsqrt(c13);                          // n^(-1/6)
            const double rs = kRS13 * (y3 * y3);
            if (rs < 1.0) {
                const double lr = -0.47747065276706023 - (1.0 / 3.0) * l;      // log rs
                o.e += n * (A * lr + B + C * rs * lr + D * rs);
                o.v += lr * (A + (2.0 / 3.0) * C * rs) + (B - A / 3.0) + rs / 3.0 * (2.0 * D - C);
            } else {
                const double sr = 0.78762331789974325 * y3;           // sqrt(rs) = sqrt(kRS13) n^(-1/6)
                const double dn = 1.0 + b1 * sr + b2 * rs;
                const double q = fm_rsqrt(dn);
                const double idn = q * q;
                o.e += n * ga * idn;
                o.v += ga * (1.0 + (7.0 / 6.0) * b1 * sr + (4.0 / 3.0) * b2 * rs) * (idn * idn);
            }
        }
    }
    if (mask & PAD_LOCAL_IONEL) { o.e += n * vext; o.v += vext; }
    return o;
}

// v += local terms, one block-reduced energy sum; two points per thread and iteration (16-byte accesses)
__global__ void __launch_bounds__(PAD_THREADS) local_fast_kernel(const double* __restrict__ den, const double* __restrict__ v_ext,
                                                                double* __restrict__ v /* may be null */, size_t n, int mask, int accumulate,
                                                                double* __restrict__ partials) {
    fm_load_tables();
    double acc[1] = {0.0};
    const size_t n2 = n / 2, stride = (size_t)gridDim.x * PAD_THREADS;
    for (size_t i = (size_t)blockIdx.x * PAD_THREADS + threadIdx.x; i < n2; i += stride) {
        const double2 d = reinterpret_cast<const double2*>(den)[i];
        double2 ve = make_double2(0.0, 0.0);
        if (mask & PAD_LOCAL_IONEL) ve = reinterpret_cast<const double2*>(v_ext)[i];
        const LocalOut a = local_terms_fast(d.x, mask, ve.x), b = local_terms_fast(d.y, mask, ve.y);
        acc[0] += a.e + b.e;
        if (v) {
            double2 vv = accumulate ? reinterpret_cast<double2*>(v)[i] : make_double2(0.0, 0.0);
            vv.x += a.v; vv.y += b.v;
            reinterpret_cast<double2*>(v)[i] = vv;
        }
    }
    if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
        const LocalOut a = local_terms_fast(den[n - 1], mask, (mask & PAD_LOCAL_IONEL) ? v_ext[n - 1] : 0.0);
        acc[0] += a.e;
        if (v) v[n - 1] = (accumulate ? v[n - 1] : 0.0) + a.v;
    }
    block_reduce_store<1>(acc, partials);
}

}  // namespace
// pad_eval_local (functionals.cu) for 16-byte aligned fields: the table-log kernel above (the log / exp tables live in this
// translation unit)
int pad_local_fast(pad_plan* p, const double* den, const double* v_ext, int mask, double* E_out, double* v_out, int accumulate, cudaStream_t s) {
    PAD_TRY(ensure_twiddles(p->device));
    const int grid = pad_grid_for(p->N / 2 > 0 ? p->N / 2 : 1);
    local_fast_kernel<<<grid, PAD_THREADS, 0, s>>>(den, v_ext, v_out, p->N, mask, accumulate, p->partials);
    ++g_pad_launches;
    PAD_CUDA(cudaGetLastError());
    if (E_out) {
        FinalizeArgs h;
        h.nblocks = grid; h.nterms = 1; h.accumulate = accumulate;
        for (int t = 0; t < PAD_MAX_RED; ++t) h.coef[t] = 0.0;
        h.coef[0] = p->dV;
        h.sums_out = nullptr;
        h.E_out = E_out;
        pad_launch_finalize(p, h, s);
    }
    return PAD_OK;
}
namespace {

struct PostHartreeLocal {
    static constexpr bool kDen = true, kVin = true;
    static constexpr int NST = 0;
    double* v_out;
    const double* v_ext;                       // IonElectron (may be null when the bit is not set)
    int mask;
    __device__ void apply(size_t g, double2 n, double2 v, const double* u0, const double* u1, double* acc, double*, double*) const {
        double2 ve = make_double2(0.0, 0.0);
        if (mask & PAD_LOCAL_IONEL) ve = *reinterpret_cast<const double2*>(v_ext + g);
        const LocalOut a = local_terms_point(n.x, mask, ve.x), b = local_terms_point(n.y, mask, ve.y);
        acc[0] += n.x * u0[0] + n.y * u1[0];
        acc[1] += a.e + b.e;
        *reinterpret_cast<double2*>(v_out + g) = make_double2(v.x + u0[0] + a.v, v.y + u1[0] + b.v);
    }
    static constexpr int NACC = 0;
    typedef int Ctx;
    __device__ Ctx begin() const { return 0; }
    template <int F>
    __device__ void fold(const Ctx&, double, double, double*) const {}
    __device__ void finish(const Ctx&, size_t g, double2 n, const double*, const double*, double uA, double uB, double* acc, double*,
                           double*) const {
        const double u0[1] = {uA}, u1[1] = {uB};
        apply(g, n, *reinterpret_cast<const double2*>(v_out + g), u0, u1, acc, nullptr, nullptr);
    }
};

struct PostWgcFinH {                           // final pass of the fused term list: + Hartree potential, NRED = 1: sum n v_H
    static constexpr bool kDen = true, kVin = true;
    static constexpr int NST = 0;
    const double* scal;
    double* v_out;
    double beta;
    __device__ void apply(size_t g, double2 n, double2 v, const double* u0, const double* u1, double* acc, double*, double*) const {
        const double n_ref = scal[S_NREF];
        const double2 f = wgc_fin_pair(n, n_ref, beta, make_double2(u0[0], u1[0]), make_double2(u0[1], u1[1]), make_double2(u0[2], u1[2]));
        v.x += f.x + u0[3];
        v.y += f.y + u1[3];
        acc[0] += n.x * u0[3] + n.y * u1[3];
        *reinterpret_cast<double2*>(v_out + g) = v;
    }
    static constexpr int NACC = 2;
    typedef WgcCtx Ctx;
    __device__ Ctx begin() const { return WgcCtx{scal[S_NREF]}; }
    template <int F>
    __device__ void fold(const Ctx& c, double n, double u, double* a) const { wgc_fold<F>(c, n, u, a); }
    __device__ void finish(const Ctx&, size_t g, double2 n, const double* aA, const double* aB, double vhA, double vhB, double* acc,
                           double*, double*) const {
        double2 v = *reinterpret_cast<const double2*>(v_out + g);
        v.x += wgc_fin_point_cw(n.x, beta, aA[0], aA[1]) + vhA;
        v.y += wgc_fin_point_cw(n.y, beta, aB[0], aB[1]) + vhB;
        acc[0] += n.x * vhA + n.y * vhB;
        *reinterpret_cast<double2*>(v_out + g) = v;
    }
};

// reciprocal-space kernel over the padded layout: f(unpadded index, padded index, kpoint)
template <class F>
__global__ void __launch_bounds__(PAD_THREADS) ksp_kernel(KGeom g, uint32_t nk, int nzp, F f) {
    const uint32_t stride = gridDim.x * PAD_THREADS;
    for (uint32_t idx = blockIdx.x * PAD_THREADS + threadIdx.x; idx < nk; idx += stride) {
        const KPoint k = make_kpoint(g, idx);
        const uint32_t row = idx / (uint32_t)g.nzh;
        f(idx, (size_t)row * nzp + (uint32_t)k.j2, k);
    }
}

template <class F>
void launch_ksp(pad_plan* p, cudaStream_t s, F f) {
    ksp_kernel<F><<<pad_grid_for(p->Nk), PAD_THREADS, 0, s>>>(p->geom, (uint32_t)p->Nk, p->nzp, f);
    ++g_pad_launches;
}


// (x, y) transform of nf padded half-spectra, in place: own strided passes where the shape allows, else cuFFT
int xy_transform(pad_plan* p, cudaStream_t s, cd* const* B, int nf, int dir) {
    if (g_pad_own_xy && own_xy_shape(p)) {
        if (dir < 0) {
            PAD_TRY(launch_spass(p, s, 1, -1, B, nf));
            PAD_TRY(launch_spass(p, s, 0, -1, B, nf));
        } else {
            PAD_TRY(launch_spass(p, s, 0, +1, B, nf));
            PAD_TRY(launch_spass(p, s, 1, +1, B, nf));
        }
        return PAD_OK;
    }
    for (int i = 0; i < nf; ++i) PAD_TRY(xy_exec(p, s, B[i], dir));
    return PAD_OK;
}

// y forward, fused x-forward/multiply/x-inverse, y inverse for the coupled fields B[0..NF-1] and,
// if lap != null, the independent field lap (multiplied by -k^2/N).
// (Blocking these passes over z-chunk groups so that a group stays in L2 was measured and dropped: the B200 L2
//  keeps ~64 MB between kernels at ~9 TB/s, a group of that size is 2 of 17 chunks, and launches that small
//  lose more to their tails than the L2 hits win; see DESIGN.md.)
template <int NF, class Mix>
int xy_convolve_own(pad_plan* p, cudaStream_t s, cd* const* B, cd* lap, Mix mix) {
    cd* all[4];
    int nall = 0;
    for (int i = 0; i < NF; ++i) all[nall++] = B[i];
    if (lap) all[nall++] = lap;
    PAD_TRY(launch_spass(p, s, 1, -1, all, nall));
    pad_stage_mark(lap ? "y-fwd (4 fields)" : "y-fwd (3 fields)", s);
    PAD_TRY((launch_xmix<NF>(p, s, B, mix)));
    pad_stage_mark("x-fwd * kernel-mix * x-inv (3 fields)", s);
    if (lap) {
        cd* one[1] = {lap};
        PAD_TRY((launch_xmix<1>(p, s, one, MixLaplace{p->geom.inv_n})));
        pad_stage_mark("x-fwd * (-k^2) * x-inv (1 field)", s);
    }
    PAD_TRY(launch_spass(p, s, 1, +1, all, nall));
    pad_stage_mark(lap ? "y-inv (4 fields)" : "y-inv (3 fields)", s);
    return PAD_OK;
}

}  // namespace

// =================================================================================================
//  public: custom 3-D r2c / c2r (used by tests and by pad_gradient-like helpers)
// =================================================================================================
extern "C" int pad_fast_fft_supported(const pad_plan* p) { return p && fast_shape(p) ? 1 : 0; }
extern "C" int pad_pipe_supported(const pad_plan* p) { return p && fast_shape(p) && pipe_shape(p) ? 1 : 0; }
extern "C" int pad_pipe_status(pad_plan* p, void* stream) {
    if (!p) { pad_set_error("pad_pipe_status: null plan"); return PAD_ERR_ARG; }
    if (!p->pipe_ctl) return -1;
    PAD_CUDA(cudaSetDevice(p->device));
    PAD_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    unsigned err = 0;
    PAD_CUDA(cudaMemcpy(&err, &reinterpret_cast<PipeCtl*>(p->pipe_ctl)->error, sizeof(err), cudaMemcpyDeviceToHost));
    return err ? 1 : 0;
}

// out: padded half-spectrum (n0, n1, nzp) complex; returns nzp through *nzp_out
extern "C" int pad_rfft3_fast(pad_plan* p, const double* in, double* out_cplx_padded, int* nzp_out, void* stream) {
    if (!p || !in || !out_cplx_padded) { pad_set_error("pad_rfft3_fast: null argument"); return PAD_ERR_ARG; }
    if (!fast_shape(p)) { pad_set_error("pad_rfft3_fast: n2 = %d not supported (128, 256, 512)", p->n2); return PAD_ERR_ARG; }
    PAD_CUDA(cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    PAD_TRY(ensure_twiddles(p->device));
    if (nzp_out) *nzp_out = p->nzp;
    cd* o = reinterpret_cast<cd*>(out_cplx_padded);
    GenCopy gen{};
    cd* one[1] = {o};
    if (pipe_shape(p)) {
        ZDISPATCH(p, PAD_TRY((launch_zy_fwd<M, TPL, 1>(p, s, gen, in, nullptr, one))));
        return launch_spass(p, s, 0, -1, one, 1);
    }
    ZDISPATCH(p, PAD_TRY((launch_zfwd<M, TPL, 1>(p, s, gen, in, nullptr, o, nullptr, nullptr, nullptr))));
    PAD_TRY(xy_transform(p, s, one, 1, -1));
    return PAD_OK;
}

// in: padded half-spectrum (destroyed); out: real field, unnormalised (N x the inverse)
extern "C" int pad_irfft3_fast(pad_plan* p, double* in_cplx_padded, double* out, void* stream) {
    if (!p || !in_cplx_padded || !out) { pad_set_error("pad_irfft3_fast: null argument"); return PAD_ERR_ARG; }
    if (!fast_shape(p)) { pad_set_error("pad_irfft3_fast: n2 = %d not supported (128, 256, 512)", p->n2); return PAD_ERR_ARG; }
    PAD_CUDA(cudaSetDevice(p->device));
    cudaStream_t s = (cudaStream_t)stream;
    PAD_TRY(ensure_twiddles(p->device));
    cd* i = reinterpret_cast<cd*>(in_cplx_padded);
    cd* one[1] = {i};
    PostStore post{out};
    if (pipe_shape(p)) {
        PAD_TRY(launch_spass(p, s, 0, +1, one, 1));
        ZDISPATCH(p, PAD_TRY((launch_yz_inv<M, TPL, 1, 0, PostStore, 0>(p, s, post, GenNone{}, one, nullptr, nullptr, nullptr))));
        return PAD_OK;
    }
    PAD_TRY(xy_transform(p, s, one, 1, +1));
    ZDISPATCH(p, PAD_TRY((launch_zinv<M, TPL, 1, 0>(p, s, post, i, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr))));
    return PAD_OK;
}

// =================================================================================================
//  WGC99 on the fused pipeline.  Called by pad_eval_wgc99 after the kernel cache and S_NREF are ready.
// =================================================================================================
int pad_wgc99_fast_supported(const pad_plan* p) { return fast_shape(p) ? 1 : 0; }

int pad_wgc99_total_supported(const pad_plan* p) { return fast_shape(p) && g_pad_own_xy && own_xy_shape(p) ? 1 : 0; }

namespace {
FinalizeArgs wgc_energy_args(const pad_plan* p, int nblocks, int nterms, int accumulate, double* E_out) {
    FinalizeArgs a;
    a.nblocks = nblocks; a.nterms = nterms; a.accumulate = accumulate;
    for (int t = 0; t < PAD_MAX_RED; ++t) a.coef[t] = 0.0;
    a.coef[0] = p->dV; a.coef[1] = -0.5 * p->dV; a.coef[2] = kCTF * p->dV; a.coef[3] = p->dV;
    a.sums_out = nullptr;
    a.E_out = E_out;
    return a;
}

// inverse y pass + [z c2r + post-op (+ gen + z r2c of NFW new fields) ] + forward y pass of the new fields: one pipelined
// kernel, or y^-1 | fused z kernel | y as three launches
template <int NF, int NRED, class Post, int NFW, class GenF>
int wgc_inverse_stage(pad_plan* p, cudaStream_t s, bool piped, Post post, GenF genf, cd* const* B, const double* den, const double* vin,
                      const FinalizeArgs* fin, const char* mark_yinv, const char* mark_z, const char* mark_yfwd, const char* mark_piped) {
    if (piped) {
        ZDISPATCH(p, PAD_TRY((launch_yz_inv<M, TPL, NF, NRED, Post, NFW>(p, s, post, genf, B, den, vin, fin))));
        pad_stage_mark(mark_piped, s);
        return PAD_OK;
    }
    PAD_TRY(launch_spass(p, s, 1, +1, B, NF));
    pad_stage_mark(mark_yinv, s);
    int grid = 1;
    ZDISPATCH(p, PAD_TRY((launch_zinv<M, TPL, NF, NRED, Post, NFW, GenF>(p, s, post, B[0], B[1], B[2], NF > 3 ? B[3] : nullptr, den, vin, &grid, genf))));
    pad_stage_mark(mark_z, s);
    if (NRED > 0 && fin) {
        FinalizeArgs a = *fin;
        a.nblocks = grid;
        pad_launch_finalize(p, a, s);
    }
    if (NFW > 0) {
        PAD_TRY(launch_spass(p, s, 1, -1, B, NFW));
        pad_stage_mark(mark_yfwd, s);
    }
    return PAD_OK;
}
}  // namespace

// ex != null: the fused term list (local terms in the mid pass, Hartree as a fourth field of the second batch)
int pad_wgc99_fast(pad_plan* p, const double* den, double alpha, double beta, const double* kern, double* E_out,
                   double* v_out, int accumulate, cudaStream_t s, const pad_wgc_extras* ex) {
    PAD_TRY(ensure_twiddles(p->device));
    const bool own = g_pad_own_xy && own_xy_shape(p);
    const bool want_v = v_out != nullptr;
    if (ex && !(own && want_v)) { pad_set_error("pad_wgc99_fast: the fused term list needs the own (x, y) passes and a potential"); return PAD_ERR_ARG; }
    if (!own) PAD_TRY(ensure_xy(p, s));
    cd* B[4];
    for (int i = 0; i < 4; ++i) PAD_TRY(get_zbuf(p, i, &B[i]));
    const double* scal = p->scal;
    const double inv_n = p->geom.inv_n;
    const KGeom geom = p->geom;
    // fold only where the fused x pass reads the table (own passes); the k-space kernel of the cuFFT (x, y) fallback indexes it plainly
    const bool ortho = p->recip[1] == 0.0 && p->recip[2] == 0.0 && p->recip[3] == 0.0 && p->recip[5] == 0.0 && p->recip[6] == 0.0 &&
                       p->recip[7] == 0.0;
    const MixWgc mixw{reinterpret_cast<const double2*>(kern), (g_pad_fold_table && ortho && own && !p->dist) ? 1 : 0};      // (a slab holds only its own rows of the table)
    GenWgcA genA{scal, beta};

    if (own && want_v) {
        // [gen + z + y] -> x.mix.x^-1 (+ Laplacian field) -> [y^-1 + z^-1 + mid + gen + z + y] -> x.mix.x^-1 (+ Coulomb field)
        //   -> [y^-1 + z^-1 + fin]; the bracketed groups are ONE pipelined kernel each (option "pipe") or y | z | y launches
        //   with the mid pass and the forward z pass of the second batch in one kernel
        const bool piped = pipe_shape(p);
        if (piped) {
            ZDISPATCH(p, PAD_TRY((launch_zy_fwd<M, TPL, 4>(p, s, genA, den, nullptr, B))));
            pad_stage_mark("[gen a,a.th,a.th2,chi + z-r2c + y-fwd] (4 fields)", s);
        } else {
            ZDISPATCH(p, PAD_TRY((launch_zfwd<M, TPL, 4>(p, s, genA, den, nullptr, B[0], B[1], B[2], B[3]))));
            pad_stage_mark("gen a,a.th,a.th2,chi + z-r2c (4 fields)", s);
            PAD_TRY(launch_spass(p, s, 1, -1, B, 4));
            pad_stage_mark("y-fwd (4 fields)", s);
        }
        PAD_TRY((launch_xmix<3>(p, s, B, mixw)));
        pad_stage_mark("x-fwd * kernel-mix * x-inv (3 fields)", s);
        {
            cd* one[1] = {B[3]};
            PAD_TRY((launch_xmix<1>(p, s, one, MixLaplace{inv_n})));
            pad_stage_mark("x-fwd * (-k^2) * x-inv (1 field)", s);
        }
        const bool hartree = ex && ex->hartree;
        const FinalizeArgs a = wgc_energy_args(p, 0, ex ? 4 : 3, accumulate, E_out);
        const FinalizeArgs* fa = E_out ? &a : nullptr;
        if (ex && !g_pad_fuse_mid && !piped && g_pad_local_tail) {
            // the plain (pair-optimised) WGC99 passes; the Hartree field rides along through y / x / y^-1 and is brought back by a
            // one-field inverse z pass of its own that also evaluates the local terms (PostHartreeLocal)
            double* Pbuf;
            PAD_TRY(pad_get_rbuf(p, 7, &Pbuf));
            const FinalizeArgs a3 = wgc_energy_args(p, 0, 3, accumulate, E_out);
            PostWgcMid mid{scal, v_out, Pbuf, alpha, accumulate, 1};
            PAD_TRY((wgc_inverse_stage<4, 3, PostWgcMid, 0>(p, s, false, mid, GenNone{}, B, den, nullptr, E_out ? &a3 : nullptr,
                                                           "y-inv (4 fields)", "z-c2r (4 fields) + energy/v1/P", "", "")));
            if (hartree) {
                ZDISPATCH(p, PAD_TRY((launch_zfwd<M, TPL, 4>(p, s, GenWgcP4{scal}, den, Pbuf, B[0], B[1], B[2], B[3]))));
                pad_stage_mark("gen P,P.th,P.th2,n + z-r2c (4 fields)", s);
            } else {
                ZDISPATCH(p, PAD_TRY((launch_zfwd<M, TPL, 3>(p, s, GenWgcP{scal}, den, Pbuf, B[0], B[1], B[2], nullptr))));
                pad_stage_mark("gen P,P.th,P.th2 + z-r2c (3 fields)", s);
            }
            const int nb = hartree ? 4 : 3;
            PAD_TRY(launch_spass(p, s, 1, -1, B, nb));
            pad_stage_mark(hartree ? "y-fwd (4 fields)" : "y-fwd (3 fields)", s);
            PAD_TRY((launch_xmix<3>(p, s, B, mixw)));
            pad_stage_mark("x-fwd * kernel-mix * x-inv (3 fields)", s);
            if (hartree) {
                cd* one[1] = {B[3]};
                PAD_TRY((launch_xmix<1>(p, s, one, MixCoulomb{inv_n})));
                pad_stage_mark("x-fwd * (4 pi / k^2) * x-inv (1 field)", s);
            }
            PAD_TRY(launch_spass(p, s, 1, +1, B, nb));
            pad_stage_mark(hartree ? "y-inv (4 fields)" : "y-inv (3 fields)", s);
            PostWgcFin fin{scal, v_out, beta};
            ZDISPATCH(p, PAD_TRY((launch_zinv<M, TPL, 3, 0>(p, s, fin, B[0], B[1], B[2], nullptr, den, v_out, nullptr))));
            pad_stage_mark("z-c2r (3 fields) + v2", s);
            // The local terms: inside the Hartree tail they cost 305 us at 256^3 (8 warps / SM: the dependent chains of the
            // transcendental functions have nothing to hide behind), in a full-occupancy elementwise kernel with the table
            // log / exp far less -- option local_tail = 2 keeps them in the tail.
            const bool aligned = ((reinterpret_cast<uintptr_t>(den) | reinterpret_cast<uintptr_t>(v_out) |
                                   reinterpret_cast<uintptr_t>(ex->v_ext)) & 15) == 0;
            const bool in_tail = hartree && (g_pad_local_tail == 2 || !aligned);
            if (hartree) {
                int grid = 1;
                PostHartreeLocal tail{v_out, ex->v_ext, in_tail ? ex->local_mask : 0};
                ZDISPATCH(p, PAD_TRY((launch_zinv<M, TPL, 1, 2>(p, s, tail, B[3], nullptr, nullptr, nullptr, den, v_out, &grid))));
                pad_stage_mark(in_tail ? "z-c2r (Hartree) + local terms" : "z-c2r (Hartree)", s);
                if (E_out) {
                    FinalizeArgs h = wgc_energy_args(p, grid, 2, 1, E_out);
                    h.coef[0] = 0.5 * p->dV; h.coef[1] = p->dV;
                    pad_launch_finalize(p, h, s);
                }
            }
            if (ex->local_mask && !in_tail) {
                if (aligned) {
                    const int grid = pad_grid_for(p->N / 2);
                    local_fast_kernel<<<grid, PAD_THREADS, 0, s>>>(den, ex->v_ext, v_out, p->N, ex->local_mask, 1, p->partials);
                    ++g_pad_launches;
                    PAD_CUDA(cudaGetLastError());
                    if (E_out) {
                        FinalizeArgs h = wgc_energy_args(p, grid, 1, 1, E_out);
                        h.coef[0] = p->dV;
                        pad_launch_finalize(p, h, s);
                    }
                } else {
                    PAD_TRY(pad_eval_local(p, den, ex->v_ext, ex->local_mask, E_out, v_out, 1, (void*)s));
                }
                pad_stage_mark("local terms", s);
            }
            return PAD_OK;
        }
        if (ex && !g_pad_fuse_mid && !piped) {
            // local terms in the mid pass; P = n^alpha goes through HBM to a separate (16 warps / SM) forward z kernel that
            // also transforms the density itself when the Hartree term is wanted
            double* Pbuf;
            PAD_TRY(pad_get_rbuf(p, 7, &Pbuf));
            PostWgcMidT mid{scal, v_out, ex->v_ext, Pbuf, alpha, accumulate, ex->local_mask};
            PAD_TRY((wgc_inverse_stage<4, 4, PostWgcMidT, 0>(p, s, false, mid, GenNone{}, B, den, nullptr, fa, "y-inv (4 fields)",
                                                            "z-c2r (4 fields) + energy/v1/local/P", "", "")));
            if (hartree) {
                ZDISPATCH(p, PAD_TRY((launch_zfwd<M, TPL, 4>(p, s, GenWgcP4{scal}, den, Pbuf, B[0], B[1], B[2], B[3]))));
                pad_stage_mark("gen P,P.th,P.th2,n + z-r2c (4 fields)", s);
                PAD_TRY(launch_spass(p, s, 1, -1, B, 4));
                pad_stage_mark("y-fwd (4 fields)", s);
            } else {
                ZDISPATCH(p, PAD_TRY((launch_zfwd<M, TPL, 3>(p, s, GenWgcP{scal}, den, Pbuf, B[0], B[1], B[2], nullptr))));
                pad_stage_mark("gen P,P.th,P.th2 + z-r2c (3 fields)", s);
                PAD_TRY(launch_spass(p, s, 1, -1, B, 3));
                pad_stage_mark("y-fwd (3 fields)", s);
            }
        } else if (ex && hartree) {
            PostWgcMidT mid{scal, v_out, ex->v_ext, nullptr, alpha, accumulate, ex->local_mask};
            PAD_TRY((wgc_inverse_stage<4, 4, PostWgcMidT, 4>(p, s, piped, mid, GenWgcP4{scal}, B, den, nullptr, fa, "y-inv (4 fields)",
                                                            "z-c2r (4) + energy/v1/local + gen P..,n + z-r2c (4)", "y-fwd (4 fields)",
                                                            "[y-inv (4) + z-c2r + energy/v1/local + gen P..,n + z-r2c + y-fwd (4)]")));
        } else if (ex) {
            PostWgcMidT mid{scal, v_out, ex->v_ext, nullptr, alpha, accumulate, ex->local_mask};
            PAD_TRY((wgc_inverse_stage<4, 4, PostWgcMidT, 3>(p, s, piped, mid, GenWgcP{scal}, B, den, nullptr, fa, "y-inv (4 fields)",
                                                            "z-c2r (4) + energy/v1/local + gen P.. + z-r2c (3)", "y-fwd (3 fields)",
                                                            "[y-inv (4) + z-c2r + energy/v1/local + gen P.. + z-r2c + y-fwd (3)]")));
        } else if (!g_pad_fuse_mid && !piped) {
            // mid pass and the forward z pass of the second batch as two kernels: P = n^alpha travels through HBM
            double* Pbuf;
            PAD_TRY(pad_get_rbuf(p, 7, &Pbuf));
            PostWgcMid mid{scal, v_out, Pbuf, alpha, accumulate, 1};
            PAD_TRY((wgc_inverse_stage<4, 3, PostWgcMid, 0>(p, s, false, mid, GenNone{}, B, den, nullptr, fa, "y-inv (4 fields)",
                                                           "z-c2r (4 fields) + energy/v1/P", "", "")));
            ZDISPATCH(p, PAD_TRY((launch_zfwd<M, TPL, 3>(p, s, GenWgcP{scal}, den, Pbuf, B[0], B[1], B[2], nullptr))));
            pad_stage_mark("gen P,P.th,P.th2 + z-r2c (3 fields)", s);
            PAD_TRY(launch_spass(p, s, 1, -1, B, 3));
            pad_stage_mark("y-fwd (3 fields)", s);
        } else {
            PostWgcMid mid{scal, v_out, nullptr, alpha, accumulate, 1};
            PAD_TRY((wgc_inverse_stage<4, 3, PostWgcMid, 3>(p, s, piped, mid, GenWgcP{scal}, B, den, nullptr, fa, "y-inv (4 fields)",
                                                           "z-c2r (4) + energy/v1 + gen P.. + z-r2c (3)", "y-fwd (3 fields)",
                                                           "[y-inv (4) + z-c2r + energy/v1 + gen P.. + z-r2c + y-fwd (3)]")));
        }
        PAD_TRY((launch_xmix<3>(p, s, B, mixw)));
        pad_stage_mark("x-fwd * kernel-mix * x-inv (3 fields)", s);
        if (hartree) {
            cd* one[1] = {B[3]};
            PAD_TRY((launch_xmix<1>(p, s, one, MixCoulomb{inv_n})));
            pad_stage_mark("x-fwd * (4 pi / k^2) * x-inv (1 field)", s);
            FinalizeArgs h = wgc_energy_args(p, 0, 1, 1, E_out);
            h.coef[0] = 0.5 * p->dV;
            PostWgcFinH fin{scal, v_out, beta};
            PAD_TRY((wgc_inverse_stage<4, 1, PostWgcFinH, 0>(p, s, piped, fin, GenNone{}, B, den, v_out, E_out ? &h : nullptr, "y-inv (4 fields)",
                                                            "z-c2r (4 fields) + v2 + Hartree", "", "[y-inv (4) + z-c2r + v2 + Hartree]")));
        } else {
            PostWgcFin fin{scal, v_out, beta};
            PAD_TRY((wgc_inverse_stage<3, 0, PostWgcFin, 0>(p, s, piped, fin, GenNone{}, B, den, v_out, nullptr, "y-inv (3 fields)",
                                                           "z-c2r (3 fields) + v2", "", "[y-inv (3) + z-c2r + v2]")));
        }
        return PAD_OK;
    }

    // energy only, or (x, y) lengths the own strided passes do not cover: one kernel per pass, cuFFT for (x, y) if needed
    double* Pbuf;
    PAD_TRY(pad_get_rbuf(p, 7, &Pbuf));
    ZDISPATCH(p, PAD_TRY((launch_zfwd<M, TPL, 4>(p, s, genA, den, nullptr, B[0], B[1], B[2], B[3]))));
    pad_stage_mark("gen a,a.th,a.th2,chi + z-r2c (4 fields)", s);
    if (own) {
        PAD_TRY((xy_convolve_own<3>(p, s, B, B[3], mixw)));
    } else {
        for (int i = 0; i < 4; ++i) PAD_TRY(xy_exec(p, s, B[i], -1));
        cd *CA = B[0], *CB = B[1], *CC = B[2], *CX = B[3];
        launch_ksp(p, s, [=] __device__(uint32_t idx, size_t pidx, const KPoint& k) {
            cd q[3] = {CA[pidx], CB[pidx], CC[pidx]};
            mixw.apply(mixw.fetch(MixWgc::Line{0, 0, 0}, 0, pidx, true), q);
            CA[pidx] = q[0]; CB[pidx] = q[1]; CC[pidx] = q[2];
            const double m = -inv_n * sym_even(k, [](double kx, double ky, double kz) { return kx * kx + ky * ky + kz * kz; });
            const cd X = CX[pidx];
            CX[pidx] = cd{X.x * m, X.y * m};
        });
        PAD_CUDA(cudaGetLastError());
        for (int i = 0; i < 4; ++i) PAD_TRY(xy_exec(p, s, B[i], +1));
    }
    int grid = 1;
    PostWgcMid mid{scal, v_out, Pbuf, alpha, accumulate, want_v ? 1 : 0};
    ZDISPATCH(p, PAD_TRY((launch_zinv<M, TPL, 4, 3>(p, s, mid, B[0], B[1], B[2], B[3], den, nullptr, &grid))));
    pad_stage_mark("z-c2r (4 fields) + energy/v1/P", s);
    if (E_out) pad_launch_finalize(p, wgc_energy_args(p, grid, 3, accumulate, E_out), s);
    if (!want_v) return PAD_OK;

    GenWgcP genP{scal};
    ZDISPATCH(p, PAD_TRY((launch_zfwd<M, TPL, 3>(p, s, genP, den, Pbuf, B[0], B[1], B[2], nullptr))));
    pad_stage_mark("gen P,P.th,P.th2 + z-r2c (3 fields)", s);
    for (int i = 0; i < 3; ++i) PAD_TRY(xy_exec(p, s, B[i], -1));
    {
        cd *CA = B[0], *CB = B[1], *CC = B[2];
        launch_ksp(p, s, [=] __device__(uint32_t idx, size_t pidx, const KPoint& k) {
            cd q[3] = {CA[pidx], CB[pidx], CC[pidx]};
            mixw.apply(mixw.fetch(MixWgc::Line{0, 0, 0}, 0, pidx, true), q);
            CA[pidx] = q[0]; CB[pidx] = q[1]; CC[pidx] = q[2];
        });
        PAD_CUDA(cudaGetLastError());
    }
    for (int i = 0; i < 3; ++i) PAD_TRY(xy_exec(p, s, B[i], +1));
    PostWgcFin fin{scal, v_out, beta};
    ZDISPATCH(p, PAD_TRY((launch_zinv<M, TPL, 3, 0>(p, s, fin, B[0], B[1], B[2], nullptr, den, v_out, nullptr))));
    pad_stage_mark("z-c2r (3 fields) + v2", s);
    return PAD_OK;
}

// =================================================================================================
//  Wang-Teter family (TF + vW + non-local term with the Lindhard kernel, functionals.py:644-725) on the fused
//  pipeline: ONE round trip -- [gen n^beta - n0^beta (, n^alpha - n0^alpha), chi + z r2c] -> y -> [x . (K | -k^2) . x^-1]
//  -> y^-1 -> [z c2r + energies + potential].  Called by pad_eval_wt after n0 and the kernel prefactor are in the
//  scalar block (S_TMP0 + 0..3: 1/(2 kF), 5 / (9 alpha beta n0^(alpha+beta-5/3)), n0^alpha, n0^beta).
// =================================================================================================
template <bool TWO>
struct GenWt {
    static constexpr int NST = 3, NIN = 1;      // staged: n, n^beta, n^alpha
    const double* scal;
    double alpha, beta;
    __device__ void stage(const double2* in, double* a, double* b) const {
        double2 pb, pa;
        if (TWO) pow2_pos_pair(in[0], beta, alpha, pb, pa);
        else pa = pb = pow_pos_pair(in[0], beta);
        a[0] = in[0].x; a[1] = pb.x; a[2] = pa.x;
        b[0] = in[0].y; b[1] = pb.y; b[2] = pa.y;
    }
    template <int F>
    __device__ double field(const double* s) const {
        if constexpr (F == 0) return s[1] - scal[S_TMP0 + 3];
        else if constexpr (TWO && F == 1) return s[2] - scal[S_TMP0 + 2];
        else {
            if (fm_ok(s[0])) return fm_sqrt_from_rsqrt(s[0], fm_rsqrt(s[0]));
            return s[0] != 0.0 ? sqrt(s[0]) : 0.0;
        }
    }
};

// 1 / G^-1(eta) - 3 eta^2 - 1 with the Lindhard function of functionals.py:617-628
__device__ __forceinline__ double lindhard_minus_z(double eta) {
    double ginv;
    if (eta == 0.0) ginv = 1.0;
    else if (eta == 1.0) ginv = 0.5;
    else ginv = 0.5 + ((1.0 - eta * eta) / (4.0 * eta)) * log(fabs((1.0 + eta) / (1.0 - eta)));
    return 1.0 / ginv - 3.0 * eta * eta - 1.0;
}

// Lindhard table of the fused Wang-Teter pipeline: depends on the lattice and on kF(n0) only; rebuilt when the lattice
// changes (host key) or n0 does (device key, as for the WGC99 kernel)
__global__ void __launch_bounds__(PAD_THREADS) wt_build_kernel(KGeom g, uint32_t nk, int nzp, double* __restrict__ table,
                                                              double* scal, int force) {
    if (!force && scal[S_N0] == scal[S_WT_KEY]) return;
    const double inv2kF = scal[S_TMP0 + 0];
    const uint32_t stride = gridDim.x * PAD_THREADS;
    for (uint32_t idx = blockIdx.x * PAD_THREADS + threadIdx.x; idx < nk; idx += stride) {
        const KPoint k = make_kpoint(g, idx);
        const uint32_t row = idx / (uint32_t)g.nzh;
        table[(size_t)row * nzp + (uint32_t)k.j2] = sym_even(k, [=](double x, double y, double w) {
            const double k2 = x * x + y * y + w * w;
            return lindhard_minus_z((k2 != 0.0 ? sqrt(k2) : 0.0) * inv2kF);
        });
    }
}
__global__ void wt_key_kernel(double* scal) { scal[S_WT_KEY] = scal[S_N0]; }

template <bool TWO>
struct MixWt {                         // fields 0 (, 1): Lindhard kernel / N;  last field: -k^2 / N
    static constexpr int kRing = 8;
    const double* scal;
    const double* table;               // [(kx n1 + ky) nzp + z]
    double inv_n;
    int fold;                          // orthorhombic cell: read only the |kx|, |ky| quarter of the table (see MixWgc)
    struct Coef { double nl, lap; };
    struct Line { KLine kl; size_t prow, kxs; };
    __device__ __forceinline__ Line line(const KGeom& g, int ky, int z) const {
        const int fy = ky <= g.n1 - ky ? ky : g.n1 - ky;
        return Line{make_kline(g, ky, z), (size_t)fy * g.nzp_pad + z, (size_t)g.n1_loc * g.nzp_pad};
    }
    __device__ __forceinline__ Coef fetch(const Line& l, int kx, size_t pidx, bool live) const {
        Coef c{0.0, 0.0};
        if (!live) return c;
        if (fold) {
            const int fx = kx <= l.kl.n0 - kx ? kx : l.kl.n0 - kx;
            c.nl = __ldg(table + l.prow + (size_t)fx * l.kxs);
        } else {
            c.nl = __ldcs(table + pidx);
        }
        c.lap = -inv_n * kline_sym_even(l.kl, kx, [](double k2) { return k2; });
        return c;
    }
    __device__ __forceinline__ void apply(const Coef& c, cd* q) const {
        const double m = c.nl * inv_n * scal[S_TMP0 + 1];
        q[0] = cd{q[0].x * m, q[0].y * m};
        if (TWO) q[1] = cd{q[1].x * m, q[1].y * m};
        constexpr int L = TWO ? 2 : 1;
        q[L] = cd{q[L].x * c.lap, q[L].y * c.lap};
    }
};

struct WtOut {
    double v, e_tf, e_vw, e_nl;
};
__device__ __noinline__ WtOut wt_point(double n, double alpha, double beta, bool two, double n0a, double conv_b, double conv_a,
                                      double lap) {
    WtOut o;
    if (fm_ok(n)) {
        const double l = fm_log(n);
        const double pb = fm_exp(beta * l);
        const double pa = two ? fm_exp(alpha * l) : pb;
        const double c2 = fm_exp((2.0 / 3.0) * l);
        const double y = fm_rsqrt(n);
        const double chi = fm_sqrt_from_rsqrt(n, y);
        o.e_tf = kCTF * n * c2;
        o.e_vw = chi * lap;
        o.e_nl = (pa - n0a) * conv_b;
        o.v = (5.0 / 3.0) * kCTF * c2 - 0.5 * lap * y + kCTF * (alpha * pa * conv_b + beta * pb * conv_a) * (y * y);
        return o;
    }
    const double ln = log(n);
    const double pb = exp(beta * ln);
    const double pa = two ? exp(alpha * ln) : pb;
    const double c = cbrt(n);
    const double chi = n != 0.0 ? sqrt(n) : 0.0;
    o.e_tf = kCTF * n * c * c;
    o.e_vw = chi * lap;
    o.e_nl = (pa - n0a) * conv_b;
    double v = (5.0 / 3.0) * kCTF * c * c;
    if (n != 0.0) v += -0.5 * lap / chi;
    v += kCTF * (alpha * pa * conv_b + beta * pb * conv_a) / n;
    o.v = v;
    return o;
}

struct WtOut2 {
    double2 v;
    double e_tf, e_vw, e_nl;
};
// both points of a packed pair in one call (independent chains interleave, see pow_pos_pair)
__device__ __noinline__ WtOut2 wt_pair(double2 n, double alpha, double beta, bool two, double n0a, double2 conv_b, double2 conv_a,
                                      double2 lap) {
    WtOut2 o;
    if (fm_ok(n.x) && fm_ok(n.y)) {
        const double lx = fm_log(n.x), ly = fm_log(n.y);
        const double pbx = fm_exp(beta * lx), pby = fm_exp(beta * ly);
        const double pax = two ? fm_exp(alpha * lx) : pbx, pay = two ? fm_exp(alpha * ly) : pby;
        const double c2x = fm_exp((2.0 / 3.0) * lx), c2y = fm_exp((2.0 / 3.0) * ly);
        const double yx = fm_rsqrt(n.x), yy = fm_rsqrt(n.y);
        const double chx = fm_sqrt_from_rsqrt(n.x, yx), chy = fm_sqrt_from_rsqrt(n.y, yy);
        o.e_tf = kCTF * (n.x * c2x + n.y * c2y);
        o.e_vw = chx * lap.x + chy * lap.y;
        o.e_nl = (pax - n0a) * conv_b.x + (pay - n0a) * conv_b.y;
        o.v.x = (5.0 / 3.0) * kCTF * c2x - 0.5 * lap.x * yx + kCTF * (alpha * pax * conv_b.x + beta * pbx * conv_a.x) * (yx * yx);
        o.v.y = (5.0 / 3.0) * kCTF * c2y - 0.5 * lap.y * yy + kCTF * (alpha * pay * conv_b.y + beta * pby * conv_a.y) * (yy * yy);
        return o;
    }
    const WtOut a = wt_point(n.x, alpha, beta, two, n0a, conv_b.x, conv_a.x, lap.x);
    const WtOut b = wt_point(n.y, alpha, beta, two, n0a, conv_b.y, conv_a.y, lap.y);
    o.v = make_double2(a.v, b.v);
    o.e_tf = a.e_tf + b.e_tf; o.e_vw = a.e_vw + b.e_vw; o.e_nl = a.e_nl + b.e_nl;
    return o;
}

template <bool TWO>
struct PostWt {
    static constexpr bool kDen = true, kVin = false;
    static constexpr int NST = 0;
    const double* scal;
    double* v_out;
    double alpha, beta;
    int accumulate, want_v;
    __device__ void apply(size_t g, double2 n, double2, const double* u0, const double* u1, double* acc, double*, double*) const {
        constexpr int L = TWO ? 2 : 1;
        const double n0a = scal[S_TMP0 + 2];
        const WtOut2 o = wt_pair(n, alpha, beta, TWO, n0a, make_double2(u0[0], u1[0]),
                                 TWO ? make_double2(u0[1], u1[1]) : make_double2(u0[0], u1[0]), make_double2(u0[L], u1[L]));
        acc[0] += o.e_tf; acc[1] += o.e_vw; acc[2] += o.e_nl;
        if (want_v) {
            double2 vo = make_double2(0.0, 0.0);
            if (accumulate) vo = *reinterpret_cast<const double2*>(v_out + g);
            *reinterpret_cast<double2*>(v_out + g) = make_double2(vo.x + o.v.x, vo.y + o.v.y);
        }
    }
    // streamed kernel: the convolution(s) are kept as they are, lap(chi) last
    static constexpr int NACC = TWO ? 2 : 1;
    struct Ctx { double n0a; };
    __device__ Ctx begin() const { return Ctx{scal[S_TMP0 + 2]}; }
    template <int F>
    __device__ void fold(const Ctx&, double, double u, double* a) const { a[F < NACC ? F : 0] = u; }
    __device__ void finish(const Ctx& c, size_t g, double2 n, const double* aA, const double* aB, double lapA, double lapB, double* acc,
                           double*, double*) const {
        const WtOut a = wt_point(n.x, alpha, beta, TWO, c.n0a, aA[0], TWO ? aA[NACC - 1] : aA[0], lapA);
        const WtOut b = wt_point(n.y, alpha, beta, TWO, c.n0a, aB[0], TWO ? aB[NACC - 1] : aB[0], lapB);
        acc[0] += a.e_tf; acc[1] += a.e_vw; acc[2] += a.e_nl;
        acc[0] += b.e_tf; acc[1] += b.e_vw; acc[2] += b.e_nl;
        if (want_v) {
            double2 vo = make_double2(0.0, 0.0);
            if (accumulate) vo = *reinterpret_cast<const double2*>(v_out + g);
            *reinterpret_cast<double2*>(v_out + g) = make_double2(vo.x + a.v, vo.y + b.v);
        }
    }
};

template <bool TWO>
static int wt_fast_impl(pad_plan* p, const double* den, double alpha, double beta, double* E_out, double* v_out,
                        int accumulate, cudaStream_t s) {
    constexpr int NF = TWO ? 3 : 2;
    PAD_TRY(ensure_twiddles(p->device));
    cd* B[4] = {nullptr, nullptr, nullptr, nullptr};
    for (int i = 0; i < NF; ++i) PAD_TRY(get_zbuf(p, i, &B[i]));
    const double* scal = p->scal;
    pad_stage_begin(s);
    {   // Lindhard table (padded layout), cached per lattice and n0
        bool fresh = false;
        if (!p->wt_kern) {
            const size_t bytes = sizeof(double) * (size_t)p->n0 * (p->dist ? p->n1_loc : p->n1) * p->nzp;      // the plan's own rows
            PAD_CUDA(cudaMalloc(&p->wt_kern, bytes));
            PAD_CUDA(cudaMemsetAsync(p->wt_kern, 0, bytes, s));
            p->bytes_allocated += bytes;
            fresh = true;
        }
        const bool same = !fresh && p->wt_kern_generation == p->box_generation;
        p->wt_kern_generation = p->box_generation;
        wt_build_kernel<<<same ? 148 : pad_grid_for(p->Nk), PAD_THREADS, 0, s>>>(p->geom, (uint32_t)p->Nk, p->nzp, p->wt_kern, p->scal, same ? 0 : 1);
        wt_key_kernel<<<1, 1, 0, s>>>(p->scal);
        g_pad_launches += 2;
        PAD_CUDA(cudaGetLastError());
    }
    pad_stage_mark("WT: Lindhard table check", s);
    GenWt<TWO> gen{scal, alpha, beta};
    const int wt_fold = (g_pad_fold_table && !p->dist && p->recip[1] == 0.0 && p->recip[2] == 0.0 && p->recip[3] == 0.0 && p->recip[5] == 0.0 &&
                         p->recip[6] == 0.0 && p->recip[7] == 0.0) ? 1 : 0;
    if (pipe_shape(p)) {
        ZDISPATCH(p, PAD_TRY((launch_zy_fwd<M, TPL, NF>(p, s, gen, den, nullptr, B))));
        pad_stage_mark("WT: [gen fields + z-r2c + y-fwd]", s);
        PAD_TRY((launch_xmix<NF>(p, s, B, MixWt<TWO>{scal, p->wt_kern, p->geom.inv_n, wt_fold})));
        pad_stage_mark("WT: x-fwd * (Lindhard | -k^2) * x-inv", s);
        FinalizeArgs a;
        a.nblocks = 0; a.nterms = 3; a.accumulate = accumulate;
        for (int t = 0; t < PAD_MAX_RED; ++t) a.coef[t] = 0.0;
        a.coef[0] = p->dV; a.coef[1] = -0.5 * p->dV; a.coef[2] = kCTF * p->dV;
        a.sums_out = nullptr;
        a.E_out = E_out;
        PostWt<TWO> post{scal, v_out, alpha, beta, accumulate, v_out ? 1 : 0};
        ZDISPATCH(p, PAD_TRY((launch_yz_inv<M, TPL, NF, 3, PostWt<TWO>, 0>(p, s, post, GenNone{}, B, den, nullptr, E_out ? &a : nullptr))));
        pad_stage_mark("WT: [y-inv + z-c2r + energies + potential]", s);
        return PAD_OK;
    }
    ZDISPATCH(p, PAD_TRY((launch_zfwd<M, TPL, NF>(p, s, gen, den, nullptr, B[0], B[1], B[2], nullptr))));
    pad_stage_mark("WT: gen fields + z-r2c", s);
    PAD_TRY(launch_spass(p, s, 1, -1, B, NF));
    pad_stage_mark("WT: y-fwd", s);
    PAD_TRY((launch_xmix<NF>(p, s, B, MixWt<TWO>{scal, p->wt_kern, p->geom.inv_n, wt_fold})));
    pad_stage_mark("WT: x-fwd * (Lindhard | -k^2) * x-inv", s);
    PAD_TRY(launch_spass(p, s, 1, +1, B, NF));
    pad_stage_mark("WT: y-inv", s);
    int grid = 1;
    PostWt<TWO> post{scal, v_out, alpha, beta, accumulate, v_out ? 1 : 0};
    ZDISPATCH(p, PAD_TRY((launch_zinv<M, TPL, NF, 3>(p, s, post, B[0], B[1], B[2], nullptr, den, nullptr, &grid))));
    pad_stage_mark("WT: z-c2r + energies + potential", s);
    if (E_out) {
        FinalizeArgs a;
        a.nblocks = grid; a.nterms = 3; a.accumulate = accumulate;
        for (int t = 0; t < PAD_MAX_RED; ++t) a.coef[t] = 0.0;
        a.coef[0] = p->dV; a.coef[1] = -0.5 * p->dV; a.coef[2] = kCTF * p->dV;
        a.sums_out = nullptr;
        a.E_out = E_out;
        pad_launch_finalize(p, a, s);
    }
    return PAD_OK;
}

// =================================================================================================
//  PerdewBurkeErnzerhof (functionals.py:1597-1635) on the fused passes: 8 transforms in 9 launches
//     [z r2c of n] -> y -> [x . (i k_c / N, c = x, y, z) . x^-1: one spectrum in, three out] -> y^-1 (3)
//       -> [z c2r (3) + PBE energy density, f_n -> v, w_c = 2 f_sigma d_c n + z r2c (3)] -> y (3)
//       -> [x . (i k . w / N) . x^-1: three in, one out] -> y^-1 -> [z c2r: v -= div w]
//  The multipliers i k_c use the effective wave vector of the special points (sym_kvec), as the cuFFT route does.
// =================================================================================================
struct MixGradCoef {
    double kx, ky, kz;
};
struct MixGrad {                       // q[0] = F  ->  q[c] = i k_c F / N
    static constexpr int kRing = 1;
    double inv_n;
    typedef MixGradCoef Coef;
    struct Line { const KGeom* g; int ky, z; };
    __device__ __forceinline__ Line line(const KGeom& g, int ky, int z) const { return Line{&g, ky, z}; }
    __device__ __forceinline__ Coef fetch(const Line& l, int kx, size_t, bool live) const {
        Coef c{0.0, 0.0, 0.0};
        if (live) {
            const KPoint p = make_kpoint_at(*l.g, kx, l.ky, l.z);
            sym_kvec(p, c.kx, c.ky, c.kz);
            c.kx *= inv_n; c.ky *= inv_n; c.kz *= inv_n;
        }
        return c;
    }
    __device__ __forceinline__ void apply(const Coef& k, cd* q) const {
        const cd a = q[0];
        q[0] = cd{-a.y * k.kx, a.x * k.kx};
        q[1] = cd{-a.y * k.ky, a.x * k.ky};
        q[2] = cd{-a.y * k.kz, a.x * k.kz};
    }
};
struct MixDiv {                        // q[0] = i (k . (q0, q1, q2)) / N
    static constexpr int kRing = 1;
    double inv_n;
    typedef MixGradCoef Coef;
    typedef MixGrad::Line Line;
    __device__ __forceinline__ Line line(const KGeom& g, int ky, int z) const { return Line{&g, ky, z}; }
    __device__ __forceinline__ Coef fetch(const Line& l, int kx, size_t pidx, bool live) const { return MixGrad{inv_n}.fetch(l, kx, pidx, live); }
    __device__ __forceinline__ void apply(const Coef& k, cd* q) const {
        const double re = k.kx * q[0].x + k.ky * q[1].x + k.kz * q[2].x, im = k.kx * q[0].y + k.ky * q[1].y + k.kz * q[2].y;
        q[0] = cd{-im, re};
    }
};

struct PbeOut {
    double f, f_rho, wx, wy, wz;
};
__device__ __noinline__ PbeOut pbe_point_w(double n, double gx, double gy, double gz, int which) {
    PbeOut o;
    double f_sig;
    pbe_point(n, gx * gx + gy * gy + gz * gz, cbrt(n), (which & 1) != 0, (which & 2) != 0, o.f, o.f_rho, f_sig);
    const double w = 2.0 * f_sig;
    o.wx = w * gx; o.wy = w * gy; o.wz = w * gz;
    return o;
}
// The PBE point math does NOT ride on the inverse z pass: with it inside (and the forward z transform of w behind it, one
// kernel, 255 registers, 8 warps per SM) that kernel took 1140 us at 256^3 -- the transcendental chains have nothing to hide
// behind at that occupancy (the same finding as for the local terms of the WGC99 list).  So: a plain three-field inverse z pass
// stores the gradient, a full-occupancy elementwise kernel does the point math in place (grad n -> w), a three-input forward z
// pass transforms w.
struct PostStore3 {                    // plain c2r of three real fields
    static constexpr bool kDen = false, kVin = false;
    static constexpr int NST = 0;
    double *o0, *o1, *o2;
    __device__ void apply(size_t g, double2, double2, const double* u0, const double* u1, double*, double*, double*) const {
        *reinterpret_cast<double2*>(o0 + g) = make_double2(u0[0], u1[0]);
        *reinterpret_cast<double2*>(o1 + g) = make_double2(u0[1], u1[1]);
        *reinterpret_cast<double2*>(o2 + g) = make_double2(u0[2], u1[2]);
    }
    static constexpr int NACC = 0;
    typedef int Ctx;
    __device__ Ctx begin() const { return 0; }
    template <int F>
    __device__ void fold(const Ctx&, double, double, double*) const {}
    __device__ void finish(const Ctx&, size_t, double2, const double*, const double*, double, double, double*, double*, double*) const {}
};
struct GenCopy3 {                      // plain r2c of three real fields
    static constexpr int NST = 3, NIN = 3;
    __device__ void stage(const double2* in, double* a, double* b) const {
        a[0] = in[0].x; a[1] = in[1].x; a[2] = in[2].x;
        b[0] = in[0].y; b[1] = in[1].y; b[2] = in[2].y;
    }
    template <int F>
    __device__ double field(const double* s) const { return s[F]; }
};
// pbe_point (xc.cuh) with the table log / exp and rsqrt-based reciprocals of fastmath.cuh: one log of n gives n^(1/3), r_s and
// sqrt(r_s); the library version (cbrt, sqrt, two logs, an exp and a dozen divisions) was 621 us of the 1.81 ms of a 256^3
// evaluation at full occupancy.  Same formulas, same +1e-30 guards; arguments outside the fast range take pbe_point.
__device__ __forceinline__ double fm_recip(double x) {
    const double y = fm_rsqrt(x);
    return y * y;
}
__device__ __forceinline__ void pbe_point_fast(double n, double sig, bool do_x, bool do_c, double& f, double& f_rho, double& f_sig) {
    if (!(n > 1e-20 && n < 1e20 && sig < 1e40)) {          // (keeps every intermediate of the fast path far from the exponent limits)
        pbe_point(n, sig, cbrt(n), do_x, do_c, f, f_rho, f_sig);
        return;
    }
    f = 0.0; f_rho = 0.0; f_sig = 0.0;
    const double l = fm_log(n);
    const double c13 = fm_exp((1.0 / 3.0) * l);
    const double inv_n = fm_recip(n);
    if (do_x) {
        const double cs = 0.026121172985233605;       // (1/4)(3 pi^2)^(-2/3)
        const double kap = 0.804, mu = 0.2195164512208958;
        const double ex = kCX * n * c13;
        const double r83 = n * n * c13 * c13;
        const double ir83 = fm_recip(r83);
        const double s2 = cs * sig * ir83;
        const double q = 1.0 + mu / kap * s2;
        const double iq = fm_recip(q);
        const double Fx = 1.0 + kap - kap * iq, dF = mu * (iq * iq);
        f += Fx * ex;
        f_rho += Fx * (4.0 / 3.0) * kCX * c13 + ex * dF * (-8.0 / 3.0) * s2 * inv_n;
        f_sig += ex * dF * cs * ir83;
    }
    if (do_c) {
        const double A1 = 0.0310907, a1 = 0.2137, b1 = 7.5957, b2 = 3.5876, b3 = 1.6382, b4 = 0.49294;
        const double be = 0.066725, ga = 0.0310906908696549;   // (1 - ln 2) / pi^2
        const double ct = 0.0634682060977037;                  // (1/16)(pi/3)^(1/3)
        const double s6 = fm_exp((-1.0 / 6.0) * l);            // n^(-1/6)
        const double sr = 0.78762331789974325 * s6;           // sqrt(r_s) = sqrt(kRS13) n^(-1/6)
        const double rs = sr * sr;
        const double isr = fm_recip(sr);
        const double Q = 2.0 * A1 * (b1 * sr + b2 * rs + b3 * rs * sr + b4 * rs * rs);
        const double iQ = fm_recip(Q);
        const double lg = fm_log(1.0 + iQ);
        const double eps = -2.0 * A1 * (1.0 + a1 * rs) * lg;
        const double dQ = A1 * (b1 * isr + 2.0 * b2 + 3.0 * b3 * sr + 4.0 * b4 * rs);
        const double deps = (-2.0 * A1 * a1 * lg + 2.0 * A1 * (1.0 + a1 * rs) * dQ * fm_recip(Q * (Q + 1.0))) * (-rs * inv_n * (1.0 / 3.0));
        const double ee = fm_exp(-eps * (1.0 / ga));
        const double em1 = ee - 1.0 + 1e-30;
        if (!(em1 > 1e-20)) {           // r_s -> infinity: leave the cancellation to the library path
            double f2, r2, s2_;
            pbe_point(n, sig, c13, false, true, f2, r2, s2_);
            f += f2; f_rho += r2; f_sig += s2_;
            return;
        }
        const double Aa = be / ga * fm_recip(em1);
        const double dAa = Aa * Aa / be * ee * deps;
        const double r73 = n * n * c13 + 1e-30;
        const double ir73 = fm_recip(r73);
        const double t2 = ct * sig * ir73;
        const double dt2_rho = -ct * sig * (7.0 / 3.0) * n * c13 * (ir73 * ir73);
        const double dt2_sig = ct * ir73;
        const double X = Aa * t2;
        const double num = 1.0 + X, dnm = 1.0 + X + X * X;
        const double idnm = fm_recip(dnm);
        const double Rr = num * idnm;
        const double dR = -X * (2.0 + X) * (idnm * idnm);
        const double inner = 1.0 + be / ga * t2 * Rr;
        const double H = ga * fm_log(inner);
        const double iinner = fm_recip(inner);
        const double dH_rho = be * iinner * (Rr * dt2_rho + t2 * dR * (Aa * dt2_rho + t2 * dAa));
        const double dH_sig = be * iinner * (Rr + t2 * dR * Aa) * dt2_sig;
        f += n * (eps + H);
        f_rho += eps + H + n * (deps + dH_rho);
        f_sig += n * dH_sig;
    }
}

// n, grad n -> energy density (one block-reduced sum), v (+)= f_n, grad n <- w = 2 f_sigma grad n; two points per thread
__global__ void __launch_bounds__(PAD_THREADS) pbe_point_kernel(const double* __restrict__ den, double* __restrict__ gx, double* __restrict__ gy,
                                                               double* __restrict__ gz, double* __restrict__ v, size_t n, int which,
                                                               int accumulate, double* __restrict__ partials) {
    fm_load_tables();
    double acc[1] = {0.0};
    const size_t n2 = n / 2, stride = (size_t)gridDim.x * PAD_THREADS;
    for (size_t i = (size_t)blockIdx.x * PAD_THREADS + threadIdx.x; i < n2; i += stride) {
        const double2 d = reinterpret_cast<const double2*>(den)[i];
        double2 x = reinterpret_cast<double2*>(gx)[i], y = reinterpret_cast<double2*>(gy)[i], z = reinterpret_cast<double2*>(gz)[i];
        double fa, ra, sa, fb, rb, sb;
        pbe_point_fast(d.x, x.x * x.x + y.x * y.x + z.x * z.x, (which & 1) != 0, (which & 2) != 0, fa, ra, sa);
        pbe_point_fast(d.y, x.y * x.y + y.y * y.y + z.y * z.y, (which & 1) != 0, (which & 2) != 0, fb, rb, sb);
        acc[0] += fa + fb;
        if (v) {
            double2 vv = accumulate ? reinterpret_cast<double2*>(v)[i] : make_double2(0.0, 0.0);
            vv.x += ra; vv.y += rb;
            reinterpret_cast<double2*>(v)[i] = vv;
            sa *= 2.0; sb *= 2.0;
            reinterpret_cast<double2*>(gx)[i] = make_double2(sa * x.x, sb * x.y);
            reinterpret_cast<double2*>(gy)[i] = make_double2(sa * y.x, sb * y.y);
            reinterpret_cast<double2*>(gz)[i] = make_double2(sa * z.x, sb * z.y);
        }
    }
    if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {          // odd grids (cuFFT route): the last point
        const size_t i = n - 1;
        double fa, ra, sa;
        pbe_point_fast(den[i], gx[i] * gx[i] + gy[i] * gy[i] + gz[i] * gz[i], (which & 1) != 0, (which & 2) != 0, fa, ra, sa);
        acc[0] += fa;
        if (v) {
            v[i] = (accumulate ? v[i] : 0.0) + ra;
            sa *= 2.0;
            gx[i] *= sa; gy[i] *= sa; gz[i] *= sa;
        }
    }
    block_reduce_store<1>(acc, partials);
}

template <bool ACC>
struct PostPbeA {                      // (kept for comparison, option pbe_fast = 2) gradient -> energy density, f_n -> v, staged w for the forward part
    static constexpr bool kDen = true, kVin = ACC;
    static constexpr int NST = 3;
    double* v_out;                     // null: energy only
    int which;
    __device__ void apply(size_t g, double2 n, double2 v, const double* u0, const double* u1, double* acc, double* sta, double* stb) const {
        const PbeOut a = pbe_point_w(n.x, u0[0], u0[1], u0[2], which), b = pbe_point_w(n.y, u1[0], u1[1], u1[2], which);
        acc[0] += a.f + b.f;
        sta[0] = a.wx; sta[1] = a.wy; sta[2] = a.wz;
        stb[0] = b.wx; stb[1] = b.wy; stb[2] = b.wz;
        if (v_out) *reinterpret_cast<double2*>(v_out + g) = make_double2((ACC ? v.x : 0.0) + a.f_rho, (ACC ? v.y : 0.0) + b.f_rho);
    }
    static constexpr int NACC = 0;
    typedef int Ctx;
    __device__ Ctx begin() const { return 0; }
    template <int F>
    __device__ void fold(const Ctx&, double, double, double*) const {}
    __device__ void finish(const Ctx&, size_t, double2, const double*, const double*, double, double, double*, double*, double*) const {}
};
struct GenPbeW {                       // forward part: the staged w_x, w_y, w_z
    static constexpr int NST = 3, NIN = 0;
    __device__ void stage(const double2*, double*, double*) const {}
    template <int F>
    __device__ double field(const double* s) const { return s[F]; }
};
struct PostPbeDiv {                    // v -= div w
    static constexpr bool kDen = false, kVin = true;
    static constexpr int NST = 0;
    double* v_out;
    __device__ void apply(size_t g, double2, double2 v, const double* u0, const double* u1, double*, double*, double*) const {
        *reinterpret_cast<double2*>(v_out + g) = make_double2(v.x - u0[0], v.y - u1[0]);
    }
    static constexpr int NACC = 0;
    typedef int Ctx;
    __device__ Ctx begin() const { return 0; }
    template <int F>
    __device__ void fold(const Ctx&, double, double, double*) const {}
    __device__ void finish(const Ctx&, size_t, double2, const double*, const double*, double, double, double*, double*, double*) const {}
};

// the point kernel on its own (the cuFFT route of pad_eval_pbe uses it too; the log / exp tables live in this translation unit):
// energy density partial sums -> plan partials (returns the grid for the finalize), v (+)= f_n, (gx, gy, gz) <- w
int pad_pbe_pointwise(pad_plan* p, cudaStream_t s, const double* den, double* gx, double* gy, double* gz, double* v, int which,
                      int accumulate, int* grid_out) {
    PAD_TRY(ensure_twiddles(p->device));
    const int grid = pad_grid_for(p->N / 2 > 0 ? p->N / 2 : 1);
    pbe_point_kernel<<<grid, PAD_THREADS, 0, s>>>(den, gx, gy, gz, v, p->N, which, accumulate, p->partials);
    ++g_pad_launches;
    PAD_CUDA(cudaGetLastError());
    if (grid_out) *grid_out = grid;
    return PAD_OK;
}

int pad_pbe_fast_supported(const pad_plan* p) { return !p->dist && fast_shape(p) && g_pad_own_xy && own_xy_shape(p) ? 1 : 0; }

int pad_pbe_fast(pad_plan* p, const double* den, int which, double* E_out, double* v_out, int accumulate, cudaStream_t s) {
    PAD_TRY(ensure_twiddles(p->device));
    cd* B[3];
    for (int i = 0; i < 3; ++i) PAD_TRY(get_zbuf(p, i, &B[i]));
    const double inv_n = p->geom.inv_n;
    pad_stage_begin(s);
    ZDISPATCH(p, PAD_TRY((launch_zfwd<M, TPL, 1>(p, s, GenCopy{}, den, nullptr, B[0], nullptr, nullptr, nullptr))));
    pad_stage_mark("PBE: z-r2c", s);
    PAD_TRY(launch_spass(p, s, 1, -1, B, 1));
    pad_stage_mark("PBE: y-fwd", s);
    PAD_TRY((launch_xmix3_io<1, 3>(p, s, B, MixGrad{inv_n})));
    pad_stage_mark("PBE: x-fwd * (i k) * x-inv (1 -> 3)", s);
    PAD_TRY(launch_spass(p, s, 1, +1, B, 3));
    pad_stage_mark("PBE: y-inv (3)", s);
    int grid = 1;
    if (g_pad_pbe_fast != 2) {
        double* G[3];
        for (int i = 0; i < 3; ++i) PAD_TRY(pad_get_rbuf(p, i, &G[i]));
        ZDISPATCH(p, PAD_TRY((launch_zinv<M, TPL, 3, 0>(p, s, PostStore3{G[0], G[1], G[2]}, B[0], B[1], B[2], nullptr, nullptr, nullptr, nullptr))));
        pad_stage_mark("PBE: z-c2r (3)", s);
        grid = pad_grid_for(p->N / 2);
        pbe_point_kernel<<<grid, PAD_THREADS, 0, s>>>(den, G[0], G[1], G[2], v_out, p->N, which, accumulate, p->partials);
        ++g_pad_launches;
        PAD_CUDA(cudaGetLastError());
        pad_stage_mark("PBE: energy density, f_n, w (pointwise)", s);
        if (E_out) {
            FinalizeArgs a = wgc_energy_args(p, grid, 1, accumulate, E_out);
            a.coef[0] = p->dV;
            pad_launch_finalize(p, a, s);
        }
        if (!v_out) return PAD_OK;
        ZDISPATCH(p, PAD_TRY((launch_zfwd<M, TPL, 3>(p, s, GenCopy3{}, G[0], G[1], B[0], B[1], B[2], nullptr, G[2]))));
        pad_stage_mark("PBE: z-r2c (3)", s);
        PAD_TRY(launch_spass(p, s, 1, -1, B, 3));
        pad_stage_mark("PBE: y-fwd (3)", s);
        PAD_TRY((launch_xmix3_io<3, 1>(p, s, B, MixDiv{inv_n})));
        pad_stage_mark("PBE: x-fwd * (i k .) * x-inv (3 -> 1)", s);
        PAD_TRY(launch_spass(p, s, 1, +1, B, 1));
        pad_stage_mark("PBE: y-inv", s);
        ZDISPATCH(p, PAD_TRY((launch_zinv<M, TPL, 1, 0>(p, s, PostPbeDiv{v_out}, B[0], nullptr, nullptr, nullptr, nullptr, v_out, nullptr))));
        pad_stage_mark("PBE: z-c2r + v -= div w", s);
        return PAD_OK;
    }
    if (!v_out) {
        PostPbeA<false> post{nullptr, which};
        ZDISPATCH(p, PAD_TRY((launch_zinv<M, TPL, 3, 1>(p, s, post, B[0], B[1], B[2], nullptr, den, nullptr, &grid))));
    } else if (accumulate) {
        PostPbeA<true> post{v_out, which};
        ZDISPATCH(p, PAD_TRY((launch_zinv<M, TPL, 3, 1, PostPbeA<true>, 3, GenPbeW>(p, s, post, B[0], B[1], B[2], nullptr, den, v_out, &grid, GenPbeW{}))));
    } else {
        PostPbeA<false> post{v_out, which};
        ZDISPATCH(p, PAD_TRY((launch_zinv<M, TPL, 3, 1, PostPbeA<false>, 3, GenPbeW>(p, s, post, B[0], B[1], B[2], nullptr, den, nullptr, &grid, GenPbeW{}))));
    }
    pad_stage_mark("PBE: z-c2r (3) + energy density, f_n, w + z-r2c (3)", s);
    if (E_out) {
        FinalizeArgs a = wgc_energy_args(p, grid, 1, accumulate, E_out);
        a.coef[0] = p->dV;
        pad_launch_finalize(p, a, s);
    }
    if (!v_out) return PAD_OK;
    PAD_TRY(launch_spass(p, s, 1, -1, B, 3));
    pad_stage_mark("PBE: y-fwd (3)", s);
    PAD_TRY((launch_xmix3_io<3, 1>(p, s, B, MixDiv{inv_n})));
    pad_stage_mark("PBE: x-fwd * (i k .) * x-inv (3 -> 1)", s);
    PAD_TRY(launch_spass(p, s, 1, +1, B, 1));
    pad_stage_mark("PBE: y-inv", s);
    ZDISPATCH(p, PAD_TRY((launch_zinv<M, TPL, 1, 0>(p, s, PostPbeDiv{v_out}, B[0], nullptr, nullptr, nullptr, nullptr, v_out, nullptr))));
    pad_stage_mark("PBE: z-c2r + v -= div w", s);
    return PAD_OK;
}

// =================================================================================================
//  Semilocal kinetic functionals (LuoKarasievTrickey, PauliGaussian: xc.cuh, semilocal_kinetic_point), optionally with PBE
//  in the same point kernel (pad_eval_total: one gradient / divergence round trip carries both energy densities and both w)
//     LKT: the PBE passes.  PG (depends on L = lap n): the x passes carry a fourth field,
//       [x . (i k_c / N, -k^2 / N) . x^-1: one in, four out]  ...  [x . (i k . w + k^2 e_L) / N . x^-1: four in, one out]
//     so that v = e_n - div(2 e_sigma grad n) + lap(e_L) comes out of the same single-field tail.
//  -k^2 is the Hermitian part (sym_even) on the special points, as in pad_laplacian.
// =================================================================================================
struct MixGradLapCoef {
    double kx, ky, kz, k2;
};
struct MixGradLap {                    // q[0] = F  ->  q[c] = i k_c F / N (c < 3), q[3] = -k^2 F / N
    static constexpr int kRing = 1;
    double inv_n;
    typedef MixGradLapCoef Coef;
    typedef MixGrad::Line Line;
    __device__ __forceinline__ Line line(const KGeom& g, int ky, int z) const { return Line{&g, ky, z}; }
    __device__ __forceinline__ Coef fetch(const Line& l, int kx, size_t, bool live) const {
        Coef c{0.0, 0.0, 0.0, 0.0};
        if (live) {
            const KPoint p = make_kpoint_at(*l.g, kx, l.ky, l.z);
            sym_kvec(p, c.kx, c.ky, c.kz);
            c.kx *= inv_n; c.ky *= inv_n; c.kz *= inv_n;
            c.k2 = inv_n * sym_even(p, [](double x, double y, double z) { return x * x + y * y + z * z; });
        }
        return c;
    }
    __device__ __forceinline__ void apply(const Coef& k, cd* q) const {
        const cd a = q[0];
        q[0] = cd{-a.y * k.kx, a.x * k.kx};
        q[1] = cd{-a.y * k.ky, a.x * k.ky};
        q[2] = cd{-a.y * k.kz, a.x * k.kz};
        q[3] = cd{-a.x * k.k2, -a.y * k.k2};
    }
};
struct MixDivLap {                     // q[0] = (i k . (q0, q1, q2) + k^2 q3) / N  (the tail subtracts it from v)
    static constexpr int kRing = 1;
    double inv_n;
    typedef MixGradLapCoef Coef;
    typedef MixGrad::Line Line;
    __device__ __forceinline__ Line line(const KGeom& g, int ky, int z) const { return Line{&g, ky, z}; }
    __device__ __forceinline__ Coef fetch(const Line& l, int kx, size_t pidx, bool live) const { return MixGradLap{inv_n}.fetch(l, kx, pidx, live); }
    __device__ __forceinline__ void apply(const Coef& k, cd* q) const {
        const double re = k.kx * q[0].x + k.ky * q[1].x + k.kz * q[2].x, im = k.kx * q[0].y + k.ky * q[1].y + k.kz * q[2].y;
        q[0] = cd{-im + k.k2 * q[3].x, re + k.k2 * q[3].y};
    }
};
struct PostStore4 {                    // plain c2r of four real fields
    static constexpr bool kDen = false, kVin = false;
    static constexpr int NST = 0;
    double *o0, *o1, *o2, *o3;
    __device__ void apply(size_t g, double2, double2, const double* u0, const double* u1, double*, double*, double*) const {
        *reinterpret_cast<double2*>(o0 + g) = make_double2(u0[0], u1[0]);
        *reinterpret_cast<double2*>(o1 + g) = make_double2(u0[1], u1[1]);
        *reinterpret_cast<double2*>(o2 + g) = make_double2(u0[2], u1[2]);
        *reinterpret_cast<double2*>(o3 + g) = make_double2(u0[3], u1[3]);
    }
    static constexpr int NACC = 0;
    typedef int Ctx;
    __device__ Ctx begin() const { return 0; }
    template <int F>
    __device__ void fold(const Ctx&, double, double, double*) const {}
    __device__ void finish(const Ctx&, size_t, double2, const double*, const double*, double, double, double*, double*, double*) const {}
};
struct GenCopy4 {                      // plain r2c of four real fields
    static constexpr int NST = 4, NIN = 4;
    __device__ void stage(const double2* in, double* a, double* b) const {
        a[0] = in[0].x; a[1] = in[1].x; a[2] = in[2].x; a[3] = in[3].x;
        b[0] = in[0].y; b[1] = in[1].y; b[2] = in[2].y; b[3] = in[3].y;
    }
    template <int F>
    __device__ double field(const double* s) const { return s[F]; }
};

// semilocal_kinetic_point (xc.cuh) with the table log / exp of fastmath.cuh: one log of n and two exps give n^(2/3) and
// n^(-8/3); LKT adds exp(-a s) (1/cosh and tanh from it: 2 e^-x / (1 + e^-2x) cannot overflow), PG exp(-mu p).  Arguments
// outside the fast range take the library version.
__device__ __forceinline__ void semilocal_kinetic_point_fast(double n, double sig, double lap, int variant, double p0, double p1,
                                                             double& e, double& e_n, double& e_sig, double& e_lap) {
    if (!(n > 1e-20 && n < 1e20 && sig < 1e40 && fabs(lap) < 1e40)) {
        semilocal_kinetic_point(n, sig, lap, variant, p0, p1, e, e_n, e_sig, e_lap);
        return;
    }
    const double l = fm_log(n);
    const double n23 = fm_exp((2.0 / 3.0) * l), im83 = fm_exp((-8.0 / 3.0) * l);      // n^(2/3), n^(-8/3)
    const double p = kSlC * sig * im83;
    double F, Fp, qFq = 0.0;
    e_lap = 0.0;
    if (variant == 0) {
        const double x = p0 * sqrt(p);
        const double em = fm_exp(-fmin(x, 300.0)), em2 = em * em;                       // e^-x (e^-300: sech below 1e-130)
        const double ir = fm_recip(1.0 + em2);
        const double sech = 2.0 * em * ir;
        const double tox = x < 0.0625 ? tanh_over_x_series(x) : (1.0 - em2) * ir * fm_recip(x);
        F = sech + (5.0 / 3.0) * p;
        Fp = 5.0 / 3.0 - 0.5 * p0 * p0 * sech * tox;
    } else {
        const double q = kSlC * lap * (n * im83), g = fm_exp(-fmin(p0 * p, 700.0));
        F = (5.0 / 3.0) * p + g + p1 * q * q;
        Fp = 5.0 / 3.0 - p0 * g;
        qFq = 2.0 * p1 * q * q;
        e_lap = kCTF * kSlC * 2.0 * p1 * q;
    }
    e = kCTF * n * n23 * F;
    e_n = kCTF * n23 * ((5.0 / 3.0) * F - (8.0 / 3.0) * p * Fp - (5.0 / 3.0) * qFq);
    e_sig = kCTF * kSlC * Fp * fm_recip(n);
}

// n, grad n (, lap n) -> energy density (one block-reduced sum), v (+)= e_n, grad n <- w = 2 e_sigma grad n (, lap n <- e_L);
// with P.pbe the PBE terms are added to e, e_n, e_sigma at the same point.  Plain one-point-per-thread loads: any alignment,
// any N (the cuFFT route takes odd grids and caller-owned pointers)
template <bool LAP>
__global__ void __launch_bounds__(PAD_THREADS) semilocal_point_kernel(const double* __restrict__ den, double* __restrict__ gx,
                                                                     double* __restrict__ gy, double* __restrict__ gz,
                                                                     double* __restrict__ lap, double* __restrict__ v, size_t n,
                                                                     pad_semilocal_args P, int accumulate,
                                                                     double* __restrict__ partials) {
    fm_load_tables();
    double acc[1] = {0.0};
    const size_t stride = (size_t)gridDim.x * PAD_THREADS;
    for (size_t i = (size_t)blockIdx.x * PAD_THREADS + threadIdx.x; i < n; i += stride) {
        const double d = den[i], x = gx[i], y = gy[i], z = gz[i];
        const double sig = x * x + y * y + z * z;
        double e, e_n, e_s, e_l;
        semilocal_kinetic_point_fast(d, sig, LAP ? lap[i] : 0.0, P.variant, P.p0, P.p1, e, e_n, e_s, e_l);
        if (P.pbe) {
            double f, f_n, f_s;
            pbe_point_fast(d, sig, (P.pbe & 1) != 0, (P.pbe & 2) != 0, f, f_n, f_s);
            e += f; e_n += f_n; e_s += f_s;
        }
        acc[0] += e;
        if (v) {
            v[i] = (accumulate ? v[i] : 0.0) + e_n;
            const double w = 2.0 * e_s;
            gx[i] = w * x; gy[i] = w * y; gz[i] = w * z;
            if (LAP) lap[i] = e_l;
        }
    }
    block_reduce_store<1>(acc, partials);
}

int pad_semilocal_pointwise(pad_plan* p, cudaStream_t s, const double* den, double* gx, double* gy, double* gz, double* lap, double* v,
                            const pad_semilocal_args& P, int accumulate, int* grid_out) {
    PAD_TRY(ensure_twiddles(p->device));
    const int grid = pad_grid_for(p->N);
    if (lap) semilocal_point_kernel<true><<<grid, PAD_THREADS, 0, s>>>(den, gx, gy, gz, lap, v, p->N, P, accumulate, p->partials);
    else semilocal_point_kernel<false><<<grid, PAD_THREADS, 0, s>>>(den, gx, gy, gz, nullptr, v, p->N, P, accumulate, p->partials);
    ++g_pad_launches;
    PAD_CUDA(cudaGetLastError());
    if (grid_out) *grid_out = grid;
    return PAD_OK;
}

int pad_semilocal_fast(pad_plan* p, const double* den, const pad_semilocal_args& P, double* E_out, double* v_out, int accumulate,
                       cudaStream_t s) {
    PAD_TRY(ensure_twiddles(p->device));
    const bool lap = P.variant == PAD_SEMILOCAL_PG;
    const int nf = lap ? 4 : 3;
    cd* B[4];
    double* G[4];
    for (int i = 0; i < nf; ++i) { PAD_TRY(get_zbuf(p, i, &B[i])); PAD_TRY(pad_get_rbuf(p, i, &G[i])); }
    const double inv_n = p->geom.inv_n;
    pad_stage_begin(s);
    ZDISPATCH(p, PAD_TRY((launch_zfwd<M, TPL, 1>(p, s, GenCopy{}, den, nullptr, B[0], nullptr, nullptr, nullptr))));
    pad_stage_mark("semilocal: z-r2c", s);
    PAD_TRY(launch_spass(p, s, 1, -1, B, 1));
    pad_stage_mark("semilocal: y-fwd", s);
    if (lap) PAD_TRY((launch_xmix3_io<1, 4, MixGradLap, 4>(p, s, B, MixGradLap{inv_n})));
    else PAD_TRY((launch_xmix3_io<1, 3>(p, s, B, MixGrad{inv_n})));
    pad_stage_mark("semilocal: x-fwd * (i k [, -k^2]) * x-inv (1 -> 3 | 4)", s);
    PAD_TRY(launch_spass(p, s, 1, +1, B, nf));
    pad_stage_mark("semilocal: y-inv (3 | 4)", s);
    if (lap) ZDISPATCH(p, PAD_TRY((launch_zinv<M, TPL, 4, 0>(p, s, PostStore4{G[0], G[1], G[2], G[3]}, B[0], B[1], B[2], B[3], nullptr, nullptr, nullptr))));
    else ZDISPATCH(p, PAD_TRY((launch_zinv<M, TPL, 3, 0>(p, s, PostStore3{G[0], G[1], G[2]}, B[0], B[1], B[2], nullptr, nullptr, nullptr, nullptr))));
    pad_stage_mark("semilocal: z-c2r (3 | 4)", s);
    int grid = 1;
    PAD_TRY(pad_semilocal_pointwise(p, s, den, G[0], G[1], G[2], lap ? G[3] : nullptr, v_out, P, accumulate, &grid));
    pad_stage_mark("semilocal: energy density, e_n, w [, e_L] (pointwise)", s);
    if (E_out) {
        FinalizeArgs a = wgc_energy_args(p, grid, 1, accumulate, E_out);
        a.coef[0] = p->dV;
        pad_launch_finalize(p, a, s);
    }
    if (!v_out) return PAD_OK;
    if (lap) ZDISPATCH(p, PAD_TRY((launch_zfwd<M, TPL, 4>(p, s, GenCopy4{}, G[0], G[1], B[0], B[1], B[2], B[3], G[2], G[3]))));
    else ZDISPATCH(p, PAD_TRY((launch_zfwd<M, TPL, 3>(p, s, GenCopy3{}, G[0], G[1], B[0], B[1], B[2], nullptr, G[2]))));
    pad_stage_mark("semilocal: z-r2c (3 | 4)", s);
    PAD_TRY(launch_spass(p, s, 1, -1, B, nf));
    pad_stage_mark("semilocal: y-fwd (3 | 4)", s);
    if (lap) PAD_TRY((launch_xmix3_io<4, 1, MixDivLap, 4>(p, s, B, MixDivLap{inv_n})));
    else PAD_TRY((launch_xmix3_io<3, 1>(p, s, B, MixDiv{inv_n})));
    pad_stage_mark("semilocal: x-fwd * (i k . [, k^2]) * x-inv (3 | 4 -> 1)", s);
    PAD_TRY(launch_spass(p, s, 1, +1, B, 1));
    pad_stage_mark("semilocal: y-inv", s);
    ZDISPATCH(p, PAD_TRY((launch_zinv<M, TPL, 1, 0>(p, s, PostPbeDiv{v_out}, B[0], nullptr, nullptr, nullptr, nullptr, v_out, nullptr))));
    pad_stage_mark("semilocal: z-c2r + v -= div w [- lap e_L]", s);
    return PAD_OK;
}

// Hartree term alone (functionals.py:49-72) on the fused passes: [z r2c of n] -> y -> [x . 4 pi / (k^2 N) . x^-1] -> y^-1 ->
// [z c2r + sum n v_H + potential]; v_out must be given (the energy-only call keeps the cuFFT route).  accumulate: v_out += v_H.
int pad_hartree_fast_supported(const pad_plan* p) { return fast_shape(p) && g_pad_own_xy && own_xy_shape(p) ? 1 : 0; }

int pad_hartree_fast(pad_plan* p, const double* den, double* E_out, double* v_out, int accumulate, cudaStream_t s) {
    PAD_TRY(ensure_twiddles(p->device));
    cd* B[1];
    PAD_TRY(get_zbuf(p, 0, &B[0]));
    if (!accumulate) PAD_CUDA(cudaMemsetAsync(v_out, 0, sizeof(double) * p->N, s));
    pad_stage_begin(s);
    ZDISPATCH(p, PAD_TRY((launch_zfwd<M, TPL, 1>(p, s, GenCopy{}, den, nullptr, B[0], nullptr, nullptr, nullptr))));
    pad_stage_mark("Hartree: z-r2c", s);
    PAD_TRY(launch_spass(p, s, 1, -1, B, 1));
    pad_stage_mark("Hartree: y-fwd", s);
    PAD_TRY((launch_xmix<1>(p, s, B, MixCoulomb{p->geom.inv_n})));
    pad_stage_mark("Hartree: x-fwd * (4 pi / k^2) * x-inv", s);
    PAD_TRY(launch_spass(p, s, 1, +1, B, 1));
    pad_stage_mark("Hartree: y-inv", s);
    int grid = 1;
    PostHartreeLocal tail{v_out, nullptr, 0};
    ZDISPATCH(p, PAD_TRY((launch_zinv<M, TPL, 1, 2>(p, s, tail, B[0], nullptr, nullptr, nullptr, den, v_out, &grid))));
    pad_stage_mark("Hartree: z-c2r + energy + potential", s);
    if (E_out) {
        FinalizeArgs h = wgc_energy_args(p, grid, 2, accumulate, E_out);
        h.coef[0] = 0.5 * p->dV; h.coef[1] = 0.0;
        pad_launch_finalize(p, h, s);
    }
    return PAD_OK;
}

int pad_wt_fast_supported(const pad_plan* p) { return fast_shape(p) && g_pad_own_xy && own_xy_shape(p) ? 1 : 0; }

int pad_wt_fast(pad_plan* p, const double* den, double alpha, double beta, double* E_out, double* v_out, int accumulate,
                cudaStream_t s) {
    return alpha != beta ? wt_fast_impl<true>(p, den, alpha, beta, E_out, v_out, accumulate, s)
                         : wt_fast_impl<false>(p, den, alpha, beta, E_out, v_out, accumulate, s);
}

// fastmath.cuh against the library functions: out[0..n) = fm_exp(e * fm_log(x)), out[n..2n) = sqrt via fm_rsqrt,
// out[2n..3n) = fm_rsqrt(x)^2 (used as 1/x); ref[...] the same from exp/log, sqrt and division
__global__ void fastmath_probe_kernel(const double* x, size_t n, double e, double* out, double* ref) {
    fm_load_tables();
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const double v = x[i];
        const double y = fm_rsqrt(v);
        out[i] = fm_exp(e * fm_log(v));
        out[n + i] = fm_sqrt_from_rsqrt(v, y);
        out[2 * n + i] = y * y;
        ref[i] = pow(v, e);
        ref[n + i] = sqrt(v);
        ref[2 * n + i] = 1.0 / v;
    }
}
extern "C" int pad_dbg_fastmath(const double* x, size_t n, double e, double* out3n, double* ref3n, void* stream) {
    int dev = 0;
    PAD_CUDA(cudaGetDevice(&dev));
    PAD_TRY(ensure_twiddles(dev));
    fastmath_probe_kernel<<<592, 256, 0, (cudaStream_t)stream>>>(x, n, e, out3n, ref3n);
    PAD_CUDA(cudaGetLastError());
    return PAD_OK;
}

// in-place complex FFT of one padded half-spectrum along axis 0 or 1 (own strided pass); unnormalised
extern "C" int pad_fft_axis_fast(pad_plan* p, double* cplx_padded, int axis, int dir, void* stream) {
    if (!p || !cplx_padded || (axis != 0 && axis != 1)) { pad_set_error("pad_fft_axis_fast: bad argument"); return PAD_ERR_ARG; }
    if (!spass_len_ok(axis == 0 ? p->n0 : p->n1)) {
        pad_set_error("pad_fft_axis_fast: axis length %d not supported (64, 128, 256, 512)", axis == 0 ? p->n0 : p->n1);
        return PAD_ERR_ARG;
    }
    PAD_CUDA(cudaSetDevice(p->device));
    PAD_TRY(ensure_twiddles(p->device));
    cd* one[1] = {reinterpret_cast<cd*>(cplx_padded)};
    return launch_spass(p, (cudaStream_t)stream, axis, dir, one, 1);
}
