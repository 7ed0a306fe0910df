// assemble.cuh -- on-device operator assembly (HBM-bound kernels).
//   minmax_kernel        : min/max of the sound-speed map            (solve_helmholtz.py:62 arguments)
//   stencil_params_kernel: optimal 9-point weights (b,d,e)           (solve_helmholtz.py:104-154)
//   assemble_kernel      : nine coefficient planes of the mixed-grid (solve_helmholtz.py:158-260)
//                          PML Helmholtz operator, one thread per grid node, coalesced plane stores.
//                          LOSSY = true: complex slowness sigma = s - i kappa, k^2 = w^2 sigma^2 (DESIGN.md section 7d).
// Algorithmic bytes per node and frequency: read vel (sizeof R) + write 9 complex coefficients
// (9 * 2 * sizeof R) = 76 B (c64) / 152 B (c128).
#pragma once
#include "common.cuh"

namespace ust {

template <typename R>
__global__ void __launch_bounds__(1024) minmax_kernel(const R* __restrict__ vel, long long n, double* __restrict__ out2) {
    __shared__ double smin[32], smax[32];
    double lo = 1e300, hi = -1e300;
    for (long long i = threadIdx.x; i < n; i += blockDim.x) {
        double v = (double)vel[i];
        lo = fmin(lo, v);
        hi = fmax(hi, v);
    }
    for (int o = 16; o > 0; o >>= 1) {
        lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) { smin[w] = lo; smax[w] = hi; }
    __syncthreads();
    if (w == 0) {
        lo = (l < (blockDim.x >> 5)) ? smin[l] : 1e300;
        hi = (l < (blockDim.x >> 5)) ? smax[l] : -1e300;
        for (int o = 16; o > 0; o >>= 1) {
            lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
            hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        }
        if (l == 0) { out2[0] = lo; out2[1] = hi; }
    }
}

// One block per frequency, 1024 threads (1000 active = 100 angles x 10 wavelengths), float64 throughout.
__global__ void __launch_bounds__(1024) stencil_params_kernel(const double* __restrict__ vminmax, const double* __restrict__ freqs,
                                                               double h, double g, double* __restrict__ bde) {
    const int fi = blockIdx.x;
    const double f = freqs[fi];
    const double vmin = vminmax[0], vmax = vminmax[1];
    const int l = 100, r = 10;
    const double PI = 3.14159265358979323846;
    double s[5] = {0, 0, 0, 0, 0};  // a11 a12 a22 r1 r2
    int t = threadIdx.x;
    if (t < l * r) {
        int ni = t / l;  // 0..9   (n-1)
        int mi = t % l;  // 0..99  (m-1)
        double Gmin = vmin / (f * h), Gmax = vmax / (f * h);
        double theta = mi * PI / (4.0 * (l - 1));
        double G = 1.0 / (1.0 / Gmax + (double)ni / (r - 1) * (1.0 / Gmin - 1.0 / Gmax));
        double P = cos(g * 2.0 * PI * cos(theta) / G);
        double Q = cos(2.0 * PI * sin(theta) / G);
        double ig2 = 1.0 / (g * g);
        double S1 = (1.0 + ig2) * G * G * (1.0 - P - Q + P * Q);
        double S2 = PI * PI * (2.0 - P - Q);
        double S3 = 2.0 * PI * PI * (1.0 - P * Q);
        double S4 = 2.0 * PI * PI + G * G * ((1.0 + ig2) * P * Q - P - Q * ig2);
        double b = 5.0 / 6.0;
        double y = S4 - b * S1;
        s[0] = S2 * S2; s[1] = S2 * S3; s[2] = S3 * S3; s[3] = S2 * y; s[4] = S3 * y;
    }
    __shared__ double red[5][32];
    int w = threadIdx.x >> 5, ln = threadIdx.x & 31;
    for (int q = 0; q < 5; ++q) {
        double v = s[q];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (ln == 0) red[q][w] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a[5];
        for (int q = 0; q < 5; ++q) {
            double v = 0;
            for (int i = 0; i < 32; ++i) v += red[q][i];
            a[q] = v;
        }
        double det = a[0] * a[2] - a[1] * a[1];
        bde[3 * fi + 0] = 5.0 / 6.0;
        bde[3 * fi + 1] = (a[3] * a[2] - a[1] * a[4]) / det;
        bde[3 * fi + 2] = (a[0] * a[4] - a[1] * a[3]) / det;
    }
}

struct AsmArgs {
    Geom g;
    double h, gr;  // grid step, anisotropy ratio dy/dx
    int stencil;   // 0 python (clamped out-of-bounds gathers), 1 matlab
    int nfreq;
    int exp;       // timing experiment (UST_EXP & 8): store constants only -- what the store pattern alone costs
};

// 1 / v^2 per node in float64, once per model (every frequency and every one of a node's nine neighbours reuses it: the
// nine FP64 divisions k = w / v per node and frequency were what made the assembly FP64-pipe bound instead of HBM bound)
template <typename R>
__global__ void __launch_bounds__(256) inv_v2_kernel(const R* __restrict__ vel, double* __restrict__ out, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { const double v = (double)vel[i]; out[i] = 1.0 / (v * v); }
}

// Lossy models: sigma^2 = (s - i kappa)^2 per node in float64, interleaved (re, im).  Re is formed as 1/v^2 - kappa^2 with 1/v^2
// exactly as inv_v2_kernel forms it, so that kappa = 0 gives the lossless operator's doubles; Im = -2 kappa / v.
template <typename R>
__global__ void __launch_bounds__(256) sig2_kernel(const R* __restrict__ vel, const R* __restrict__ kappa, double2* __restrict__ out, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const double v = (double)vel[i], k = (double)kappa[i];
        out[i] = make_double2(1.0 / (v * v) - k * k, -2.0 * k / v);
    }
}

constexpr int ASM_MAXF = 32;  // frequencies per assemble_kernel launch (the host loops over chunks)

// General (absorbing-layer) node: complex FP64 products.  Kept out of line: it needs ~100 registers, and inlined it made EVERY
// thread of assemble_kernel pay for local-memory spills although ~90 % of the nodes of a benchmark grid take the real-arithmetic
// path.  fc = the per-frequency constants staged by the kernel ([nfreq][12] doubles in shared memory).  LOSSY: `inv_v2` holds the
// complex sigma^2 (sig2_kernel, double2 per node) instead of the real 1/v^2.
template <typename R, bool LOSSY>
__device__ __noinline__ void assemble_pml_node(const AsmArgs& a, int x, int y, const double* __restrict__ inv_v2, const cx<R>* __restrict__ exn,
                                               const cx<R>* __restrict__ rexh, const cx<R>* __restrict__ eyn, const cx<R>* __restrict__ reyh,
                                               const double* fcp, cx<R>* __restrict__ out0, int f_lo, int f_hi) {
    typedef cx<double> Z;
    const int Nx = a.g.Nx, Ny = a.g.Ny;
    const size_t pl = (size_t)Nx * Ny;
    const double ih2 = 1.0 / (a.h * a.h), ig2 = 1.0 / (a.gr * a.gr);
    const double (*fc)[12] = reinterpret_cast<const double (*)[12]>(fcp);
    double iv2[3][3];  // 1 / v^2 on the 3x3 neighbourhood (re-read here: passing the caller's copy by reference would pin it in local memory)
    Z s2[3][3];        // LOSSY: sigma^2 on the 3x3 neighbourhood
#pragma unroll
    for (int j = 0; j < 3; ++j)
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            if constexpr (LOSSY) {
                const double2 t = reinterpret_cast<const double2*>(inv_v2)[(size_t)(y - 1 + j) * Nx + (x - 1 + i)];
                s2[j][i] = Z(t.x, t.y);
            } else {
                iv2[j][i] = inv_v2[(size_t)(y - 1 + j) * Nx + (x - 1 + i)];
            }
        }
    // PML factors around the node
    Z ex_[3], ey_[3], rxh[3], ryh[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        int xx = x - 1 + j, yy = y - 1 + j;
        cx<R> t;
        t = exn[xx]; ex_[j] = Z(t.re, t.im);
        t = eyn[yy]; ey_[j] = Z(t.re, t.im);
        int xc = min(xx, Nx - 2), yc = min(yy, Ny - 2);  // JAX clamps out-of-range gathers (SURVEY A.3)
        t = rexh[xc]; rxh[j] = Z(t.re, t.im);
        t = reyh[yc]; ryh[j] = Z(t.re, t.im);
    }
    // A(yy,xx) = ey(node yy) / ex(xx+1/2) ; B(yy,xx) = ex(node xx) / ey(yy+1/2); local index 0,1,2 = -1,0,+1
    auto A = [&](int jy, int ix) { return ey_[jy] * rxh[ix]; };
    auto B = [&](int jy, int ix) { return ex_[ix] * ryh[jy]; };
    const bool py = (a.stencil == 0);
    const Z A_dr = py ? A(0, 2) : A(0, 1);
    const Z B_ul = py ? B(2, 0) : B(1, 0);
    const Z A_ur = py ? A(2, 2) : A(2, 1);
    const Z B_ur = py ? B(2, 2) : B(1, 2);
    for (int fi = f_lo; fi < f_hi; ++fi) {
        const double w2 = fc[fi][0], b = fc[fi][1], beta = fc[fi][2], cc = fc[fi][6], d4 = fc[fi][7], e4 = fc[fi][8];
        const double bih2 = fc[fi][10], betaih2 = fc[fi][11];
        // q = C k^2 on the 3x3 neighbourhood, k^2 = w^2 / v^2 (LOSSY: w^2 sigma^2)
        Z q[3][3];
#pragma unroll
        for (int j = 0; j < 3; ++j)
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                if constexpr (LOSSY) q[j][i] = Z(w2 * s2[j][i].re, w2 * s2[j][i].im) * (ex_[i] * ey_[j]);
                else q[j][i] = (w2 * iv2[j][i]) * (ex_[i] * ey_[j]);
            }
        Z v[9];
        v[PL_C] = cc * q[1][1] - bih2 * (A(1, 1) + A(1, 0) + ig2 * (B(1, 1) + B(0, 1)));
        v[PL_L] = ih2 * (b * A(1, 0) - (beta * ig2) * (B(1, 0) + B(0, 0))) + d4 * q[1][0];
        v[PL_R] = ih2 * (b * A(1, 1) - (beta * ig2) * (B(1, 2) + B(0, 2))) + d4 * q[1][2];
        v[PL_D] = ih2 * ((b * ig2) * B(0, 1) - beta * (A(0, 1) + A(0, 0))) + d4 * q[0][1];
        v[PL_U] = ih2 * ((b * ig2) * B(1, 1) - beta * (A(2, 1) + A(2, 0))) + d4 * q[2][1];
        v[PL_DL] = betaih2 * (A(0, 0) + ig2 * B(0, 0)) + e4 * q[0][0];
        v[PL_DR] = betaih2 * (A_dr + ig2 * B(0, 2)) + e4 * q[0][2];
        v[PL_UL] = betaih2 * (A(2, 0) + ig2 * B_ul) + e4 * q[2][0];
        v[PL_UR] = betaih2 * (A_ur + ig2 * B_ur) + e4 * q[2][2];
        cx<R>* out = out0 + (size_t)fi * 9 * pl;
#pragma unroll
        for (int p = 0; p < 9; ++p) out[p * pl] = cx<R>((R)v[p].re, (R)v[p].im);
    }
}


// PML vectors (complex R): exn[x]=e_x(node x), rexh[x]=1/e_x(x+1/2) (x<=Nx-2), eyn[y], reyh[y].
// One thread per grid node, looping over the launch's frequencies: the stretch factors around the node and the nine 1/v^2
// values are loaded once and serve every frequency; each store instruction of a warp writes 256 contiguous bytes of one plane.
// grid = (ceil(Nx/256), Ny), 256 threads.  LOSSY: `inv_v2` is the double2 sigma^2 of sig2_kernel; the flat nodes keep their real
// stencil part and gain an imaginary mass term (the stretch factors are 1 there, so only k^2 is complex).
template <typename R, bool LOSSY>
__global__ void __launch_bounds__(256, 4) assemble_kernel(AsmArgs a, const double* __restrict__ inv_v2, const cx<R>* __restrict__ exn,
                                                        const cx<R>* __restrict__ rexh, const cx<R>* __restrict__ eyn,
                                                        const cx<R>* __restrict__ reyh, const double* __restrict__ freqs,
                                                        const double* __restrict__ bde, cx<R>* __restrict__ planes) {
    typedef cx<double> Z;
    const int Nx = a.g.Nx, Ny = a.g.Ny;
    // per-frequency constants, computed once per CTA (the launch carries at most ASM_MAXF frequencies): in the frequency loop
    // below they were four dependent global loads + ~12 FP64 operations per node and frequency, and the loads -- evicted from L1
    // by the kernel's own store stream -- were what the warps waited for (ncu: long-scoreboard stall 12 cycles per issue)
    __shared__ double fc[ASM_MAXF][12];
    {
        const double PI = 3.14159265358979323846;
        const double ih2 = 1.0 / (a.h * a.h), ig2 = 1.0 / (a.gr * a.gr);
        for (int fi = threadIdx.x; fi < a.nfreq; fi += blockDim.x) {
            const double w = 2.0 * PI * freqs[fi], w2 = w * w;
            const double b = bde[3 * fi], d = bde[3 * fi + 1], e = bde[3 * fi + 2];
            const double beta = (1.0 - b) * 0.5;
            fc[fi][0] = w2; fc[fi][1] = b; fc[fi][2] = beta;
            fc[fi][3] = ih2 * (b - (beta * ig2) * 2.0);      // edge_x (flat nodes)
            fc[fi][4] = ih2 * ((b * ig2) - beta * 2.0);      // edge_y
            fc[fi][5] = (beta * ih2) * (1.0 + ig2);          // corner
            fc[fi][6] = 1.0 - d - e; fc[fi][7] = d * 0.25; fc[fi][8] = e * 0.25;
            fc[fi][9] = (b * ih2) * (2.0 + ig2 * 2.0);       // centre (flat nodes)
            fc[fi][10] = b * ih2; fc[fi][11] = beta * ih2;
        }
        __syncthreads();
    }
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    // grid rows from both ends inwards: the rows inside the absorbing layer cost ~10 x the arithmetic of an interior row and
    // would otherwise form the tail of the launch (the last CTAs dispatched would be the slowest ones)
    const int y = (blockIdx.y & 1) ? Ny - 1 - (int)(blockIdx.y >> 1) : (int)(blockIdx.y >> 1);
    if (x >= Nx) return;
    const size_t pl = (size_t)Nx * Ny;
    cx<R>* out0 = planes + (size_t)y * Nx + x;
    if (a.exp) {
        for (int fi = 0; fi < a.nfreq; ++fi)
#pragma unroll
            for (int p = 0; p < 9; ++p) out0[((size_t)fi * 9 + p) * pl] = cx<R>((R)fc[fi][p], (R)0);
        return;
    }
    if (x == 0 || y == 0 || x == Nx - 1 || y == Ny - 1) {
        for (int fi = 0; fi < a.nfreq; ++fi)
#pragma unroll
            for (int p = 0; p < 9; ++p) out0[((size_t)fi * 9 + p) * pl] = cxzero<R>();
        return;
    }
    // Outside the absorbing layer every stretch factor is exactly 1: A = B = C = 1, the coefficients are real and the complex
    // FP64 products of the general path (what kept this kernel off the HBM roofline) reduce to nine multiply-adds per
    // frequency.  Same values as the general path (multiplying by an exact 1 is exact), ~90 % of the nodes of a benchmark grid.
    // The test reads the stretch factors without keeping them: held as 24 doubles across the branch they pushed the kernel
    // over its register budget and every thread paid for local-memory spills (ncu: long-scoreboard stalls).
    bool flat = true;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const int xx = x - 1 + j, yy = y - 1 + j;
        const int xc = min(xx, Nx - 2), yc = min(yy, Ny - 2);  // JAX clamps out-of-range gathers (SURVEY A.3)
        const cx<R> t0 = exn[xx], t1 = eyn[yy], t2 = rexh[xc], t3 = reyh[yc];
        flat = flat && t0.re == R(1) && t0.im == R(0) && t1.re == R(1) && t1.im == R(0) &&
               t2.re == R(1) && t2.im == R(0) && t3.re == R(1) && t3.im == R(0);
    }
    if (LOSSY && flat) {
        const double2* s2 = reinterpret_cast<const double2*>(inv_v2);
        double sr[3][3], si[3][3];  // sigma^2 on the 3x3 neighbourhood
#pragma unroll
        for (int j = 0; j < 3; ++j)
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const double2 t = s2[(size_t)(y - 1 + j) * Nx + (x - 1 + i)];
                sr[j][i] = t.x; si[j][i] = t.y;
            }
        for (int fi = 0; fi < a.nfreq; ++fi) {
            const double w2 = fc[fi][0], edge_x = fc[fi][3], edge_y = fc[fi][4], corner = fc[fi][5];
            const double cc = fc[fi][6], d4 = fc[fi][7], e4 = fc[fi][8], ctr = fc[fi][9];
            double r[9], m[9];
            r[PL_C] = cc * (w2 * sr[1][1]) - ctr;          m[PL_C] = cc * (w2 * si[1][1]);
            r[PL_L] = edge_x + d4 * (w2 * sr[1][0]);       m[PL_L] = d4 * (w2 * si[1][0]);
            r[PL_R] = edge_x + d4 * (w2 * sr[1][2]);       m[PL_R] = d4 * (w2 * si[1][2]);
            r[PL_D] = edge_y + d4 * (w2 * sr[0][1]);       m[PL_D] = d4 * (w2 * si[0][1]);
            r[PL_U] = edge_y + d4 * (w2 * sr[2][1]);       m[PL_U] = d4 * (w2 * si[2][1]);
            r[PL_DL] = corner + e4 * (w2 * sr[0][0]);      m[PL_DL] = e4 * (w2 * si[0][0]);
            r[PL_DR] = corner + e4 * (w2 * sr[0][2]);      m[PL_DR] = e4 * (w2 * si[0][2]);
            r[PL_UL] = corner + e4 * (w2 * sr[2][0]);      m[PL_UL] = e4 * (w2 * si[2][0]);
            r[PL_UR] = corner + e4 * (w2 * sr[2][2]);      m[PL_UR] = e4 * (w2 * si[2][2]);
            cx<R>* out = out0 + (size_t)fi * 9 * pl;
#pragma unroll
            for (int p = 0; p < 9; ++p) out[p * pl] = cx<R>((R)r[p], (R)m[p]);
        }
        return;
    }
    if (!LOSSY && flat) {
        double iv2[3][3];  // 1 / v^2 on the 3x3 neighbourhood
#pragma unroll
        for (int j = 0; j < 3; ++j)
#pragma unroll
            for (int i = 0; i < 3; ++i) iv2[j][i] = inv_v2[(size_t)(y - 1 + j) * Nx + (x - 1 + i)];
        for (int fi = 0; fi < a.nfreq; ++fi) {
            const double w2 = fc[fi][0], edge_x = fc[fi][3], edge_y = fc[fi][4], corner = fc[fi][5];
            const double cc = fc[fi][6], d4 = fc[fi][7], e4 = fc[fi][8], ctr = fc[fi][9];
            double r[9];
            r[PL_C] = cc * (w2 * iv2[1][1]) - ctr;
            r[PL_L] = edge_x + d4 * (w2 * iv2[1][0]);
            r[PL_R] = edge_x + d4 * (w2 * iv2[1][2]);
            r[PL_D] = edge_y + d4 * (w2 * iv2[0][1]);
            r[PL_U] = edge_y + d4 * (w2 * iv2[2][1]);
            r[PL_DL] = corner + e4 * (w2 * iv2[0][0]);
            r[PL_DR] = corner + e4 * (w2 * iv2[0][2]);
            r[PL_UL] = corner + e4 * (w2 * iv2[2][0]);
            r[PL_UR] = corner + e4 * (w2 * iv2[2][2]);
            cx<R>* out = out0 + (size_t)fi * 9 * pl;
#pragma unroll
            for (int p = 0; p < 9; ++p) out[p * pl] = cx<R>((R)r[p], (R)0);
        }
        return;
    }
    assemble_pml_node<R, LOSSY>(a, x, y, inv_v2, exn, rexh, eyn, reyh, &fc[0][0], out0, 0, a.nfreq);
}

}  // namespace ust
