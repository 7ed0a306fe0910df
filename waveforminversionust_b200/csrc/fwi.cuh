// fwi.cuh -- fused HBM-bound kernels around the solves (nonlinearcg.py:213-301, fwi_loss_function.py:53-102).
//   onehot_scatter_kernel : one-hot source columns                         (fwi_script.py:72-74)
//   receiver_kernel       : receiver gather, source-strength estimate, residual, loss, adjoint-source
//                           scatter, one CTA per (transmitter, frequency)  (nonlinearcg.py:220-254)
//   gradient_kernel       : grad = sum_f sum_t -Re(conj(VIRT) * ADJ_WV),  VIRT = 2 w^2 s alpha_t u_t
//                           one warp per pixel, warp-shuffle reduction     (nonlinearcg.py:258,264-265)
//                           LOSSY: gradients w.r.t. s and kappa of the complex slowness s - i kappa (DESIGN.md section 7d)
//   pert_rhs_kernel       : RHS of the perturbation solve  -VIRT * sd      (nonlinearcg.py:279-281)
//   gradient_mass_kernel, pert_rhs_mass_kernel : the discrete gradient mode's gradient and perturbation RHS, with the
//                           stencil's 9-point mass weights and the PML factor (DESIGN.md section 7f)
//   linesearch_kernel     : dREC gather and the two step-size scalars      (nonlinearcg.py:22-28,284-298)
//   gn_receiver_kernel    : Gauss-Newton product: J v = perturbation field at the kept receivers, and sum |J v|^2
//   gn_scatter_kernel     : Gauss-Newton product: J v back at the receiver nodes as the adjoint source of J^H (J v)
// Algorithmic bytes of gradient_kernel: 2 complex reads per (pixel, source, frequency) = 16 B (c64).
#pragma once
#include "common.cuh"

namespace ust {

template <typename R>
__global__ void onehot_scatter_kernel(cx<R>* __restrict__ U, size_t stride_f, const int* __restrict__ src_lin, int nt, int nfreq) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nt * nfreq) return;
    int f = i / nt, t = i % nt;
    U[(size_t)f * stride_f + (size_t)src_lin[t] * nt + t] = cxone<R>();
}

__device__ __forceinline__ double warp_sum(double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <int NV>
__device__ __forceinline__ void block_sum(double (&v)[NV], double* sh /* NV*32 */) {
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
#pragma unroll
    for (int q = 0; q < NV; ++q) {
        double s = warp_sum(v[q]);
        if (l == 0) sh[q * 32 + w] = s;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < NV; ++q) {
        double s = (l < nw) ? sh[q * 32 + l] : 0.0;
        v[q] = warp_sum(s);
    }
    __syncthreads();
}

template <typename R>
struct RecvArgs {
    const cx<R>* U;    // [nfreq][N*nt] forward fields (unscaled)
    cx<R>* Lam;        // [nfreq][N*nt] adjoint right-hand side, pre-zeroed
    size_t stride_f;
    const cx<R>* rec;  // [nfreq][nt][nelem] observed data
    const int* rx_lin; // [nelem] row-major node of every element
    const int* mask;   // [nt][nm]
    // [nt][nm] receivers that snap to one node: next kept receiver (mask order) on the same node, nm if none, stored as
    // -1 - next when j is not the first on its node.  The first adds the residuals of all of them, in that order, and stores
    // the sum once, so the adjoint source is the derivative of the loss (which counts every kept receiver) and is
    // deterministic.  Without shared nodes every entry is nm and each receiver stores its own residual.
    const int* rx_next;
    cx<R>* src_est;    // [nfreq][nt]
    double* loss;      // scalar accumulator
    int nt, nm, nelem;
};

template <typename R>
__global__ void __launch_bounds__(256) receiver_kernel(RecvArgs<R> a) {
    __shared__ double sh[4 * 32];
    const int t = blockIdx.x, f = blockIdx.y;
    const cx<R>* Uf = a.U + (size_t)f * a.stride_f;
    const cx<R>* recf = a.rec + ((size_t)f * a.nt + t) * a.nelem;
    const int* mk = a.mask + (size_t)t * a.nm;
    double s[4] = {0, 0, 0, 0};  // Re/Im <sim,rec>, <sim,sim>
    for (int j = threadIdx.x; j < a.nm; j += blockDim.x) {
        int e = mk[j];
        cx<R> sim = Uf[(size_t)a.rx_lin[e] * a.nt + t];
        cx<R> ob = recf[e];
        // vdot conjugates its first argument: conj(sim)*rec
        s[0] += (double)sim.re * ob.re + (double)sim.im * ob.im;
        s[1] += (double)sim.re * ob.im - (double)sim.im * ob.re;
        s[2] += (double)sim.re * sim.re + (double)sim.im * sim.im;
    }
    block_sum<4>(s, sh);
    const double inv = 1.0 / s[2];
    const double ar = s[0] * inv, ai = s[1] * inv;
    if (threadIdx.x == 0) a.src_est[(size_t)f * a.nt + t] = cx<R>((R)ar, (R)ai);
    const cx<R> alpha((R)ar, (R)ai);
    cx<R>* Lf = a.Lam + (size_t)f * a.stride_f;
    const int* nx = a.rx_next + (size_t)t * a.nm;
    double l2[1] = {0};
    for (int j = threadIdx.x; j < a.nm; j += blockDim.x) {
        int e = mk[j];
        size_t o = (size_t)a.rx_lin[e] * a.nt + t;
        cx<R> sim = alpha * Uf[o];
        cx<R> ob = recf[e];
        cx<R> d = sim - ob;
        l2[0] += (double)d.re * d.re + (double)d.im * d.im;
        int k = nx[j];
        if (k < 0) continue;  // a receiver before this one on the same node stores the sum
        for (; k < a.nm; k = -1 - nx[k]) d = d + (sim - recf[mk[k]]);
        Lf[o] = d;  // adjoint source (nonlinearcg.py:248-254; summed over receivers sharing the node)
    }
    block_sum<1>(l2, sh);
    if (threadIdx.x == 0) atomicAdd(a.loss, 0.5 * l2[0]);
}

template <typename R>
struct GradArgs {
    const cx<R>* U;
    const cx<R>* Lam;
    size_t stride_f;
    const cx<R>* src_est;  // [nfreq][nt]
    const double* freqs;   // [nfreq]
    const R* slow;         // [N]
    R* grad;               // [N]
    long long N;
    int nt, nfreq;
    const R* kappa;        // [N] LOSSY only: attenuation slowness
    R* grad_kappa;         // [N] LOSSY only
};

// One warp per pixel.  The nt sources of a (pixel, frequency) are contiguous: complex64 lanes read 16 bytes (two sources)
// per load from u, lambda and the source estimates, form alpha u in FP32 and accumulate Re(conj(alpha u) lambda) in four
// independent FP32 partials that are folded into FP64 once per frequency (a handful of terms per partial, so the FP32
// rounding stays at the level of the complex64 inputs while the dependent chain is four times shorter than one FP64
// accumulator's); complex128 keeps the FP64 path.  Loads of consecutive iterations are independent: the unrolled loop keeps
// several 16-byte requests per lane in flight.
// LOSSY: with z_f = sum_t conj(alpha_t u_t) lambda_t the kernel also accumulates Im z_f, in four more FP32 partials beside the
// four of Re z_f (which keep the lossless kernel's exact structure, so kappa = 0 reproduces its grad_s bit for bit), and writes
//   A = sum_f -2 w^2 Re z_f,  B = sum_f -2 w^2 Im z_f,  grad_s = s A - kappa B,  grad_kappa = -s B - kappa A.
template <typename R, bool LOSSY>
__global__ void __launch_bounds__(256) gradient_kernel(GradArgs<R> a) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const double PI = 3.14159265358979323846;
    const bool vec = sizeof(R) == 4 && (a.nt & 1) == 0 && (a.stride_f & 1) == 0;
    for (long long p = warp; p < a.N; p += nwarps) {
        double tot = 0.0, tot_im = 0.0;
        for (int f = 0; f < a.nfreq; ++f) {
            const cx<R>* u = a.U + (size_t)f * a.stride_f + (size_t)p * a.nt;
            const cx<R>* l = a.Lam + (size_t)f * a.stride_f + (size_t)p * a.nt;
            const cx<R>* al = a.src_est + (size_t)f * a.nt;
            double acc = 0.0, acc_im = 0.0;
            if constexpr (sizeof(R) == 4) {
                if (vec) {
                    const float4* u4 = reinterpret_cast<const float4*>(u);
                    const float4* l4 = reinterpret_cast<const float4*>(l);
                    const float4* a4 = reinterpret_cast<const float4*>(al);
                    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
                    float q0 = 0.f, q1 = 0.f, q2 = 0.f, q3 = 0.f;
                    const int n2 = a.nt >> 1;
#pragma unroll 4
                    for (int t = lane; t < n2; t += 32) {
                        const float4 uu = __ldcs(u4 + t), ll = __ldcs(l4 + t);  // streamed once: do not displace the operand planes in L2
                        const float4 aa = a4[t];
                        const float ar = aa.x * uu.x - aa.y * uu.y, ai = aa.x * uu.y + aa.y * uu.x;  // alpha_t u_t
                        const float br = aa.z * uu.z - aa.w * uu.w, bi = aa.z * uu.w + aa.w * uu.z;
                        s0 = fmaf(ar, ll.x, s0); s1 = fmaf(ai, ll.y, s1);  // Re(conj(alpha u) lambda)
                        s2 = fmaf(br, ll.z, s2); s3 = fmaf(bi, ll.w, s3);
                        if constexpr (LOSSY) {  // Im(conj(alpha u) lambda)
                            q0 = fmaf(ar, ll.y, q0); q1 = fmaf(-ai, ll.x, q1);
                            q2 = fmaf(br, ll.w, q2); q3 = fmaf(-bi, ll.z, q3);
                        }
                    }
                    acc = ((double)s0 + (double)s1) + ((double)s2 + (double)s3);
                    if constexpr (LOSSY) acc_im = ((double)q0 + (double)q1) + ((double)q2 + (double)q3);
                } else {
                    for (int t = lane; t < a.nt; t += 32) {
                        cx<R> uu = al[t] * u[t];
                        cx<R> ll = l[t];
                        acc += (double)uu.re * ll.re + (double)uu.im * ll.im;
                        if constexpr (LOSSY) acc_im += (double)uu.re * ll.im - (double)uu.im * ll.re;
                    }
                }
            } else {
                for (int t = lane; t < a.nt; t += 32) {
                    cx<R> uu = al[t] * u[t];   // alpha_t u_t
                    cx<R> ll = l[t];
                    acc += (double)uu.re * ll.re + (double)uu.im * ll.im;  // Re(conj(uu) * ll)
                    if constexpr (LOSSY) acc_im += (double)uu.re * ll.im - (double)uu.im * ll.re;  // Im(conj(uu) * ll)
                }
            }
            double w = 2.0 * PI * a.freqs[f];
            tot += -2.0 * w * w * acc;
            if constexpr (LOSSY) tot_im += -2.0 * w * w * acc_im;
        }
        tot = warp_sum(tot);
        if constexpr (LOSSY) {
            tot_im = warp_sum(tot_im);
            if (lane == 0) {
                const double s = (double)a.slow[p], k = (double)a.kappa[p];
                a.grad[p] = (R)(tot * s - tot_im * k);
                a.grad_kappa[p] = (R)(-s * tot_im - k * tot);
            }
        } else {
            if (lane == 0) a.grad[p] = (R)(tot * (double)a.slow[p]);
        }
    }
}

// RHS of the perturbation solve: -VIRT*sd = -(2 w^2 s alpha_t u_t) * sd, written into Out (may alias Lam)
template <typename R>
struct PertArgs {
    const cx<R>* U;
    cx<R>* Out;
    size_t stride_f;
    const cx<R>* src_est;
    const double* freqs;
    const R* slow;
    const R* sd;
    long long N;
    int nt, nfreq;
    const R* kappa;     // [N] LOSSY only: attenuation slowness
    const R* sd_kappa;  // [N] LOSSY only: kappa part of the direction
};

// LOSSY (complex slowness sigma = s - i kappa, DESIGN.md section 7e): the RHS is -2 w^2 sigma alpha_t u_t (sd - i sd_kappa), with
// the coefficient c = -2 w^2 (s - i kappa)(sd - i sd_kappa) formed in FP64 and cast once.  Its real part keeps the lossless
// association ((-2 w w) s) sd and only adds terms that are zero at kappa = 0, sd_kappa = 0, so the lossy kernel then writes the
// lossless RHS bit for bit (up to the sign of zero entries).
template <typename R, bool LOSSY>
__global__ void __launch_bounds__(256) pert_rhs_kernel(PertArgs<R> a) {
    const double PI = 3.14159265358979323846;
    const long long total = a.N * a.nt;
    const int f = blockIdx.y;
    const double w = 2.0 * PI * a.freqs[f];
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        long long p = i / a.nt;
        int t = (int)(i % a.nt);
        if constexpr (LOSSY) {
            const double s = (double)a.slow[p], k = (double)a.kappa[p], ds = (double)a.sd[p], dk = (double)a.sd_kappa[p];
            const double m = -2.0 * w * w;
            const R cr = (R)(m * s * ds - m * k * dk);  // Re c = -2 w^2 (s ds - kappa dk)
            const R ci = (R)(-m * (s * dk + k * ds));    // Im c = +2 w^2 (s dk + kappa ds)
            cx<R> v = a.src_est[(size_t)f * a.nt + t] * a.U[(size_t)f * a.stride_f + i];
            a.Out[(size_t)f * a.stride_f + i] = cx<R>(cr * v.re - ci * v.im, cr * v.im + ci * v.re);
        } else {
            R c = (R)(-2.0 * w * w * (double)a.slow[p] * (double)a.sd[p]);
            cx<R> v = a.src_est[(size_t)f * a.nt + t] * a.U[(size_t)f * a.stride_f + i];
            a.Out[(size_t)f * a.stride_f + i] = cx<R>(c * v.re, c * v.im);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Discrete gradient mode (UST_GRAD_DISCRETE, DESIGN.md section 7f): the exact derivative of the discrete forward map at fixed
// stencil weights (b, d, e).  Interior row i of the operator holds the mass term sum_{j in N9(i)} w_ij C_j w^2 sigma_j^2 u_j with
// w_ij = 1-d-e, d/4, e/4 at the centre, edge and corner offsets and C = e_x e_y; ring rows are identity rows.  So
//   (dH u)_i = sum_j w_ij C_j 2 w^2 sigma_j dsigma_j u_j  (interior i, 0 on the ring),   J v = P H^-1(-dH alpha u),
//   z_j = conj(C_j) sum_t conj(alpha_t u_tj) (W lambda_t)_j,  (W lambda)_j = sum_{i in N9(j), i interior} w_ij lambda_i,
// and A, B, grad_s, grad_kappa follow from z as in gradient_kernel.  With w = delta and C = 1 this is the reference's J.
// Both kernels give a warp a segment of MASS_SEG pixels of one grid row and slide a 3x3 window of source-units along it, so a
// lane loads three new columns per pixel instead of nine (4.5 loads per pixel with the segment's halo columns).  Rows y-1 and
// y+1 are loaded again by the warps of the neighbouring rows; whether L2 serves those loads is not established: the measured
// time (DESIGN.md section 7f) is what they would cost from HBM.  A unit is what a lane loads in one step: two complex64
// sources (16 B) or one complex.
constexpr int MASS_SEG = 4;

template <typename R>
struct MassArgs {
    const cx<R>* exn;   // [Nx] e_x at the nodes
    const cx<R>* eyn;   // [Ny] e_y at the nodes
    const double* bde;  // [nfreq][3] stencil weights of the launch's frequencies
    int Nx, Ny;
};

template <typename R, int NS>
struct alignas(NS * sizeof(cx<R>)) Unit { cx<R> c[NS]; };

template <typename U>
__device__ __forceinline__ U ld_stream(const U* p) {  // read-once stream: do not displace the fields the window re-reads
    U r;
    if constexpr (sizeof(U) == 16) { const float4 v = __ldcs(reinterpret_cast<const float4*>(p)); memcpy(&r, &v, 16); }
    else { const float2 v = __ldcs(reinterpret_cast<const float2*>(p)); memcpy(&r, &v, 8); }
    return r;
}

// unit k of the three rows y-1, y, y+1 at column x; zero where the node is not an interior row (keep_ring: where it is off the grid)
template <typename R, int NS>
__device__ __forceinline__ void mass_column(Unit<R, NS> (&col)[3], const cx<R>* F, const MassArgs<R>& m, int nt, int y, int x, int k,
                                            bool keep_ring) {
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const int yy = y - 1 + r;
        const bool ok = keep_ring ? (x >= 0 && x < m.Nx && yy >= 0 && yy < m.Ny) : (x > 0 && x < m.Nx - 1 && yy > 0 && yy < m.Ny - 1);
        if (ok) col[r] = reinterpret_cast<const Unit<R, NS>*>(F + ((size_t)yy * m.Nx + x) * nt)[k];
        else {
#pragma unroll
            for (int s = 0; s < NS; ++s) col[r].c[s] = cxzero<R>();
        }
    }
}

// (W f) at the centre of the window: c0 * centre + d4 * edges + e4 * corners
template <typename R, int NS>
__device__ __forceinline__ cx<R> mass_apply(int s, R c0, R d4, R e4, const Unit<R, NS> (&L)[3], const Unit<R, NS> (&M)[3],
                                            const Unit<R, NS> (&Rt)[3]) {
    const cx<R> edge = (M[0].c[s] + M[2].c[s]) + (L[1].c[s] + Rt[1].c[s]);
    const cx<R> corner = (L[0].c[s] + L[2].c[s]) + (Rt[0].c[s] + Rt[2].c[s]);
    return c0 * M[1].c[s] + d4 * edge + e4 * corner;
}

// Gradient of the discrete mode: one warp per MASS_SEG-pixel row segment, lanes over source-units; the per-pixel partials of
// Re / Im z_f are folded into FP64 once per frequency, as in gradient_kernel.
template <typename R, int NS, bool LOSSY>
__global__ void __launch_bounds__(256) gradient_mass_kernel(GradArgs<R> a, MassArgs<R> m) {
    typedef Unit<R, NS> V;
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const double PI = 3.14159265358979323846;
    const int nseg = (m.Nx + MASS_SEG - 1) / MASS_SEG, nunits = a.nt / NS;
    for (long long item = warp; item < (long long)m.Ny * nseg; item += nwarps) {
        const int y = (int)(item / nseg), x0 = (int)(item % nseg) * MASS_SEG;
        const int np = min(MASS_SEG, m.Nx - x0);
        double tr[MASS_SEG], ti[MASS_SEG];
#pragma unroll
        for (int i = 0; i < MASS_SEG; ++i) tr[i] = ti[i] = 0.0;
        for (int f = 0; f < a.nfreq; ++f) {
            const cx<R>* u = a.U + (size_t)f * a.stride_f;
            const cx<R>* l = a.Lam + (size_t)f * a.stride_f;
            const V* al = reinterpret_cast<const V*>(a.src_est + (size_t)f * a.nt);
            const double d = m.bde[3 * f + 1], e = m.bde[3 * f + 2];
            const R c0 = (R)(1.0 - d - e), d4 = (R)(d * 0.25), e4 = (R)(e * 0.25);
            R zr[MASS_SEG], zi[MASS_SEG];
#pragma unroll
            for (int i = 0; i < MASS_SEG; ++i) zr[i] = zi[i] = R(0);
            for (int k = lane; k < nunits; k += 32) {
                V L[3], M[3], Rt[3];
                mass_column(L, l, m, a.nt, y, x0 - 1, k, false);
                mass_column(M, l, m, a.nt, y, x0, k, false);
                const V aa = al[k];
#pragma unroll
                for (int i = 0; i < MASS_SEG; ++i) {
                    if (i < np) {
                        mass_column(Rt, l, m, a.nt, y, x0 + i + 1, k, false);
                        const V uu = ld_stream(reinterpret_cast<const V*>(u + ((size_t)y * m.Nx + x0 + i) * a.nt) + k);
#pragma unroll
                        for (int s = 0; s < NS; ++s) {
                            const cx<R> au = aa.c[s] * uu.c[s], wl = mass_apply<R, NS>(s, c0, d4, e4, L, M, Rt);
                            zr[i] += au.re * wl.re + au.im * wl.im;  // Re(conj(alpha u) W lambda)
                            zi[i] += au.re * wl.im - au.im * wl.re;  // Im(conj(alpha u) W lambda)
                        }
#pragma unroll
                        for (int r = 0; r < 3; ++r) { L[r] = M[r]; M[r] = Rt[r]; }
                    }
                }
            }
            const double w = 2.0 * PI * a.freqs[f], q = -2.0 * w * w;
            const cx<R> ey = m.eyn[y];
#pragma unroll
            for (int i = 0; i < MASS_SEG; ++i) {
                if (i < np) {
                    const cx<R> ex = m.exn[x0 + i];
                    const double cr = (double)ex.re * ey.re - (double)ex.im * ey.im, ci = (double)ex.re * ey.im + (double)ex.im * ey.re;
                    tr[i] += q * (cr * zr[i] + ci * zi[i]);  // Re(conj(C) z)
                    ti[i] += q * (cr * zi[i] - ci * zr[i]);  // Im(conj(C) z)
                }
            }
        }
#pragma unroll
        for (int i = 0; i < MASS_SEG; ++i) {
            if (i < np) {
                const double A = warp_sum(tr[i]), B = warp_sum(ti[i]);
                const long long p = (long long)y * m.Nx + x0 + i;
                if (lane == 0) {
                    const double s = (double)a.slow[p];
                    if constexpr (LOSSY) {
                        const double k = (double)a.kappa[p];
                        a.grad[p] = (R)(A * s - B * k);
                        a.grad_kappa[p] = (R)(-s * B - k * A);
                    } else {
                        a.grad[p] = (R)(A * s);
                    }
                }
            }
        }
    }
}

// Perturbation RHS of the discrete mode: Out_i = alpha_t sum_{j in N9(i)} w_ij c_j u_tj on interior rows, 0 on the ring, with
// c_j = -2 w^2 C_j sigma_j dsigma_j formed in FP64 once per node and frequency into the warp's shared-memory tile.
// grid = (blocks, nfreq); one warp per MASS_SEG-pixel row segment.  Two blocks per SM: unbounded, ptxas gives it 151-160
// registers and one block (8 warps) per SM.
template <typename R, int NS, bool LOSSY>
__global__ void __launch_bounds__(256, 2) pert_rhs_mass_kernel(PertArgs<R> a, MassArgs<R> m) {
    typedef Unit<R, NS> V;
    __shared__ cx<R> coef_all[8][3][MASS_SEG + 2];
    const int lane = threadIdx.x & 31;
    cx<R> (*coef)[MASS_SEG + 2] = coef_all[threadIdx.x >> 5];
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const double PI = 3.14159265358979323846;
    const int f = blockIdx.y;
    const double w = 2.0 * PI * a.freqs[f], q = -2.0 * w * w;
    const double d = m.bde[3 * f + 1], e = m.bde[3 * f + 2];
    const R c0 = (R)(1.0 - d - e), d4 = (R)(d * 0.25), e4 = (R)(e * 0.25);
    const cx<R>* u = a.U + (size_t)f * a.stride_f;
    cx<R>* out = a.Out + (size_t)f * a.stride_f;
    const V* al = reinterpret_cast<const V*>(a.src_est + (size_t)f * a.nt);
    const int nseg = (m.Nx + MASS_SEG - 1) / MASS_SEG, nunits = a.nt / NS;
    for (long long item = warp; item < (long long)m.Ny * nseg; item += nwarps) {
        const int y = (int)(item / nseg), x0 = (int)(item % nseg) * MASS_SEG;
        const int np = min(MASS_SEG, m.Nx - x0);
        __syncwarp();
        if (lane < 3 * (MASS_SEG + 2)) {
            const int r = lane / (MASS_SEG + 2), c = lane % (MASS_SEG + 2);
            const int yy = y - 1 + r, xx = x0 - 1 + c;
            double cr = 0.0, ci = 0.0;
            if (yy >= 0 && yy < m.Ny && xx >= 0 && xx < m.Nx) {
                const long long p = (long long)yy * m.Nx + xx;
                const cx<R> ex = m.exn[xx], ey = m.eyn[yy];
                const double Cr = (double)ex.re * ey.re - (double)ex.im * ey.im, Ci = (double)ex.re * ey.im + (double)ex.im * ey.re;
                double gr = (double)a.slow[p] * (double)a.sd[p], gi = 0.0;  // sigma dsigma
                if constexpr (LOSSY) {
                    const double s = (double)a.slow[p], k = (double)a.kappa[p], ds = (double)a.sd[p], dk = (double)a.sd_kappa[p];
                    gr = s * ds - k * dk;
                    gi = -(s * dk + k * ds);
                }
                cr = q * (Cr * gr - Ci * gi);
                ci = q * (Cr * gi + Ci * gr);
            }
            coef[r][c] = cx<R>((R)cr, (R)ci);
        }
        __syncwarp();
        const bool ring_row = y == 0 || y == m.Ny - 1;
        for (int k = lane; k < nunits; k += 32) {
            V L[3], M[3], Rt[3];
            mass_column(L, u, m, a.nt, y, x0 - 1, k, true);
            mass_column(M, u, m, a.nt, y, x0, k, true);
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
                for (int s = 0; s < NS; ++s) { L[r].c[s] = coef[r][0] * L[r].c[s]; M[r].c[s] = coef[r][1] * M[r].c[s]; }
            const V aa = al[k];
#pragma unroll
            for (int i = 0; i < MASS_SEG; ++i) {
                if (i < np) {
                    mass_column(Rt, u, m, a.nt, y, x0 + i + 1, k, true);
#pragma unroll
                    for (int r = 0; r < 3; ++r)
#pragma unroll
                        for (int s = 0; s < NS; ++s) Rt[r].c[s] = coef[r][i + 2] * Rt[r].c[s];
                    const int x = x0 + i;
                    V o;
#pragma unroll
                    for (int s = 0; s < NS; ++s)
                        o.c[s] = (ring_row || x == 0 || x == m.Nx - 1) ? cxzero<R>() : aa.c[s] * mass_apply<R, NS>(s, c0, d4, e4, L, M, Rt);
                    reinterpret_cast<V*>(out + ((size_t)y * m.Nx + x) * a.nt)[k] = o;
#pragma unroll
                    for (int r = 0; r < 3; ++r) { L[r] = M[r]; M[r] = Rt[r]; }
                }
            }
        }
    }
}

// num = Re<dREC, REC_DATA - REC_SIM>, den = Re<dREC, dREC> over kept receivers (nonlinearcg.py:22-28)
template <typename R>
struct LineArgs {
    const cx<R>* U;     // forward fields (unscaled)
    const cx<R>* Pert;  // perturbation fields
    size_t stride_f;
    const cx<R>* rec;
    const int* rx_lin;
    const int* mask;
    const cx<R>* src_est;
    double* out2;
    int nt, nm, nelem;
};

template <typename R>
__global__ void __launch_bounds__(256) linesearch_kernel(LineArgs<R> a) {
    __shared__ double sh[2 * 32];
    const int t = blockIdx.x, f = blockIdx.y;
    const cx<R>* Uf = a.U + (size_t)f * a.stride_f;
    const cx<R>* Pf = a.Pert + (size_t)f * a.stride_f;
    const cx<R>* recf = a.rec + ((size_t)f * a.nt + t) * a.nelem;
    const int* mk = a.mask + (size_t)t * a.nm;
    const cx<R> alpha = a.src_est[(size_t)f * a.nt + t];
    double s[2] = {0, 0};
    for (int j = threadIdx.x; j < a.nm; j += blockDim.x) {
        int e = mk[j];
        size_t o = (size_t)a.rx_lin[e] * a.nt + t;
        cx<R> d = Pf[o];
        cx<R> r = recf[e] - alpha * Uf[o];
        s[0] += (double)d.re * r.re + (double)d.im * r.im;
        s[1] += (double)d.re * d.re + (double)d.im * d.im;
    }
    block_sum<2>(s, sh);
    if (threadIdx.x == 0) {
        atomicAdd(a.out2 + 0, s[0]);
        atomicAdd(a.out2 + 1, s[1]);
    }
}

// Gauss-Newton product H_GN v = Re(J^H J v) (ustfwi.cu gn_hvp_enqueue).  After the perturbation solve Pert = H^-1(-VIRT v),
// J v of transmitter t is Pert at its kept receivers: gathered into drec [nfreq][nt][nm] (mask order, what linesearch_kernel
// reads as dREC) with sum |J v|^2 -> *jv2.  One CTA per (transmitter, frequency).
template <typename R>
struct GnRecvArgs {
    const cx<R>* Pert;  // perturbation fields [nfreq][N*nt]
    cx<R>* Lam;         // adjoint right-hand side [nfreq][N*nt], zeroed between the two kernels (gn_scatter_kernel)
    size_t stride_f;
    const int* rx_lin;
    const int* mask;
    const int* rx_next; // [nt][nm] receivers sharing a node (RecvArgs::rx_next)
    cx<R>* drec;        // [nfreq][nt][nm]
    double* jv2;
    int nt, nm;
};

template <typename R>
__global__ void __launch_bounds__(256) gn_receiver_kernel(GnRecvArgs<R> a) {
    __shared__ double sh[1 * 32];
    const int t = blockIdx.x, f = blockIdx.y;
    const cx<R>* Pf = a.Pert + (size_t)f * a.stride_f;
    const int* mk = a.mask + (size_t)t * a.nm;
    cx<R>* d_out = a.drec + ((size_t)f * a.nt + t) * a.nm;
    double s[1] = {0};
    for (int j = threadIdx.x; j < a.nm; j += blockDim.x) {
        const cx<R> d = Pf[(size_t)a.rx_lin[mk[j]] * a.nt + t];
        d_out[j] = d;
        s[0] += (double)d.re * d.re + (double)d.im * d.im;
    }
    block_sum<1>(s, sh);
    if (threadIdx.x == 0) atomicAdd(a.jv2, s[0]);
}

// J v as the adjoint source: the same stores as receiver_kernel's Lf[o] = d (one sum per node, in mask order), so that J^H is
// the adjoint of J and the one the gradient uses
template <typename R>
__global__ void __launch_bounds__(256) gn_scatter_kernel(GnRecvArgs<R> a) {
    const int t = blockIdx.x, f = blockIdx.y;
    cx<R>* Lf = a.Lam + (size_t)f * a.stride_f;
    const int* mk = a.mask + (size_t)t * a.nm;
    const int* nx = a.rx_next + (size_t)t * a.nm;
    const cx<R>* d_in = a.drec + ((size_t)f * a.nt + t) * a.nm;
    for (int j = threadIdx.x; j < a.nm; j += blockDim.x) {
        int k = nx[j];
        if (k < 0) continue;
        cx<R> d = d_in[j];
        for (; k < a.nm; k = -1 - nx[k]) d = d + d_in[k];
        Lf[(size_t)a.rx_lin[mk[j]] * a.nt + t] = d;
    }
}

// Residual of one forward column: r = H u_t - e_src(t) on the interior nodes, from the nine coefficient planes (what
// assemble_Helmholtz puts into row y*Nx+x, solve_helmholtz.py:242-260).  A size-independent check of the whole factor + sweep
// chain at any grid size: out2[0] += |r|^2, out2[1] += |H||u| row sums squared (the natural scale of the rounding errors).
template <typename R>
__global__ void __launch_bounds__(256) residual_onehot_kernel(Geom g, const cx<R>* __restrict__ planes_f, const cx<R>* __restrict__ U,
                                                               int nt, int t, int src_lin, double* __restrict__ out2) {
    __shared__ double sh[2 * 32];
    const long long node = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    double s[2] = {0.0, 0.0};
    if (node < g.N) {
        const int x = (int)(node % g.Nx), y = (int)(node / g.Nx);
        if (x > 0 && y > 0 && x < g.Nx - 1 && y < g.Ny - 1) {
            const size_t pl = (size_t)g.Nx * g.Ny;
            const int dy[9] = {0, 0, 0, -1, 1, -1, -1, 1, 1}, dx[9] = {0, -1, 1, 0, 0, -1, 1, -1, 1};  // plane order c,l,r,d,u,dl,dr,ul,ur
            double re = 0.0, im = 0.0, mag = 0.0;
#pragma unroll
            for (int p = 0; p < 9; ++p) {
                const cx<R> c = planes_f[p * pl + node];
                const cx<R> u = U[((size_t)(y + dy[p]) * g.Nx + (x + dx[p])) * nt + t];
                re += (double)c.re * u.re - (double)c.im * u.im;
                im += (double)c.re * u.im + (double)c.im * u.re;
                mag += sqrt(((double)c.re * c.re + (double)c.im * c.im) * ((double)u.re * u.re + (double)u.im * u.im));
            }
            if (node == src_lin) re -= 1.0;
            s[0] = re * re + im * im;
            s[1] = mag * mag;
        }
    }
    block_sum<2>(s, sh);
    if (threadIdx.x == 0) { atomicAdd(out2, s[0]); atomicAdd(out2 + 1, s[1]); }
}

// ---------------------------------------------------------------------------------------------
// Time-domain synthesis (Lecture19_Fwi/TimeDomainSimulation.m:48-56): inverse discrete-time Fourier transform of the
// frequency-domain wavefields, NOT an inverse FFT -- out[t][p] = sum_f W[t][f] * U[f][p] with
// W[t][f] = exp(i 2 pi f t) * df * resp(f) prepared by the host in double precision.
// One thread = one pixel p and IDTFT_TT consecutive time points; the weights of the CTA's time tile sit in shared
// memory, U[f][p] is read coalesced across p (the frequency stack stays L2 resident between time tiles).
// HBM roofline: the write of out (nt * npix complex).  grid = (ceil(npix/256), ceil(nt/IDTFT_TT)), 256 threads,
// dynamic smem = IDTFT_TT * nf complex.
// ---------------------------------------------------------------------------------------------
constexpr int IDTFT_TT = 8;

template <typename R>
__global__ void __launch_bounds__(256) idtft_kernel(const cx<R>* __restrict__ U, const cx<R>* __restrict__ W, cx<R>* __restrict__ out,
                                                    long long npix, int nf, int nt) {
    extern __shared__ __align__(16) unsigned char idtft_smem[];
    cx<R>* w = reinterpret_cast<cx<R>*>(idtft_smem);  // [IDTFT_TT][nf]
    const int t0 = blockIdx.y * IDTFT_TT;
    for (int e = threadIdx.x; e < IDTFT_TT * nf; e += blockDim.x) {
        const int tt = e / nf, f = e % nf;
        w[e] = (t0 + tt < nt) ? W[(size_t)(t0 + tt) * nf + f] : cxzero<R>();
    }
    __syncthreads();
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npix) return;
    cx<R> acc[IDTFT_TT];
#pragma unroll
    for (int tt = 0; tt < IDTFT_TT; ++tt) acc[tt] = cxzero<R>();
    for (int f = 0; f < nf; ++f) {
        const cx<R> u = U[(size_t)f * npix + p];
#pragma unroll
        for (int tt = 0; tt < IDTFT_TT; ++tt) cmac(acc[tt], w[tt * nf + f], u);
    }
#pragma unroll
    for (int tt = 0; tt < IDTFT_TT; ++tt)
        if (t0 + tt < nt) out[(size_t)(t0 + tt) * npix + p] = acc[tt];
}

}  // namespace ust
