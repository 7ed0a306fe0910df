// ustfwi.cu -- plan, launch schedules and the C ABI (include/ustfwi.h) of libustfwi.so.
//
// Everything here is host-side orchestration: the numerical work is in assemble.cuh (operator
// assembly), factor.cuh (two-sided block-tridiagonal factorisation), sweep.cuh (multi-RHS sweeps) and
// fwi.cuh (receiver / residual / gradient kernels).  No torch types, no exceptions across the boundary.
#include "../../include/ustfwi.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <type_traits>
#include <unordered_map>
#include <vector>

#include "assemble.cuh"
#include "common.cuh"
#include "factor.cuh"
#include "fwi.cuh"
#include "sweep.cuh"

namespace ust {
static thread_local std::string g_err;
thread_local long long g_launches = 0;
bool g_use_pdl = true;
thread_local bool g_pdl_batch_ok = true;
void set_error(const std::string& s) { g_err = s; }
}  // namespace ust

using namespace ust;

struct ust_plan {
    ust_plan_desc d;
    Geom g;
    size_t rsz, csz;  // sizeof real / complex
    double h = 0, gr = 1, a0 = 0, Lpml = 0;
    bool grid_set = false, acq_set = false, factored = false;
    bool use_tc2 = false; // TMA-fed tcgen05 engine for factor + sweeps (complex64 only)
    bool t_ring = false;  // FP32 T keeps 4 slots per frequency instead of all rows (TMA-fed engine: the sweeps read Tp)
    int prefetch_cin = 1; // L2 prefetch of a GEMM tile's Cin rows at CTA start (UST_TC2_PREFETCH=0 disables)
    // frequency groups: independent launch chains on separate streams (group 0 runs on the caller's / graph stream)
    static constexpr int MAX_GROUPS = 8;
    int ngroups = 2;
    cudaStream_t side[MAX_GROUPS] = {};
    cudaEvent_t ev_fork = nullptr, ev_join[MAX_GROUPS] = {};
    // complex128 look-ahead of the Gauss-Jordan pivot inversions: one high-priority side stream per group, forked / joined with events
    cudaStream_t pivst[MAX_GROUPS] = {};
    cudaEvent_t ev_upd[MAX_GROUPS] = {}, ev_piv[MAX_GROUPS][2] = {};
    uint16_t *Tp = nullptr, *Wp = nullptr;  // bf16 operand planes of the TC2 engine
    void* snap = nullptr;
    uint16_t *Rp = nullptr, *Cp = nullptr, *Xp = nullptr, *Pp = nullptr;  // panel / pivot planes of the TC2 Gauss-Jordan kernels
    size_t rp_stride = 0;
    CUtensorMap cmaps[2], pmaps[2];
    size_t wp_stride = 0;
    int kpad = 0;
    int gj_drain = 1, sweep_drain = 1;  // drain periods of the leading accumulator (UST_TC2_GJ_DRAIN / UST_TC2_SWEEP_DRAIN)
    float bias_fix = 2.5e-8f;  // measured truncation bias of one drained chunk (tools/exp_tc_accum.py)
    CUtensorMap amaps[2];
    int nfreq_cur = 0;
    std::vector<double> freqs_cur;
    size_t bytes = 0;
    int num_sms = 148;
    // device buffers
    void *exn = nullptr, *rexh = nullptr, *eyn = nullptr, *reyh = nullptr;
    double *d_vminmax = nullptr, *d_freqs = nullptr, *d_bde = nullptr, *d_scal = nullptr, *d_invv2 = nullptr;
    double* d_sig2 = nullptr;  // lossy models: complex sigma^2 per node (2N doubles, sig2_kernel)
    int* d_status = nullptr;
    void *planes = nullptr, *T = nullptr, *scratch = nullptr, *W = nullptr, *pbuf = nullptr;
    void *vel = nullptr, *U = nullptr, *Lam = nullptr, *src_est = nullptr, *Xh = nullptr;
    void *slow_h2d = nullptr, *rec_h2d = nullptr, *grad_d2h = nullptr;
    int *src_lin = nullptr, *rx_lin = nullptr, *mask = nullptr;
    int* rx_next = nullptr;  // [nt][nm] kept receivers sharing a node, chained in mask order (fwi.cuh RecvArgs::rx_next)
    int nt = 0, nelem = 0, nm = 0;
    bool onehot_ok = false;            // first_row / last_row valid (<= 8 column tiles)
    short first_row[8], last_row[8];   // per 128-column tile: smallest / largest interior block row holding a source
    // plan-owned copies of the FWI inputs / outputs (stable addresses for graph replay)
    void *slow_in = nullptr, *rec_in = nullptr, *grad_out = nullptr, *sd_in = nullptr;
    void *v_in = nullptr, *hv_out = nullptr, *drec = nullptr;  // Gauss-Newton product: v, H_GN v, J v at the kept receivers
    void *kappa_in = nullptr, *grad_kappa_out = nullptr;       // lossy evaluation: attenuation slowness, its gradient
    void *kappa_h2d = nullptr, *grad_kappa_d2h = nullptr;      // staging of ust_fwi_loss_grad_lossy_host
    void *vk_in = nullptr, *hv_kappa_out = nullptr;  // lossy line search / product: kappa part of the direction, of H_GN v
    // the last evaluation (ust_fwi_loss_grad[_lossy]), whose forward fields, source estimates and inputs the line search
    // and the Gauss-Newton product reuse (check_eval)
    enum EvalKind { EVAL_NONE, EVAL_LOSSLESS, EVAL_LOSSY };
    EvalKind eval_kind = EVAL_NONE;  // cleared by ust_plan_set_acquisition
    bool factored_since_eval = false;  // factor_impl ran after it: the factors no longer belong to its fields
    bool factors_lossy = false;        // the current factors are those of a lossy model
    int grad_mode = UST_GRAD_REFERENCE;  // ust_plan_set_gradient: linearisation of the evaluation, line search and product
    int eval_grad_mode = UST_GRAD_REFERENCE;  // the mode the last evaluation ran with
    bool use_graphs = true;  // UST_NO_GRAPHS=1 disables
    struct GraphEntry { cudaGraphExec_t exec = nullptr; long long launches = 0; };
    std::map<long long, GraphEntry> graphs;
    cudaEvent_t ev_in = nullptr, ev_out = nullptr;
    // pinned host staging for small parameter uploads
    double* h_stage = nullptr;  // 4*max_freq doubles
    cudaStream_t own_stream = nullptr;
    unsigned long long* trace = nullptr;  // UST_TC2_TRACE_UPDATE=step,k: in-situ phase timestamps of one update launch
    int trace_step = -1, trace_k = -1;
    int pdl_min_batch = 8;  // programmatic dependent launch only when the launch chains in flight carry more matrices than this in total
                            // (UST_PDL_MIN_BATCH; measured: 4 frequencies on one chain 145 vs 153 ms without / with, 8 frequencies on two chains 181 vs 177)
    int active_groups = 1;
    int eval_nfreq = 1;     // frequencies of the evaluation being enqueued (all groups)
    int ksplit_ok = 2;      // largest split-K cluster of the sweep GEMM (UST_KSPLIT = 1 (off), 2 or 4; measured at 2 frequencies: 43.2 / 33.7 / 40.7 ms of sweep GEMM)
    bool lookahead = true;  // next pivot block inverted by extra CTAs of the update launch (UST_NO_LOOKAHEAD=1 disables)
    // optional per-kernel-class device timing (ust_profile): event pairs around every launch
    bool prof = false;
    std::vector<cudaEvent_t> ev;
    std::vector<int> ev_cls;
    size_t ev_used = 0;
};

// brackets one kernel launch with CUDA events on the launching stream when profiling is on
struct ProfScope {
    ust_plan* p; long idx; cudaStream_t st;
    ProfScope(ust_plan* p_, int cls, cudaStream_t st_) : p(p_), idx(-1), st(st_) {
        if (p->prof && p->ev_used + 2 <= p->ev.size()) {
            idx = (long)p->ev_used; p->ev_used += 2; p->ev_cls[idx / 2] = cls;
            cudaEventRecord(p->ev[idx], st);
        }
    }
    ~ProfScope() { if (idx >= 0) cudaEventRecord(p->ev[idx + 1], st); }
};
enum ProfClass { PC_ASSEMBLE = 0, PC_SCHUR, PC_GJ_PANEL, PC_GJ_UPDATE, PC_TRI_APPLY, PC_SWEEP_GEMM, PC_RECEIVER, PC_GRADIENT, PC_T_SPLIT, PC_GJ_PIVOT, PC_GJ_ROWPANEL, PC_GJ_K0, PC_COUNT };

static int dev_alloc(ust_plan* p, void** ptr, size_t bytes) {
    UST_CUDA(cudaMalloc(ptr, bytes));
    p->bytes += bytes;
    return 0;
}

static int check_plan(const ust_plan* p) {
    if (!p) { set_error("null plan"); return 1; }
    return 0;
}

// debugging aid (UST_TC2_TRACE_UPDATE): dump the traced update launch -- CTA, SM, ns since the earliest CTA entered
static int dump_update_trace(ust_plan* p, cudaStream_t st) {
    std::vector<unsigned long long> h(19 * 1024);
    UST_CUDA(cudaStreamSynchronize(st));
    UST_CUDA(cudaMemcpy(h.data(), p->trace, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    unsigned long long t0 = ~0ull;
    for (int b = 0; b < 1024; ++b) if (h[16 * b] && h[16 * b] < t0) t0 = h[16 * b];
    for (int b = 0; b < 1024; ++b) {
        if (!h[16 * b]) continue;
        fprintf(stderr, "upd cta %4d sm %3d:", b, (int)h[16 * 1024 + b]);
        for (int i = 0; i < 16; ++i) fprintf(stderr, " %lld", h[16 * b + i] ? (long long)(h[16 * b + i] - t0) : -1LL);
        fprintf(stderr, " %lld", h[17 * 1024 + b] ? (long long)(h[17 * 1024 + b] - t0) : -1LL);  // pivot CTAs (rows 1000..): inversion done
        if (b >= 1000 && b < 1024)  // ... and the phase stamps of the blocked inversion
            for (int i = 0; i < 13; ++i) fprintf(stderr, " %lld", h[18 * 1024 + 16 * (b - 1000) + i] ? (long long)(h[18 * 1024 + 16 * (b - 1000) + i] - t0) : -1LL);
        fprintf(stderr, "\n");
    }
    UST_CUDA(cudaMemset(p->trace, 0, h.size() * sizeof(unsigned long long)));
    return 0;
}

// captured graphs bake kernel arguments (grid spacing, acquisition arrays, sizes): drop them when those change
static void drop_graphs(ust_plan* p) {
    for (auto& kv : p->graphs)
        if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    p->graphs.clear();
}

// -------------------------------------------------------------------------------------------------
// typed implementations
// -------------------------------------------------------------------------------------------------
template <typename R>
static int set_grid_impl(ust_plan* p, const double* x, const double* y, double a0, double L) {
    const int Nx = p->g.Nx, Ny = p->g.Ny;
    // h = mean(diff(x)), g = mean(diff(y))/h  (solve_helmholtz.py:24-26)
    double h = (x[Nx - 1] - x[0]) / (Nx - 1), gh = (y[Ny - 1] - y[0]) / (Ny - 1);
    p->h = h; p->gr = gh / h; p->a0 = a0; p->Lpml = L;
    // half-grid PML profiles (solve_helmholtz.py:31-56); e = 1 - i a0 (max(|x-xc|-xspan+L,0)/L)^2
    auto prof = [&](const double* c, int n, std::vector<cx<R>>& node, std::vector<cx<R>>& rhalf) {
        double cmin = c[0], cmax = c[n - 1];
        double ctr = 0.5 * (cmin + cmax), span = 0.5 * (cmax - cmin);
        node.resize(n); rhalf.resize(n);
        for (int i = 0; i < 2 * n - 1; ++i) {
            double xe = cmin + (cmax - cmin) * (double)i / (double)(2 * (n - 1));
            double s = fmax(fabs(xe - ctr) - span + L, 0.0) / L;
            double im = -a0 * s * s;
            if ((i & 1) == 0) node[i / 2] = cx<R>((R)1.0, (R)im);
            else {
                double d = 1.0 + im * im;  // 1/(1 + i im) = (1 - i im)/d
                rhalf[i / 2] = cx<R>((R)(1.0 / d), (R)(-im / d));
            }
        }
        rhalf[n - 1] = cx<R>((R)0, (R)0);
    };
    std::vector<cx<R>> exn, rexh, eyn, reyh;
    prof(x, Nx, exn, rexh);
    prof(y, Ny, eyn, reyh);
    UST_CUDA(cudaMemcpy(p->exn, exn.data(), Nx * sizeof(cx<R>), cudaMemcpyHostToDevice));
    UST_CUDA(cudaMemcpy(p->rexh, rexh.data(), Nx * sizeof(cx<R>), cudaMemcpyHostToDevice));
    UST_CUDA(cudaMemcpy(p->eyn, eyn.data(), Ny * sizeof(cx<R>), cudaMemcpyHostToDevice));
    UST_CUDA(cudaMemcpy(p->reyh, reyh.data(), Ny * sizeof(cx<R>), cudaMemcpyHostToDevice));
    p->grid_set = true;
    p->factored = false;
    return 0;
}

template <typename R>
static int gj_invert_batch(ust_plan* p, int phase, int step, int f0, int nf, cudaStream_t st, int gidx) {
    const Geom& g = p->g;
    const int nbatch = phase == PH_CHAIN ? 2 * nf : nf;
    FactorArgs<R> a;
    a.g = g; a.phase = phase; a.step = step; a.nbatch = nbatch;
    a.f0 = f0; a.zb0 = 2 * f0; a.t_ring = p->t_ring ? 1 : 0;
    // programmatic dependent launch when the chains in flight carry more than pdl_min_batch matrices, or when a launch is several
    // waves of tile CTAs anyway (one frequency at 2048^2: 2 matrices of 512 tiles each: 3017 vs 3148 ms with / without)
    ust::g_pdl_batch_ok = nbatch * p->active_groups > p->pdl_min_batch ||
                          (long long)nbatch * p->active_groups * cdiv_i(g.nP, tc2::TM) * (g.nP / tc2::TNH) > 2LL * p->num_sms;
    a.planes = (const cx<R>*)p->planes; a.T = (cx<R>*)p->T; a.scratch = (cx<R>*)p->scratch; a.pbuf = (cx<R>*)p->pbuf; a.status = p->d_status;
    a.Rp = p->Rp; a.Cp = p->Cp; a.Xp = p->Xp; a.Pp = p->Pp; a.Tp = p->Tp; a.rp_stride = p->rp_stride; a.nbmax = 2 * p->d.max_freq;
    a.inplace = p->use_tc2 ? 1 : 0; a.gj_drain = p->gj_drain; a.snap = (cx<R>*)p->snap;
    a.trace = p->trace; a.trace_step = p->trace_step; a.trace_k = p->trace_k;
    a.prefetch_cin = p->prefetch_cin;
    const int nblk = g.nP / GJ_NB;
    {
        dim3 grid(cdiv_i(g.nP, SchurTile<R>::TS), cdiv_i(g.nP, SchurTile<R>::TS), nbatch), block(16, 16);
        // TMA-fed engine: the CTA of tile (0, 0) also inverts it (= pivot block 0) and emits P_0
        const int pivot0 = (sizeof(R) == 4 && p->use_tc2) ? 1 : 0;
        ProfScope ps(p, PC_SCHUR, st);
        UST_CUDA(launch_pdl(schur_kernel<R>, grid, block, pivot0 ? gj_pivot2_scratch_bytes : 0, st, a, pivot0));
        UST_LAUNCH_CHECK();
    }
    const size_t smem = gj_rowpanel_smem<R>();
    if constexpr (sizeof(R) == 4) {
        if (p->use_tc2) {
            // everything GEMM-shaped on the TMA-fed tensor-core engine; operands travel between the kernels as bf16 planes
            {
                // block row 0 -> B planes, block column 0 -> A planes: one launch, two CTA roles
                ProfScope ps(p, PC_GJ_K0, st);
                const int nrow = cdiv_i(g.nP, tc2::TN), ncol = nblk > 1 ? cdiv_i(g.nP, 32) : 0;
                UST_CUDA(launch_pdl(gj_k0_kernel, dim3(nrow + ncol, 1, nbatch), dim3(256), 0, st, a, nrow));
            }
            UST_LAUNCH_CHECK();
            const bool la = p->lookahead && nblk > 1;
            const int tiles = cdiv_i(g.nP, tc2::TN), tiles_h = cdiv_i(g.nP, tc2::TNH);
            for (int k = 0; k < nblk; ++k) {
                {
                    ProfScope ps(p, PC_GJ_PANEL, st);
                    if (k > 0 && !la) {  // otherwise P_k came from the Schur launch / the look-ahead CTAs of the previous update launch
                        ProfScope p1(p, PC_GJ_PIVOT, st);
                        UST_CUDA(launch_pdl(gj_pivot_kernel<R>, dim3(1, 1, nbatch), dim3(256), gj_pivot2_smem_bytes, st, a, k, 0));
                        UST_LAUNCH_CHECK();
                    }
                    {
                        ProfScope p2(p, PC_GJ_ROWPANEL, st);
                        const int snap_cta = (la && k + 1 < nblk) ? 1 : 0;
                        UST_CUDA(launch_pdl(tc2_gj_rowpanel_kernel, dim3(tiles_h + snap_cta, 1, nbatch), dim3(tc2::NUM_THREADS_H), tc2::SMEM_BYTES_H, st, a, k, p->bias_fix, p->pmaps[0]));
                    }
                    UST_LAUNCH_CHECK();
                }
                if (nblk > 1) {
                    const int pivot_next = (la && k + 1 < nblk) ? 1 : 0;
                    ProfScope ps(p, PC_GJ_UPDATE, st);
                    UST_CUDA(launch_pdl(tc2_gj_update_kernel, dim3(nbatch * tiles * tiles_h + (pivot_next ? nbatch : 0)), dim3(tc2::NUM_THREADS_H),
                                        tc2::SMEM_BYTES_H, st, a, k, p->bias_fix, pivot_next, p->cmaps[0]));
                    UST_LAUNCH_CHECK();
                }
            }
            return 0;
        }
    }
    // complex128: pivot inversion k+1 one step ahead on a side stream, beside update k (gj_pivot_blocked_f64 with `form`)
    const bool la64 = sizeof(R) == 8 && p->lookahead && nblk > 1 && p->pivst[gidx] != nullptr;
    const size_t piv_smem = sizeof(R) == 8 ? gj_pivot_f64_smem_bytes : gj_pivot_smem<R>();
    for (int k = 0; k < nblk; ++k) {
        {
            ProfScope ps(p, PC_GJ_PANEL, st);
            if (k == 0 || !la64) {
                ProfScope p1(p, PC_GJ_PIVOT, st);
                gj_pivot_kernel<R><<<dim3(1, 1, nbatch), 256, piv_smem, st>>>(a, k, 0);
            } else {
                UST_CUDA(cudaStreamWaitEvent(st, p->ev_piv[gidx][k & 1], 0));  // P_k from the side stream
            }
            UST_LAUNCH_CHECK();
            {
                ProfScope p2(p, PC_GJ_ROWPANEL, st);
                gj_rowpanel_kernel<R><<<dim3(nblk, 1, nbatch), 256, smem, st>>>(a, k);
            }
            UST_LAUNCH_CHECK();
        }
        if (la64 && k + 1 < nblk) {
            cudaStream_t ps_st = p->pivst[gidx];
            UST_CUDA(cudaEventRecord(p->ev_upd[gidx], st));
            UST_CUDA(cudaStreamWaitEvent(ps_st, p->ev_upd[gidx], 0));
            {
                ProfScope p1(p, PC_GJ_PIVOT, ps_st);
                gj_pivot_kernel<R><<<dim3(1, 1, nbatch), 256, piv_smem, ps_st>>>(a, k + 1, 1);
            }
            UST_LAUNCH_CHECK();
            UST_CUDA(cudaEventRecord(p->ev_piv[gidx][(k + 1) & 1], ps_st));
        }
        if (nblk > 1) {
            {
                ProfScope ps(p, PC_GJ_UPDATE, st);
                gj_update_kernel<R><<<dim3(nblk, nblk - 1, nbatch), 256, 0, st>>>(a, k);
            }
            UST_LAUNCH_CHECK();
        }
    }
    return 0;
}

// frequencies / stencil weights -> device.  Pageable host source: cudaMemcpyAsync stages it before returning, so the
// caller's arrays may be reused immediately and no host synchronisation is needed (this part is never graph-captured).
static int upload_params(ust_plan* p, int nfreq, const double* freqs, const double* bde, cudaStream_t st) {
    if (!p->grid_set) { set_error("ust_factor: ust_plan_set_grid has not been called"); return 1; }
    if (nfreq < 1 || nfreq > p->d.max_freq) { set_error("ust_factor: nfreq out of range"); return 1; }
    UST_CUDA(cudaMemcpyAsync(p->d_freqs, freqs, nfreq * sizeof(double), cudaMemcpyHostToDevice, st));
    if (bde) UST_CUDA(cudaMemcpyAsync(p->d_bde, bde, 3 * nfreq * sizeof(double), cudaMemcpyHostToDevice, st));
    p->freqs_cur.assign(freqs, freqs + nfreq);
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// Frequency groups.  The factor / sweep chains are thousands of strictly dependent launches whose CTAs are latency
// bound (a rank-64 update CTA keeps the tensor pipe ~15 % busy) and whose look-ahead pivot inversion is close to the
// critical path.  Frequencies are independent, so the frequencies of one evaluation are split into `ngroups` groups,
// each an independent chain of launches on its own stream (group 0 on the caller's / graph-capture stream): the tail
// wave and the pivot chain of one group's launch run under the other groups' tiles, and an HBM-bound launch of one
// group (tri_apply2) overlaps a tensor-bound one of another.  Results are bit-identical to one group.
// ---------------------------------------------------------------------------------------------------------------
struct Group { int f0, nf; cudaStream_t st; int idx; };

static std::vector<Group> make_groups(ust_plan* p, int f_begin, int nfreq, cudaStream_t main_st, bool allow_split = true) {
    // a group needs >= 4 frequencies (8 chains): below that its launches are single partial waves without programmatic
    // dependent launch, and two such chains side by side are slower than one (2 frequencies at 512^2: 167 vs 148 ms)
    int G = std::min(std::min(p->ngroups, nfreq / 4), (int)ust_plan::MAX_GROUPS);
    if (p->prof || !allow_split || G < 1) G = 1;  // per-launch event timing wants one chain at a time
    p->active_groups = G;
    p->eval_nfreq = nfreq;
    std::vector<Group> gs;
    for (int i = 0; i < G; ++i) {
        const int lo = (int)((long long)nfreq * i / G), hi = (int)((long long)nfreq * (i + 1) / G);
        gs.push_back({f_begin + lo, hi - lo, i == 0 ? main_st : p->side[i], i});
    }
    return gs;
}
// side streams start after everything enqueued on the main stream so far ...
static int fork_groups(ust_plan* p, const std::vector<Group>& gs) {
    if (gs.size() < 2) return 0;
    UST_CUDA(cudaEventRecord(p->ev_fork, gs[0].st));
    for (size_t i = 1; i < gs.size(); ++i) UST_CUDA(cudaStreamWaitEvent(gs[i].st, p->ev_fork, 0));
    return 0;
}
// ... and the main stream continues after all of them
static int join_groups(ust_plan* p, const std::vector<Group>& gs) {
    for (size_t i = 1; i < gs.size(); ++i) {
        UST_CUDA(cudaEventRecord(p->ev_join[i], gs[i].st));
        UST_CUDA(cudaStreamWaitEvent(gs[0].st, p->ev_join[i], 0));
    }
    return 0;
}

// stencil weights (when not injected) + status reset: once per evaluation, before the groups fork
// kappa_dev != nullptr: lossy model, sigma^2 (sig2_kernel) instead of 1/v^2
template <typename R>
static int factor_prologue(ust_plan* p, const void* vel_dev, int nfreq, bool has_bde, cudaStream_t st, const void* kappa_dev = nullptr) {
    const Geom& g = p->g;
    if (!has_bde) {
        minmax_kernel<R><<<1, 1024, 0, st>>>((const R*)vel_dev, g.N, p->d_vminmax);
        UST_LAUNCH_CHECK();
        stencil_params_kernel<<<nfreq, 1024, 0, st>>>(p->d_vminmax, p->d_freqs, p->h, p->gr, p->d_bde);
        UST_LAUNCH_CHECK();
    }
    UST_CUDA(cudaMemsetAsync(p->d_status, 0, sizeof(int), st));
    if (kappa_dev) sig2_kernel<R><<<(unsigned)((g.N + 255) / 256), 256, 0, st>>>((const R*)vel_dev, (const R*)kappa_dev, (double2*)p->d_sig2, g.N);
    else inv_v2_kernel<R><<<(unsigned)((g.N + 255) / 256), 256, 0, st>>>((const R*)vel_dev, p->d_invv2, g.N);
    UST_LAUNCH_CHECK();
    return 0;
}

// assembly + factorisation of the groups' frequencies, device work only (CUDA-graph capturable); parameters must
// already be on the device.  Launches are enqueued step by step across the groups so that the streams fill evenly
// when the launches are not replayed from a graph.
template <typename R>
static int factor_groups(ust_plan* p, const void* vel_dev, const std::vector<Group>& gs, bool lossy = false) {
    const Geom& g = p->g;
    AsmArgs aa;
    aa.g = g; aa.h = p->h; aa.gr = p->gr; aa.stencil = p->d.stencil;
    for (const Group& q : gs)
        for (int c0 = 0; c0 < q.nf; c0 += ASM_MAXF) {
            const int f0 = q.f0 + c0;
            aa.nfreq = std::min(q.nf - c0, (int)ASM_MAXF);
            ProfScope ps(p, PC_ASSEMBLE, q.st);
            const dim3 grid(cdiv_i(g.Nx, 256), g.Ny);
            if (lossy)
                assemble_kernel<R, true><<<grid, 256, 0, q.st>>>(
                    aa, p->d_sig2, (const cx<R>*)p->exn, (const cx<R>*)p->rexh, (const cx<R>*)p->eyn, (const cx<R>*)p->reyh,
                    p->d_freqs + f0, p->d_bde + 3 * f0, (cx<R>*)p->planes + (size_t)f0 * 9 * g.N);
            else
                assemble_kernel<R, false><<<grid, 256, 0, q.st>>>(
                    aa, p->d_invv2, (const cx<R>*)p->exn, (const cx<R>*)p->rexh, (const cx<R>*)p->eyn, (const cx<R>*)p->reyh,
                    p->d_freqs + f0, p->d_bde + 3 * f0, (cx<R>*)p->planes + (size_t)f0 * 9 * g.N);
            UST_LAUNCH_CHECK();
        }
    const int len = std::max(g.mid, g.M - 1 - g.mid);
    for (int s = 0; s < len; ++s)
        for (const Group& q : gs) UST_TRY(gj_invert_batch<R>(p, PH_CHAIN, s, q.f0, q.nf, q.st, q.idx));
    for (const Group& q : gs) UST_TRY(gj_invert_batch<R>(p, PH_MID, 0, q.f0, q.nf, q.st, q.idx));
    return 0;
}

template <typename R>
static int factor_enqueue(ust_plan* p, const void* vel_dev, int nfreq, bool has_bde, cudaStream_t st, const void* kappa_dev) {
    UST_TRY(factor_prologue<R>(p, vel_dev, nfreq, has_bde, st, kappa_dev));
    const std::vector<Group> gs = make_groups(p, 0, nfreq, st);
    UST_TRY(fork_groups(p, gs));
    UST_TRY(factor_groups<R>(p, vel_dev, gs, kappa_dev != nullptr));
    UST_TRY(join_groups(p, gs));
    p->nfreq_cur = nfreq;
    p->factored = true;
    return 0;
}

// kappa_dev != nullptr: the lossy operator of the complex slowness 1/vel - i kappa (ust_factor_lossy)
template <typename R>
static int factor_impl(ust_plan* p, const void* vel_dev, int nfreq, const double* freqs, const double* bde, cudaStream_t st,
                       const void* kappa_dev = nullptr) {
    p->factored_since_eval = true;
    p->factors_lossy = kappa_dev != nullptr;
    UST_TRY(upload_params(p, nfreq, freqs, bde, st));
    return factor_enqueue<R>(p, vel_dev, nfreq, bde != nullptr, st, kappa_dev);
}

template <typename R, int BM, int BN>
static int launch_sweep_gemm(ust_plan* p, const SweepArgs<R>& s, dim3 grid, cudaStream_t st) {
    {
        ProfScope ps(p, PC_SWEEP_GEMM, st);
        if (s.adjoint) sweep_gemm_kernel<R, BM, BN, true><<<grid, 256, 0, st>>>(s);
        else sweep_gemm_kernel<R, BM, BN, false><<<grid, 256, 0, st>>>(s);
    }
    UST_LAUNCH_CHECK();
    return 0;
}

template <typename R>
static int sweep_step(ust_plan* p, SweepArgs<R>& s, cudaStream_t st) {
    const Geom& g = p->g;
    const long long elems = (long long)g.nI * s.nrhs;
    ust::g_pdl_batch_ok = s.nbatch * p->active_groups > p->pdl_min_batch;
    if constexpr (sizeof(R) == 4) {
        if (p->use_tc2) {
            Tc2SweepExtra x;
            x.Wp = p->Wp + (size_t)2 * s.f0 * p->wp_stride;  // per-chain scratch: chains of frequency f are 2f, 2f+1
            x.wp_stride = p->wp_stride; x.kpad = p->kpad; x.bias_fix = p->bias_fix; x.drain_every = p->sweep_drain;
            x.prefetch_cin = p->prefetch_cin; x.ksplit = 1;
            {
                ProfScope ps(p, PC_TRI_APPLY, st);
                UST_CUDA(launch_pdl(tri_apply2_kernel, dim3(p->kpad / 8, cdiv_i(s.nrhs, tc2::TN), s.nbatch), dim3(128), 0, st, s, x));
            }
            UST_LAUNCH_CHECK();
            dim3 grid(cdiv_i(s.nrhs, tc2::TN), cdiv_i(g.nI, tc2::TM), s.nbatch);
            // Few tiles (one to four frequencies on this GPU): a launch is as long as one tile's k loop and most SMs idle; two
            // CTAs (a cluster) then share a tile's k range and add their partial tiles through distributed shared memory.
            // Decided from the whole evaluation (all chains of all groups), so that it does not depend on the grouping.
            const long long all_tiles = 2LL * p->eval_nfreq * grid.x * grid.y;
            const int nchunks = p->kpad / tc2::KC;
            x.ksplit = 1;
            if (p->ksplit_ok >= 2 && 2 * all_tiles <= p->num_sms && nchunks >= 8) x.ksplit = 2;
            if (p->ksplit_ok >= 4 && 4 * all_tiles <= p->num_sms && nchunks >= 16) x.ksplit = 4;
            {
                ProfScope ps(p, PC_SWEEP_GEMM, st);
                if (x.ksplit > 1) {
                    grid.x *= x.ksplit;
                    if (s.adjoint) UST_CUDA(launch_pdl_cluster(tc2_sweep_gemm_kernel<true>, grid, dim3(tc2::NUM_THREADS), tc2::SMEM_BYTES, st, (unsigned)x.ksplit, s, x, p->amaps[1]));
                    else UST_CUDA(launch_pdl_cluster(tc2_sweep_gemm_kernel<false>, grid, dim3(tc2::NUM_THREADS), tc2::SMEM_BYTES, st, (unsigned)x.ksplit, s, x, p->amaps[0]));
                } else if (s.adjoint) UST_CUDA(launch_pdl(tc2_sweep_gemm_kernel<true>, grid, dim3(tc2::NUM_THREADS), tc2::SMEM_BYTES, st, s, x, p->amaps[1]));
                else UST_CUDA(launch_pdl(tc2_sweep_gemm_kernel<false>, grid, dim3(tc2::NUM_THREADS), tc2::SMEM_BYTES, st, s, x, p->amaps[0]));
            }
            UST_LAUNCH_CHECK();
            return 0;
        }
    }
    {
        ProfScope ps(p, PC_TRI_APPLY, st);
        tri_apply_kernel<R><<<dim3((unsigned)((elems + 255) / 256), 1, s.nbatch), 256, 0, st>>>(s);
    }
    UST_LAUNCH_CHECK();
    const int bn = s.nrhs > 32 ? 64 : 32;
    int bm = 64;
    if ((long long)cdiv_i(g.nI, 64) * cdiv_i(s.nrhs, bn) * s.nbatch < p->num_sms) bm = 32;
    dim3 grid(cdiv_i(s.nrhs, bn), cdiv_i(g.nI, bm), s.nbatch);
    if (bm == 64 && bn == 64) return launch_sweep_gemm<R, 64, 64>(p, s, grid, st);
    if (bm == 32 && bn == 64) return launch_sweep_gemm<R, 32, 64>(p, s, grid, st);
    if (bm == 64 && bn == 32) return launch_sweep_gemm<R, 64, 32>(p, s, grid, st);
    return launch_sweep_gemm<R, 32, 32>(p, s, grid, st);
}

// All block sweeps of one multi-RHS solve for the groups' frequencies.  X holds one (N, nrhs) array per plan frequency
// slot (x_stride apart, slot 0 first); a group with x_stride == 0 solves a single caller-owned array.
template <typename R>
static int sweeps_groups(ust_plan* p, const std::vector<Group>& gs, cx<R>* X, size_t x_stride, int nrhs, int adjoint, bool onehot = false) {
    const Geom& g = p->g;
    std::vector<SweepArgs<R>> sv(gs.size());
    for (size_t i = 0; i < gs.size(); ++i) {
        SweepArgs<R>& s = sv[i];
        const int f0 = gs[i].f0;
        s.g = g; s.adjoint = adjoint; s.nrhs = nrhs;
        s.onehot = (onehot && p->onehot_ok) ? 1 : 0;
        for (int j = 0; j < 8; ++j) { s.first_row[j] = p->first_row[j]; s.last_row[j] = p->last_row[j]; }
        s.planes = (const cx<R>*)p->planes + (size_t)f0 * 9 * g.N;
        s.T = (const cx<R>*)p->T + (size_t)f0 * g.M * (size_t)g.nP * g.nP;  // FMA engines only (all rows kept)
        s.W = (cx<R>*)p->W + (size_t)2 * f0 * g.nP * p->d.max_nrhs;
        s.X = X + (size_t)f0 * x_stride; s.x_stride = x_stride; s.f0 = f0;
    }
    const int len = std::max(g.mid, g.M - 1 - g.mid);
    for (int step = 0; step < len; ++step)
        for (size_t i = 0; i < gs.size(); ++i) {
            SweepArgs<R>& s = sv[i];
            s.mode = SW_ELIM; s.phase = PH_CHAIN; s.nbatch = 2 * gs[i].nf; s.step = step;
            UST_TRY(sweep_step<R>(p, s, gs[i].st));
        }
    for (size_t i = 0; i < gs.size(); ++i) {
        SweepArgs<R>& s = sv[i];
        s.mode = SW_ELIM; s.phase = PH_MID; s.nbatch = gs[i].nf; s.step = 0;
        UST_TRY(sweep_step<R>(p, s, gs[i].st));
    }
    for (int step = len - 1; step >= 0; --step)
        for (size_t i = 0; i < gs.size(); ++i) {
            SweepArgs<R>& s = sv[i];
            s.mode = SW_BACK; s.phase = PH_CHAIN; s.nbatch = 2 * gs[i].nf; s.step = step;
            UST_TRY(sweep_step<R>(p, s, gs[i].st));
        }
    return 0;
}

template <typename R>
static int ring_fix(ust_plan* p, int ifreq, cx<R>* X, int nrhs, int adjoint, bool before, cudaStream_t st) {
    const Geom& g = p->g;
    const cx<R>* planes_f = (const cx<R>*)p->planes + (size_t)ifreq * 9 * g.N;
    if (!adjoint && before) {
        int count = 2 * g.nI + 2 * std::max(g.M - 2, 0);
        long long th = (long long)count * nrhs;
        ring_pre_kernel<R><<<(unsigned)((th + 255) / 256), 256, 0, st>>>(g, planes_f, X, nrhs, count);
        UST_LAUNCH_CHECK();
    } else if (adjoint && !before) {
        int count = 2 * g.Nx + 2 * (g.Ny - 2);
        long long th = (long long)count * nrhs;
        ring_post_adj_kernel<R><<<(unsigned)((th + 255) / 256), 256, 0, st>>>(g, planes_f, X, nrhs, count);
        UST_LAUNCH_CHECK();
    }
    return 0;
}

template <typename R>
static int solve_impl(ust_plan* p, int ifreq, void* X, int nrhs, int adjoint, cudaStream_t st) {
    if (!p->factored) { set_error("ust_solve: no factorisation (call ust_factor first)"); return 1; }
    if (ifreq < 0 || ifreq >= p->nfreq_cur) { set_error("ust_solve: ifreq out of range"); return 1; }
    if (nrhs < 1 || nrhs > p->d.max_nrhs) { set_error("ust_solve: nrhs exceeds plan max_nrhs"); return 1; }
    UST_TRY(ring_fix<R>(p, ifreq, (cx<R>*)X, nrhs, adjoint, true, st));
    // a stand-alone solve is one frequency on one chain: the split-K choice of its sweeps (sweep_step) depends on this solve
    // alone, not on how many frequencies the plan's last factorisation or evaluation had
    p->eval_nfreq = 1;
    p->active_groups = 1;
    const std::vector<Group> one = {{ifreq, 1, st}};
    UST_TRY(sweeps_groups<R>(p, one, (cx<R>*)X, 0, nrhs, adjoint));
    UST_TRY(ring_fix<R>(p, ifreq, (cx<R>*)X, nrhs, adjoint, false, st));
    return 0;
}

// standalone GEMM launchers for the engine unit test (ust_test_cgemm)
template <bool TA>
__global__ void __launch_bounds__(tc2::NUM_THREADS, 1) tc2_test_gemm_kernel(tc2::Tc2Tile t, const __grid_constant__ CUtensorMap amap) {
    extern __shared__ __align__(1024) unsigned char tc2_smem[];
    t.m0 = blockIdx.y * tc2::TM; t.n0 = blockIdx.x * tc2::TN;
    if (blockIdx.x | blockIdx.y | blockIdx.z) t.trace = nullptr;
    tc2::cgemm_tile<TA>(t, &amap, tc2_smem);
}
__global__ void __launch_bounds__(tc2::NUM_THREADS_H, 2) tc2h_test_gemm_kernel(tc2::Tc2Tile t, const __grid_constant__ CUtensorMap amap) {
    extern __shared__ __align__(1024) unsigned char tc2_smem[];
    t.m0 = blockIdx.y * tc2::TM; t.n0 = blockIdx.x * tc2::TNH;
    if (blockIdx.x | blockIdx.y | blockIdx.z) t.trace = nullptr;
    tc2::cgemm_tile_h(t, &amap, tc2_smem);
}
template <bool TA>
__global__ void __launch_bounds__(256) simt_test_gemm_kernel(GemmTile<float> t) {
    __shared__ GemmSmem<float, 64, 64> sm;
    t.m0 = blockIdx.y * 64; t.n0 = blockIdx.x * 64;
    cgemm_tile<float, 64, 64, TA>(t, sm);
}

// float64 values as (hi, lo) float32 pairs, hi + lo = value to ~1e-14 relative (for hosts that cannot hold float64: JAX with x64 disabled)
__global__ void pack_f32x2_kernel(const double* __restrict__ in, float* __restrict__ out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double v = in[i];
    const float hi = (float)v;
    out[2 * i] = hi;
    out[2 * i + 1] = (float)(v - (double)hi);
}

template <typename R>
__global__ void recip_kernel(const R* __restrict__ in, R* __restrict__ out, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = R(1) / in[i];
}

// stencil weights and PML factors of the discrete gradient mode's kernels, for the frequencies from f0 on
template <typename R>
static MassArgs<R> mass_args(const ust_plan* p, int f0) {
    MassArgs<R> m;
    m.exn = (const cx<R>*)p->exn; m.eyn = (const cx<R>*)p->eyn; m.bde = p->d_bde + 3 * f0; m.Nx = p->g.Nx; m.Ny = p->g.Ny;
    return m;
}

// Calls launch(NS) with the unit width of the discrete-mode kernels: complex64 lanes load two sources (16 B) when every pixel's
// source row is 16-byte aligned (even nt), one otherwise; complex128 lanes load one.
template <typename R, typename F>
static void with_mass_unit(const ust_plan* p, F launch) {
    if constexpr (sizeof(R) == 4) {
        if ((p->nt & 1) == 0) { launch(std::integral_constant<int, 2>()); return; }
    }
    launch(std::integral_constant<int, 1>());
}

// Gradient over all frequencies of the evaluation into ga.grad (lossy: also ga.grad_kappa): gradient_kernel, or in the discrete
// mode gradient_mass_kernel
template <typename R>
static int gradient_launch(ust_plan* p, const GradArgs<R>& ga, bool lossy, cudaStream_t st) {
    const Geom& g = p->g;
    ProfScope ps(p, PC_GRADIENT, st);
    if (p->grad_mode == UST_GRAD_DISCRETE) {
        const MassArgs<R> m = mass_args<R>(p, 0);
        const long long items = (long long)g.Ny * cdiv_i(g.Nx, MASS_SEG);
        const int blocks = (int)std::min<long long>((items + 7) / 8, (long long)p->num_sms * 8);
        with_mass_unit<R>(p, [&](auto ns) {
            if (lossy) gradient_mass_kernel<R, ns.value, true><<<blocks, 256, 0, st>>>(ga, m);
            else gradient_mass_kernel<R, ns.value, false><<<blocks, 256, 0, st>>>(ga, m);
        });
    } else {
        const int blocks = (int)std::min<long long>((g.N + 7) / 8, (long long)p->num_sms * 8);
        if (lossy) gradient_kernel<R, true><<<blocks, 256, 0, st>>>(ga);
        else gradient_kernel<R, false><<<blocks, 256, 0, st>>>(ga);
    }
    UST_LAUNCH_CHECK();
    return 0;
}

// One joint (loss, grad) evaluation, device work only (CUDA-graph capturable): reads p->slow_in / p->rec_in, writes
// p->d_scal[0] (loss) and p->grad_out.  Each frequency group runs assemble -> factor -> forward sweeps -> receivers ->
// adjoint sweeps as its own chain; the groups meet again at the gradient, which sums over all frequencies.
// lossy: also reads p->kappa_in (sigma^2 assembly) and writes p->grad_kappa_out; everything between assembly and gradient is the same.
template <typename R>
static int fwi_enqueue(ust_plan* p, int nfreq, bool has_bde, cudaStream_t st, bool lossy) {
    const Geom& g = p->g;
    const int nt = p->nt;
    const size_t stride = (size_t)g.N * nt;
    const void* slow = p->slow_in;
    double* loss_dev = p->d_scal;
    recip_kernel<R><<<(unsigned)((g.N + 255) / 256), 256, 0, st>>>((const R*)slow, (R*)p->vel, g.N);  // VEL = 1/SLOW (fwi_loss_function.py:50)
    UST_LAUNCH_CHECK();
    UST_TRY(factor_prologue<R>(p, p->vel, nfreq, has_bde, st, lossy ? p->kappa_in : nullptr));
    UST_CUDA(cudaMemsetAsync(loss_dev, 0, sizeof(double), st));
    const std::vector<Group> gs = make_groups(p, 0, nfreq, st);
    UST_TRY(fork_groups(p, gs));
    UST_TRY(factor_groups<R>(p, p->vel, gs, lossy));
    // forward: one-hot sources
    for (const Group& q : gs) {
        cx<R>* Uq = (cx<R>*)p->U + (size_t)q.f0 * stride;
        UST_CUDA(cudaMemsetAsync(Uq, 0, stride * q.nf * sizeof(cx<R>), q.st));
        onehot_scatter_kernel<R><<<cdiv_i(nt * q.nf, 256), 256, 0, q.st>>>(Uq, stride, p->src_lin, nt, q.nf);
        UST_LAUNCH_CHECK();
    }
    UST_TRY(sweeps_groups<R>(p, gs, (cx<R>*)p->U, stride, nt, 0, true));  // one-hot sources, U zero-filled above
    // receivers: alpha, residual, loss, adjoint source
    for (const Group& q : gs) {
        UST_CUDA(cudaMemsetAsync((cx<R>*)p->Lam + (size_t)q.f0 * stride, 0, stride * q.nf * sizeof(cx<R>), q.st));
        RecvArgs<R> ra;
        ra.U = (const cx<R>*)p->U + (size_t)q.f0 * stride; ra.Lam = (cx<R>*)p->Lam + (size_t)q.f0 * stride; ra.stride_f = stride;
        ra.rec = (const cx<R>*)p->rec_in + (size_t)q.f0 * nt * p->nelem;
        ra.rx_lin = p->rx_lin; ra.mask = p->mask; ra.rx_next = p->rx_next; ra.src_est = (cx<R>*)p->src_est + (size_t)q.f0 * nt; ra.loss = loss_dev;
        ra.nt = nt; ra.nm = p->nm; ra.nelem = p->nelem;
        ProfScope ps(p, PC_RECEIVER, q.st);
        receiver_kernel<R><<<dim3(nt, q.nf), 256, 0, q.st>>>(ra);
        UST_LAUNCH_CHECK();
    }
    // adjoint sweeps on the same factors
    UST_TRY(sweeps_groups<R>(p, gs, (cx<R>*)p->Lam, stride, nt, 1));
    for (const Group& q : gs)
        for (int f = q.f0; f < q.f0 + q.nf; ++f) UST_TRY(ring_fix<R>(p, f, (cx<R>*)p->Lam + (size_t)f * stride, nt, 1, false, q.st));
    UST_TRY(join_groups(p, gs));
    // gradient
    GradArgs<R> ga;
    ga.U = (const cx<R>*)p->U; ga.Lam = (const cx<R>*)p->Lam; ga.stride_f = stride; ga.src_est = (const cx<R>*)p->src_est;
    ga.freqs = p->d_freqs; ga.slow = (const R*)slow; ga.grad = (R*)p->grad_out; ga.N = g.N; ga.nt = nt; ga.nfreq = nfreq;
    ga.kappa = (const R*)p->kappa_in; ga.grad_kappa = (R*)p->grad_kappa_out;
    return gradient_launch<R>(p, ga, lossy, st);
}

// RHS of the perturbation solve for every group, from the direction `dir` (and, lossy, its kappa part p->vk_in)
template <typename R>
static int pert_rhs_groups(ust_plan* p, const std::vector<Group>& gs, const void* dir, bool lossy) {
    const int nt = p->nt;
    const size_t stride = (size_t)p->g.N * nt;
    for (const Group& q : gs) {
        PertArgs<R> pa;
        pa.U = (const cx<R>*)p->U + (size_t)q.f0 * stride; pa.Out = (cx<R>*)p->Lam + (size_t)q.f0 * stride; pa.stride_f = stride;
        pa.src_est = (const cx<R>*)p->src_est + (size_t)q.f0 * nt;
        pa.freqs = p->d_freqs + q.f0; pa.slow = (const R*)p->slow_in; pa.sd = (const R*)dir; pa.N = p->g.N; pa.nt = nt; pa.nfreq = q.nf;
        pa.kappa = (const R*)p->kappa_in; pa.sd_kappa = (const R*)p->vk_in;
        if (p->grad_mode == UST_GRAD_DISCRETE) {  // profiled as "receiver" (the reference RHS is not profiled)
            ProfScope ps(p, PC_RECEIVER, q.st);
            const MassArgs<R> m = mass_args<R>(p, q.f0);
            const long long items = (long long)p->g.Ny * cdiv_i(p->g.Nx, MASS_SEG);
            const dim3 grid((unsigned)std::min<long long>((items + 7) / 8, (long long)p->num_sms * 8), q.nf);
            with_mass_unit<R>(p, [&](auto ns) {
                if (lossy) pert_rhs_mass_kernel<R, ns.value, true><<<grid, 256, 0, q.st>>>(pa, m);
                else pert_rhs_mass_kernel<R, ns.value, false><<<grid, 256, 0, q.st>>>(pa, m);
            });
        } else {
            if (lossy) pert_rhs_kernel<R, true><<<dim3(p->num_sms * 4, q.nf), 256, 0, q.st>>>(pa);
            else pert_rhs_kernel<R, false><<<dim3(p->num_sms * 4, q.nf), 256, 0, q.st>>>(pa);
        }
        UST_LAUNCH_CHECK();
    }
    return 0;
}

// perturbation solve + line-search scalars, device work only: reads p->sd_in (lossy: also p->kappa_in and p->vk_in), writes
// p->d_scal[2..3]
template <typename R>
static int linesearch_enqueue(ust_plan* p, cudaStream_t st, bool lossy) {
    const Geom& g = p->g;
    const int nt = p->nt, nfreq = p->nfreq_cur;
    const size_t stride = (size_t)g.N * nt;
    double* out2 = p->d_scal + 2;
    UST_CUDA(cudaMemsetAsync(out2, 0, 2 * sizeof(double), st));
    const std::vector<Group> gs = make_groups(p, 0, nfreq, st);
    UST_TRY(fork_groups(p, gs));
    UST_TRY(pert_rhs_groups<R>(p, gs, p->sd_in, lossy));
    UST_TRY(sweeps_groups<R>(p, gs, (cx<R>*)p->Lam, stride, nt, 0));
    for (const Group& q : gs) {
        LineArgs<R> la;
        la.U = (const cx<R>*)p->U + (size_t)q.f0 * stride; la.Pert = (const cx<R>*)p->Lam + (size_t)q.f0 * stride; la.stride_f = stride;
        la.rec = (const cx<R>*)p->rec_in + (size_t)q.f0 * nt * p->nelem;
        la.rx_lin = p->rx_lin; la.mask = p->mask; la.src_est = (const cx<R>*)p->src_est + (size_t)q.f0 * nt; la.out2 = out2;
        la.nt = nt; la.nm = p->nm; la.nelem = p->nelem;
        linesearch_kernel<R><<<dim3(nt, q.nf), 256, 0, q.st>>>(la);
        UST_LAUNCH_CHECK();
    }
    UST_TRY(join_groups(p, gs));
    return 0;
}

// Gauss-Newton Hessian-vector product hv = Re(J^H J v) on the factors, forward fields and source estimates of the last
// evaluation, device work only: reads p->v_in, writes p->hv_out, p->drec (J v) and p->d_scal[6] (sum |J v|^2).  Per group:
// perturbation solve with RHS -VIRT*v (as linesearch_enqueue), J v gathered at the kept receivers, scattered back as the
// adjoint source, adjoint sweeps (as fwi_enqueue); the groups meet at gradient_kernel, which forms sum_f -Re(conj(VIRT) * adj).
// lossy: the complex-slowness RHS from v = [p->v_in, p->vk_in], and gradient_kernel<R, true> on p->slow_in / p->kappa_in writes
// both halves of J^H (J v): p->hv_out and p->hv_kappa_out.
template <typename R>
static int gn_hvp_enqueue(ust_plan* p, cudaStream_t st, bool lossy) {
    const Geom& g = p->g;
    const int nt = p->nt, nfreq = p->nfreq_cur;
    const size_t stride = (size_t)g.N * nt;
    double* jv2 = p->d_scal + 6;
    UST_CUDA(cudaMemsetAsync(jv2, 0, sizeof(double), st));
    const std::vector<Group> gs = make_groups(p, 0, nfreq, st);
    UST_TRY(fork_groups(p, gs));
    UST_TRY(pert_rhs_groups<R>(p, gs, p->v_in, lossy));
    UST_TRY(sweeps_groups<R>(p, gs, (cx<R>*)p->Lam, stride, nt, 0));
    for (const Group& q : gs) {
        GnRecvArgs<R> ra;
        ra.Pert = (const cx<R>*)p->Lam + (size_t)q.f0 * stride; ra.Lam = (cx<R>*)p->Lam + (size_t)q.f0 * stride; ra.stride_f = stride;
        ra.rx_lin = p->rx_lin; ra.mask = p->mask; ra.rx_next = p->rx_next; ra.drec = (cx<R>*)p->drec + (size_t)q.f0 * nt * p->nm; ra.jv2 = jv2;
        ra.nt = nt; ra.nm = p->nm;
        {
            ProfScope ps(p, PC_RECEIVER, q.st);
            gn_receiver_kernel<R><<<dim3(nt, q.nf), 256, 0, q.st>>>(ra);
        }
        UST_LAUNCH_CHECK();
        UST_CUDA(cudaMemsetAsync((cx<R>*)p->Lam + (size_t)q.f0 * stride, 0, stride * q.nf * sizeof(cx<R>), q.st));
        {
            ProfScope ps(p, PC_RECEIVER, q.st);
            gn_scatter_kernel<R><<<dim3(nt, q.nf), 256, 0, q.st>>>(ra);
        }
        UST_LAUNCH_CHECK();
    }
    UST_TRY(sweeps_groups<R>(p, gs, (cx<R>*)p->Lam, stride, nt, 1));
    for (const Group& q : gs)
        for (int f = q.f0; f < q.f0 + q.nf; ++f) UST_TRY(ring_fix<R>(p, f, (cx<R>*)p->Lam + (size_t)f * stride, nt, 1, false, q.st));
    UST_TRY(join_groups(p, gs));
    GradArgs<R> ga;
    ga.U = (const cx<R>*)p->U; ga.Lam = (const cx<R>*)p->Lam; ga.stride_f = stride; ga.src_est = (const cx<R>*)p->src_est;
    ga.freqs = p->d_freqs; ga.slow = (const R*)p->slow_in; ga.grad = (R*)p->hv_out; ga.N = g.N; ga.nt = nt; ga.nfreq = nfreq;
    ga.kappa = (const R*)p->kappa_in; ga.grad_kappa = (R*)p->hv_kappa_out;
    return gradient_launch<R>(p, ga, lossy, st);
}

// Run `enqueue` on the caller's stream directly, or -- the normal case -- as a CUDA graph captured once per key and
// replayed: a step is ~2e4 dependent launches of 5-100 us each, and at ~10 us of host time per launch the CPU, not
// the GPU, sets the pace as soon as the per-GPU batch is small.  Graphs run on the plan's own stream (the caller's may
// be the legacy default stream, which cannot be captured), fenced by events on both sides.
template <typename F>
static int run_graphed(ust_plan* p, long long key, cudaStream_t user, F enqueue) {
    if (!p->use_graphs || p->prof) return enqueue(user);
    cudaStream_t gs = p->own_stream;
    auto it = p->graphs.find(key);
    if (it == p->graphs.end()) {
        const long long before = ust::g_launches;
        UST_CUDA(cudaStreamBeginCapture(gs, cudaStreamCaptureModeThreadLocal));
        int rc = enqueue(gs);
        cudaGraph_t graph = nullptr;
        cudaError_t e = cudaStreamEndCapture(gs, &graph);
        if (rc || e != cudaSuccess || !graph) {
            if (graph) cudaGraphDestroy(graph);
            if (!rc) set_error(std::string("CUDA graph capture failed: ") + cudaGetErrorString(e));
            cudaGetLastError();
            return 1;
        }
        ust_plan::GraphEntry ge;
        ge.launches = ust::g_launches - before;
        ust::g_launches = before;  // counted again at every replay
        e = cudaGraphInstantiate(&ge.exec, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) { set_error(std::string("cudaGraphInstantiate failed: ") + cudaGetErrorString(e)); return 1; }
        it = p->graphs.emplace(key, ge).first;
    }
    UST_CUDA(cudaEventRecord(p->ev_in, user));
    UST_CUDA(cudaStreamWaitEvent(gs, p->ev_in, 0));
    UST_CUDA(cudaGraphLaunch(it->second.exec, gs));
    UST_CUDA(cudaEventRecord(p->ev_out, gs));
    UST_CUDA(cudaStreamWaitEvent(user, p->ev_out, 0));
    ust::g_launches += it->second.launches;
    return 0;
}

// graph keys of the discrete gradient mode: every key below 1000 * nfreq + 1000 gains 50, which no reference key (0, 1, 500,
// 600, 700, 701, 800, 900) reaches
static long long grad_key_offset(const ust_plan* p) { return p->grad_mode == UST_GRAD_DISCRETE ? 50 : 0; }

// kappa != nullptr: lossy evaluation (ust_fwi_loss_grad_lossy), gradient w.r.t. kappa into grad_kappa_dev
template <typename R>
static int fwi_impl(ust_plan* p, const void* slow, const void* rec, int nfreq, const double* freqs, const double* bde,
                    double* loss_dev, void* grad_dev, cudaStream_t st, const void* kappa = nullptr, void* grad_kappa_dev = nullptr) {
    const Geom& g = p->g;
    const bool lossy = kappa != nullptr;
    if (!p->acq_set) { set_error("ust_fwi_loss_grad: ust_plan_set_acquisition has not been called"); return 1; }
    if (!p->U) { set_error("ust_fwi_loss_grad: plan was created with fwi_buffers=0"); return 1; }
    if (p->nt > p->d.max_nrhs) { set_error("ust_fwi_loss_grad: nt exceeds plan max_nrhs"); return 1; }
    UST_TRY(upload_params(p, nfreq, freqs, bde, st));
    // inputs -> plan-owned buffers (stable addresses for the captured graph; the line search reads them again)
    if (slow != p->slow_in) UST_CUDA(cudaMemcpyAsync(p->slow_in, slow, g.N * sizeof(R), cudaMemcpyDeviceToDevice, st));
    if (rec != p->rec_in) UST_CUDA(cudaMemcpyAsync(p->rec_in, rec, (size_t)nfreq * p->nt * p->nelem * sizeof(cx<R>), cudaMemcpyDeviceToDevice, st));
    if (lossy) UST_CUDA(cudaMemcpyAsync(p->kappa_in, kappa, g.N * sizeof(R), cudaMemcpyDeviceToDevice, st));
    const bool has_bde = bde != nullptr;
    // lossless evaluation 0/1, line search 500, Gauss-Newton product 600, lossy evaluation 700/701, lossy line search 800,
    // lossy Gauss-Newton product 900; the discrete gradient mode adds 50 to each (grad_key_offset)
    const long long key = 1000LL * nfreq + (lossy ? 700 : 0) + (has_bde ? 1 : 0) + grad_key_offset(p);
    p->factored_since_eval = true;  // until this evaluation completes, the factors belong to no evaluation
    UST_TRY(run_graphed(p, key, st, [&](cudaStream_t s_) { return fwi_enqueue<R>(p, nfreq, has_bde, s_, lossy); }));
    p->nfreq_cur = nfreq;
    p->factored = true;
    UST_CUDA(cudaMemcpyAsync(loss_dev, p->d_scal, sizeof(double), cudaMemcpyDeviceToDevice, st));
    UST_CUDA(cudaMemcpyAsync(grad_dev, p->grad_out, g.N * sizeof(R), cudaMemcpyDeviceToDevice, st));
    if (lossy) UST_CUDA(cudaMemcpyAsync(grad_kappa_dev, p->grad_kappa_out, g.N * sizeof(R), cudaMemcpyDeviceToDevice, st));
    p->eval_kind = lossy ? ust_plan::EVAL_LOSSY : ust_plan::EVAL_LOSSLESS;
    p->eval_grad_mode = p->grad_mode;
    p->factored_since_eval = false;
    p->factors_lossy = lossy;
    if (p->trace) return dump_update_trace(p, st);
    return 0;
}

// The line search and the Gauss-Newton product run on the factors, forward fields, source estimates and inputs of the last
// evaluation: only when it was of their own kind (the lossless entry points' virtual source assumes a real slowness) and no
// factorisation has replaced its factors since.
static int check_eval(const ust_plan* p, const char* name, bool lossy) {
    const std::string n(name);
    const char* want = lossy ? "ust_fwi_loss_grad_lossy" : "ust_fwi_loss_grad";
    if (!p->U) { set_error(n + ": plan was created with fwi_buffers=0"); return 1; }
    if (!p->factored || p->eval_kind == ust_plan::EVAL_NONE) { set_error(n + ": call " + want + " first"); return 1; }
    const bool last_lossy = p->eval_kind == ust_plan::EVAL_LOSSY;
    if (p->factored_since_eval) {
        set_error(n + ": the factors were replaced (" + (p->factors_lossy ? "ust_factor_lossy" : "ust_factor / ust_solve_helmholtz_host") +
                  ") after the last " + (last_lossy ? "ust_fwi_loss_grad_lossy" : "ust_fwi_loss_grad") + "; call " + want + " again");
        return 1;
    }
    if (p->eval_grad_mode != p->grad_mode) {
        static const char* mode_name[2] = {"UST_GRAD_REFERENCE", "UST_GRAD_DISCRETE"};
        set_error(n + ": the last evaluation ran in gradient mode " + mode_name[p->eval_grad_mode] + " and the plan is now in " +
                  mode_name[p->grad_mode] + " (ust_plan_set_gradient); call " + want + " again");
        return 1;
    }
    if (last_lossy != lossy) {
        set_error(n + (lossy ? ": the last evaluation was lossless (ust_fwi_loss_grad); use the lossless entry point or call "
                               "ust_fwi_loss_grad_lossy first"
                             : ": the last evaluation was lossy (ust_fwi_loss_grad_lossy) and this entry point assumes a real "
                               "slowness; use the lossy entry point or call ust_fwi_loss_grad first"));
        return 1;
    }
    return 0;
}

// sd_kappa != nullptr: the line search of the joint direction [sd, sd_kappa] on a lossy evaluation (ust_ncg_linesearch_lossy)
template <typename R>
static int linesearch_impl(ust_plan* p, const void* sd, const void* sd_kappa, double* out2, cudaStream_t st) {
    const bool lossy = sd_kappa != nullptr;
    UST_TRY(check_eval(p, lossy ? "ust_ncg_linesearch_lossy" : "ust_ncg_linesearch", lossy));
    const size_t bytes = p->g.N * sizeof(R);
    UST_CUDA(cudaMemcpyAsync(p->sd_in, sd, bytes, cudaMemcpyDeviceToDevice, st));
    if (lossy) UST_CUDA(cudaMemcpyAsync(p->vk_in, sd_kappa, bytes, cudaMemcpyDeviceToDevice, st));
    const long long key = 1000LL * p->nfreq_cur + (lossy ? 800 : 500) + grad_key_offset(p);
    UST_TRY(run_graphed(p, key, st, [&](cudaStream_t s_) { return linesearch_enqueue<R>(p, s_, lossy); }));
    UST_CUDA(cudaMemcpyAsync(out2, p->d_scal + 2, 2 * sizeof(double), cudaMemcpyDeviceToDevice, st));
    return 0;
}

// v_kappa != nullptr: the joint product of [v, v_kappa] on a lossy evaluation, its kappa half into hv_kappa (ust_fwi_gn_hvp_lossy)
template <typename R>
static int gn_hvp_impl(ust_plan* p, const void* v, const void* v_kappa, void* hv, void* hv_kappa, double* jv2, void* jv,
                       cudaStream_t st) {
    const bool lossy = v_kappa != nullptr;
    UST_TRY(check_eval(p, lossy ? "ust_fwi_gn_hvp_lossy" : "ust_fwi_gn_hvp", lossy));
    const size_t bytes = p->g.N * sizeof(R);
    UST_CUDA(cudaMemcpyAsync(p->v_in, v, bytes, cudaMemcpyDeviceToDevice, st));
    if (lossy) UST_CUDA(cudaMemcpyAsync(p->vk_in, v_kappa, bytes, cudaMemcpyDeviceToDevice, st));
    const long long key = 1000LL * p->nfreq_cur + (lossy ? 900 : 600) + grad_key_offset(p);
    UST_TRY(run_graphed(p, key, st, [&](cudaStream_t s_) { return gn_hvp_enqueue<R>(p, s_, lossy); }));
    UST_CUDA(cudaMemcpyAsync(hv, p->hv_out, bytes, cudaMemcpyDeviceToDevice, st));
    if (lossy) UST_CUDA(cudaMemcpyAsync(hv_kappa, p->hv_kappa_out, bytes, cudaMemcpyDeviceToDevice, st));
    UST_CUDA(cudaMemcpyAsync(jv2, p->d_scal + 6, sizeof(double), cudaMemcpyDeviceToDevice, st));
    if (jv) UST_CUDA(cudaMemcpyAsync(jv, p->drec, (size_t)p->nfreq_cur * p->nt * p->nm * sizeof(cx<R>), cudaMemcpyDeviceToDevice, st));
    return 0;
}

template <typename R>
static int set_kernel_attrs() {
    UST_CUDA(cudaFuncSetAttribute(gj_pivot_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)std::max(gj_pivot_smem<R>(), sizeof(R) == 4 ? gj_pivot2_smem_bytes : gj_pivot_f64_smem_bytes)));
    // static tiles (38 KB) + the dynamic scratch of the blocked pivot-0 inversion exceed the 48 KB a kernel gets without opting in
    if (sizeof(R) == 4) UST_CUDA(cudaFuncSetAttribute(schur_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gj_pivot2_scratch_bytes));

    UST_CUDA(cudaFuncSetAttribute(gj_rowpanel_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gj_rowpanel_smem<R>()));
    if (sizeof(R) == 4) {
        UST_CUDA(cudaFuncSetAttribute(tc2_sweep_gemm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc2::SMEM_BYTES));
        UST_CUDA(cudaFuncSetAttribute(tc2_sweep_gemm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc2::SMEM_BYTES));
        UST_CUDA(cudaFuncSetAttribute(tc2_gj_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tc2::SMEM_BYTES_H));
        UST_CUDA(cudaFuncSetAttribute(tc2_gj_rowpanel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tc2::SMEM_BYTES_H));
        UST_CUDA(cudaFuncSetAttribute(tc2h_test_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tc2::SMEM_BYTES_H));
        UST_CUDA(cudaFuncSetAttribute(tc2_test_gemm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc2::SMEM_BYTES));
        UST_CUDA(cudaFuncSetAttribute(tc2_test_gemm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc2::SMEM_BYTES));
    }
    return 0;
}

#define DISPATCH(p, fn, ...) ((p)->d.dtype == UST_C64 ? fn<float>(__VA_ARGS__) : fn<double>(__VA_ARGS__))

struct IdtftCache { void* buf = nullptr; size_t cap = 0; cudaEvent_t ev = nullptr; bool used = false; };

template <typename R>
static int idtft_impl(const void* U, int nf, long long npix, const double* freqs, const double* resp, double df, const double* time, int nt,
                      void* out, cudaStream_t st) {
    const double PI = 3.14159265358979323846;
    std::vector<cx<R>> w((size_t)nt * nf);
    for (int t = 0; t < nt; ++t)
        for (int k = 0; k < nf; ++k) {
            const double ph = 2.0 * PI * freqs[k] * time[t], a = df * (resp ? resp[k] : 1.0);
            w[(size_t)t * nf + k] = cx<R>((R)(a * cos(ph)), (R)(a * sin(ph)));
        }
    // weights -> a per-device buffer that is kept between calls (grown on demand, never freed on the hot path); an event
    // orders its reuse behind the previous call's kernel, so nothing here synchronises with the host
    int dev = 0;
    UST_CUDA(cudaGetDevice(&dev));
    static std::mutex mu;
    static std::map<int, IdtftCache> caches;
    std::lock_guard<std::mutex> lock(mu);
    IdtftCache& c = caches[dev];
    const size_t need = w.size() * sizeof(cx<R>);
    if (!c.ev) UST_CUDA(cudaEventCreateWithFlags(&c.ev, cudaEventDisableTiming));
    if (need > c.cap) {
        if (c.buf) { UST_CUDA(cudaEventSynchronize(c.ev)); cudaFree(c.buf); c.buf = nullptr; c.cap = 0; }
        UST_CUDA(cudaMalloc(&c.buf, need));
        c.cap = need;
    } else if (c.used) {
        UST_CUDA(cudaStreamWaitEvent(st, c.ev, 0));
    }
    cx<R>* wd = (cx<R>*)c.buf;
    UST_CUDA(cudaMemcpyAsync(wd, w.data(), need, cudaMemcpyHostToDevice, st));  // pageable source: staged before the call returns
    const size_t smem = (size_t)IDTFT_TT * nf * sizeof(cx<R>);
    if (smem > 48 * 1024) UST_CUDA(cudaFuncSetAttribute(idtft_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    idtft_kernel<R><<<dim3((unsigned)((npix + 255) / 256), (unsigned)cdiv_i(nt, IDTFT_TT)), 256, smem, st>>>((const cx<R>*)U, wd, (cx<R>*)out, npix, nf, nt);
    UST_LAUNCH_CHECK();
    UST_CUDA(cudaEventRecord(c.ev, st));
    c.used = true;
    return 0;
}

// -------------------------------------------------------------------------------------------------
// C ABI
// -------------------------------------------------------------------------------------------------
extern "C" {

const char* ust_last_error(void) { return g_err.c_str(); }
const char* ust_version(void) { return "ustfwi 0.1 (sm_100a)"; }
int ust_idtft(int dtype, const void* U_dev, int nf, long long npix, const double* freqs, const double* resp, double df,
              const double* time, int nt, void* out_dev, void* stream) {
    if (!U_dev || !out_dev || !freqs || !time) { set_error("ust_idtft: null argument"); return 1; }
    if (nf < 1 || nt < 1 || npix < 1) { set_error("ust_idtft: empty problem"); return 1; }
    if ((size_t)IDTFT_TT * nf * (dtype == UST_C64 ? 8 : 16) > 200 * 1024) { set_error("ust_idtft: too many frequencies for one pass (split the stack)"); return 1; }
    if (dtype == UST_C64) return idtft_impl<float>(U_dev, nf, npix, freqs, resp, df, time, nt, out_dev, (cudaStream_t)stream);
    if (dtype == UST_C128) return idtft_impl<double>(U_dev, nf, npix, freqs, resp, df, time, nt, out_dev, (cudaStream_t)stream);
    set_error("ust_idtft: unknown dtype");
    return 1;
}

int ust_pack_f64_as_f32x2(const double* in_dev, float* out_dev, int n, void* stream) {
    if (!in_dev || !out_dev || n < 1) { set_error("ust_pack_f64_as_f32x2: bad arguments"); return 1; }
    pack_f32x2_kernel<<<cdiv_i(n, 128), 128, 0, (cudaStream_t)stream>>>(in_dev, out_dev, n);
    UST_LAUNCH_CHECK();
    return 0;
}

long long ust_launch_count(void) { return g_launches; }
void ust_launch_count_reset(void) { g_launches = 0; }

int ust_plan_create(const ust_plan_desc* d, ust_plan** out) {
    if (!d || !out) { set_error("ust_plan_create: null argument"); return 1; }
    if (d->nx < 5 || d->ny < 5) { set_error("ust_plan_create: grid must be at least 5x5"); return 1; }
    if (d->dtype != UST_C64 && d->dtype != UST_C128) { set_error("ust_plan_create: bad dtype"); return 1; }
    if (d->max_freq < 1 || d->max_nrhs < 1) { set_error("ust_plan_create: max_freq and max_nrhs must be >= 1"); return 1; }
    if (d->engine != UST_ENGINE_AUTO && d->engine != UST_ENGINE_SIMT && d->engine != UST_ENGINE_TC2) { set_error("ust_plan_create: unknown engine (AUTO, SIMT or TC2; the first tcgen05 engine, value 2, was removed)"); return 1; }
    if (d->engine == UST_ENGINE_TC2 && d->dtype != UST_C64) { set_error("ust_plan_create: the tensor-core engine is complex64 only (no FP64 tcgen05 kind)"); return 1; }
    int ndev = 0;
    UST_CUDA(cudaGetDeviceCount(&ndev));
    if (d->device < 0 || d->device >= ndev) { set_error("ust_plan_create: no such CUDA device"); return 1; }
    UST_CUDA(cudaSetDevice(d->device));
    ust_plan* p = new ust_plan();
    p->d = *d;
    Geom& g = p->g;
    g.Nx = d->nx; g.Ny = d->ny; g.nI = d->nx - 2; g.M = d->ny - 2;
    g.nP = ((g.nI + GJ_NB - 1) / GJ_NB) * GJ_NB;
    g.mid = g.M / 2;
    g.N = (long long)d->nx * d->ny;
    // AUTO = the TMA-fed tcgen05 engine for complex64 (FP32-accurate products, leading terms accumulated in FP32 registers);
    // complex128 has no tensor-core path (no FP64 tcgen05 kind) and runs on the FP64 FMA engine.
    p->use_tc2 = d->dtype == UST_C64 && (d->engine == UST_ENGINE_TC2 || d->engine == UST_ENGINE_AUTO);
    if (const char* e = getenv("UST_TC2_BIAS_FIX")) p->bias_fix = (float)atof(e);
    if (const char* e = getenv("UST_TC2_GJ_DRAIN")) p->gj_drain = atoi(e);
    if (const char* e = getenv("UST_TC2_SWEEP_DRAIN")) p->sweep_drain = atoi(e);
    if (const char* e = getenv("UST_TC2_PREFETCH")) p->prefetch_cin = atoi(e);
    if (const char* e = getenv("UST_GROUPS")) p->ngroups = std::max(1, std::min(atoi(e), (int)ust_plan::MAX_GROUPS));
    p->t_ring = p->use_tc2;  // the TMA-fed sweeps read the bf16 planes Tp: FP32 T is only the Schur update's previous row
    p->rsz = d->dtype == UST_C64 ? 4 : 8;
    p->csz = 2 * p->rsz;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, d->device) == cudaSuccess) p->num_sms = prop.multiProcessorCount;
    const size_t bs = (size_t)g.nP * g.nP * p->csz;
    int rc = 0;
    rc |= dev_alloc(p, &p->exn, g.Nx * p->csz);
    rc |= dev_alloc(p, &p->rexh, g.Nx * p->csz);
    rc |= dev_alloc(p, &p->eyn, g.Ny * p->csz);
    rc |= dev_alloc(p, &p->reyh, g.Ny * p->csz);
    rc |= dev_alloc(p, (void**)&p->d_vminmax, 2 * sizeof(double));
    rc |= dev_alloc(p, (void**)&p->d_freqs, d->max_freq * sizeof(double));
    rc |= dev_alloc(p, (void**)&p->d_bde, 3 * d->max_freq * sizeof(double));
    rc |= dev_alloc(p, (void**)&p->d_scal, 8 * sizeof(double));
    rc |= dev_alloc(p, (void**)&p->d_status, sizeof(int));
    rc |= dev_alloc(p, (void**)&p->d_invv2, g.N * sizeof(double));
    rc |= dev_alloc(p, (void**)&p->d_sig2, 2 * g.N * sizeof(double));
    rc |= dev_alloc(p, &p->planes, (size_t)d->max_freq * 9 * g.N * p->csz);
    rc |= dev_alloc(p, &p->T, (size_t)d->max_freq * (p->t_ring ? 4 : g.M) * bs);
    if (!(d->dtype == UST_C64 && (d->engine == UST_ENGINE_TC2 || d->engine == UST_ENGINE_AUTO))) rc |= dev_alloc(p, &p->scratch, (size_t)2 * d->max_freq * bs);  // TC2 inverts in place
    rc |= dev_alloc(p, &p->pbuf, (size_t)2 * d->max_freq * GJ_NB * GJ_NB * p->csz);
    rc |= dev_alloc(p, &p->W, (size_t)2 * d->max_freq * g.nP * d->max_nrhs * p->csz);
    rc |= dev_alloc(p, &p->vel, g.N * p->rsz);
    if (!rc && p->use_tc2) {
        p->kpad = ((g.nI + tc2::KC - 1) / tc2::KC) * tc2::KC;
        p->wp_stride = tc2::bplanes_elems(p->kpad, d->max_nrhs);
        const size_t tp_bytes = (size_t)d->max_freq * g.M * tc2::NPL_A * g.nP * g.nP * sizeof(uint16_t);
        const size_t wp_bytes = (size_t)2 * d->max_freq * p->wp_stride * sizeof(uint16_t);
        rc |= dev_alloc(p, (void**)&p->Tp, tp_bytes);
        rc |= dev_alloc(p, (void**)&p->Wp, wp_bytes);
        if (!rc && cudaMemset(p->Wp, 0, wp_bytes) != cudaSuccess) rc = 1;
        if (!rc) rc = tc2::make_aplane_maps(p->Tp, g.nP, (long long)d->max_freq * g.M, p->amaps);
        p->rp_stride = tc2::bplanes_elems(GJ_NB, g.nP);
        const size_t nbmax = (size_t)2 * d->max_freq;
        rc |= dev_alloc(p, (void**)&p->Rp, nbmax * p->rp_stride * sizeof(uint16_t));
        rc |= dev_alloc(p, (void**)&p->Xp, 2 * nbmax * p->rp_stride * sizeof(uint16_t));
        rc |= dev_alloc(p, (void**)&p->Cp, 2 * nbmax * tc2::NPL_A * g.nP * GJ_NB * sizeof(uint16_t));
        rc |= dev_alloc(p, (void**)&p->Pp, nbmax * tc2::NPL_A * GJ_NB * GJ_NB * sizeof(uint16_t));
        rc |= dev_alloc(p, &p->snap, nbmax * GJ_NB * GJ_NB * p->csz);
        if (!rc) rc = tc2::make_aplane_maps(p->Cp, g.nP, GJ_NB, (long long)(2 * nbmax), p->cmaps);
        if (!rc) rc = tc2::make_aplane_maps(p->Pp, GJ_NB, GJ_NB, (long long)nbmax, p->pmaps);
    }
    if (d->fwi_buffers) {
        rc |= dev_alloc(p, &p->U, (size_t)d->max_freq * g.N * d->max_nrhs * p->csz);
        rc |= dev_alloc(p, &p->Lam, (size_t)d->max_freq * g.N * d->max_nrhs * p->csz);
        rc |= dev_alloc(p, &p->src_est, (size_t)d->max_freq * d->max_nrhs * p->csz);
        rc |= dev_alloc(p, &p->slow_in, g.N * p->rsz);
        rc |= dev_alloc(p, &p->grad_out, g.N * p->rsz);
        rc |= dev_alloc(p, &p->sd_in, g.N * p->rsz);
        rc |= dev_alloc(p, &p->v_in, g.N * p->rsz);
        rc |= dev_alloc(p, &p->hv_out, g.N * p->rsz);
        rc |= dev_alloc(p, &p->kappa_in, g.N * p->rsz);
        rc |= dev_alloc(p, &p->grad_kappa_out, g.N * p->rsz);
        rc |= dev_alloc(p, &p->vk_in, g.N * p->rsz);
        rc |= dev_alloc(p, &p->hv_kappa_out, g.N * p->rsz);
    }
    if (const char* e = getenv("UST_NO_GRAPHS")) p->use_graphs = atoi(e) == 0;
    if (const char* e = getenv("UST_NO_PDL")) ust::g_use_pdl = atoi(e) == 0;
    if (!rc && (cudaEventCreateWithFlags(&p->ev_in, cudaEventDisableTiming) != cudaSuccess ||
                cudaEventCreateWithFlags(&p->ev_out, cudaEventDisableTiming) != cudaSuccess)) {
        set_error("ust_plan_create: event creation failed");
        rc = 1;
    }
    if (!rc && cudaMallocHost((void**)&p->h_stage, 4 * d->max_freq * sizeof(double)) != cudaSuccess) {
        set_error("ust_plan_create: cudaMallocHost failed");
        rc = 1;
    }
    if (!rc && cudaStreamCreateWithFlags(&p->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
        set_error("ust_plan_create: cudaStreamCreate failed");
        rc = 1;
    }
    if (!rc && cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming) != cudaSuccess) rc = 1;
    for (int i = 1; i < ust_plan::MAX_GROUPS && !rc; ++i)
        if (cudaStreamCreateWithFlags(&p->side[i], cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&p->ev_join[i], cudaEventDisableTiming) != cudaSuccess) {
            set_error("ust_plan_create: group stream / event creation failed");
            rc = 1;
        }
    if (!rc && d->dtype == UST_C128) {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);  // hi = numerically lowest = highest priority
        for (int i = 0; i < ust_plan::MAX_GROUPS && !rc; ++i)
            if (cudaStreamCreateWithPriority(&p->pivst[i], cudaStreamNonBlocking, hi) != cudaSuccess ||
                cudaEventCreateWithFlags(&p->ev_upd[i], cudaEventDisableTiming) != cudaSuccess ||
                cudaEventCreateWithFlags(&p->ev_piv[i][0], cudaEventDisableTiming) != cudaSuccess ||
                cudaEventCreateWithFlags(&p->ev_piv[i][1], cudaEventDisableTiming) != cudaSuccess) {
                set_error("ust_plan_create: pivot stream / event creation failed");
                rc = 1;
            }
    }
    if (const char* e = getenv("UST_NO_LOOKAHEAD")) p->lookahead = atoi(e) == 0;
    if (const char* e = getenv("UST_PDL_MIN_BATCH")) p->pdl_min_batch = atoi(e);
    if (const char* e = getenv("UST_KSPLIT")) p->ksplit_ok = atoi(e);
    if (const char* e = getenv("UST_TC2_TRACE_UPDATE")) {
        if (sscanf(e, "%d,%d", &p->trace_step, &p->trace_k) == 2 && cudaMalloc((void**)&p->trace, 19 * 1024 * sizeof(unsigned long long)) == cudaSuccess)
            cudaMemset(p->trace, 0, 19 * 1024 * sizeof(unsigned long long));
    }
    if (!rc) rc = (d->dtype == UST_C64) ? set_kernel_attrs<float>() : set_kernel_attrs<double>();
    if (!rc && cudaMemset(p->d_status, 0, sizeof(int)) != cudaSuccess) rc = 1;
    if (rc) {
        std::string keep = g_err;
        ust_plan_destroy(p);
        set_error(keep.empty() ? "ust_plan_create: allocation failed" : keep);
        return 1;
    }
    *out = p;
    return 0;
}

int ust_plan_destroy(ust_plan* p) {
    if (!p) return 0;
    cudaSetDevice(p->d.device);
    cudaDeviceSynchronize();
    void* ptrs[] = {p->exn, p->rexh, p->eyn, p->reyh, p->d_vminmax, p->d_freqs, p->d_bde, p->d_scal, p->d_status, p->d_invv2, p->d_sig2, p->planes,
                    p->T, p->scratch, p->W, p->pbuf, p->Tp, p->Wp, p->Rp, p->Cp, p->Xp, p->Pp, p->snap, p->vel, p->U, p->Lam, p->src_est, p->Xh, p->src_lin, p->rx_lin, p->mask, p->rx_next,
                    p->slow_h2d, p->rec_h2d, p->grad_d2h, p->kappa_h2d, p->grad_kappa_d2h};
    for (void* q : ptrs)
        if (q) cudaFree(q);
    drop_graphs(p);
    for (void* q : {p->slow_in, p->rec_in, p->grad_out, p->sd_in, p->v_in, p->hv_out, p->drec, p->kappa_in, p->grad_kappa_out,
                     p->vk_in, p->hv_kappa_out})
        if (q) cudaFree(q);
    if (p->ev_in) cudaEventDestroy(p->ev_in);
    if (p->ev_out) cudaEventDestroy(p->ev_out);
    if (p->h_stage) cudaFreeHost(p->h_stage);
    if (p->own_stream) cudaStreamDestroy(p->own_stream);
    if (p->ev_fork) cudaEventDestroy(p->ev_fork);
    for (int i = 0; i < ust_plan::MAX_GROUPS; ++i) {
        if (p->side[i]) cudaStreamDestroy(p->side[i]);
        if (p->ev_join[i]) cudaEventDestroy(p->ev_join[i]);
        if (p->pivst[i]) cudaStreamDestroy(p->pivst[i]);
        if (p->ev_upd[i]) cudaEventDestroy(p->ev_upd[i]);
        for (int j = 0; j < 2; ++j)
            if (p->ev_piv[i][j]) cudaEventDestroy(p->ev_piv[i][j]);
    }

    for (cudaEvent_t e : p->ev) cudaEventDestroy(e);
    delete p;
    return 0;
}

size_t ust_plan_device_bytes(const ust_plan* p) { return p ? p->bytes : 0; }

int ust_plan_set_groups(ust_plan* p, int ngroups) {
    UST_TRY(check_plan(p));
    if (ngroups < 1 || ngroups > ust_plan::MAX_GROUPS) { set_error("ust_plan_set_groups: 1 <= ngroups <= 8"); return 1; }
    if (ngroups == p->ngroups) return 0;
    UST_CUDA(cudaSetDevice(p->d.device));
    UST_CUDA(cudaDeviceSynchronize());
    drop_graphs(p);  // the captured graphs bake the fork / join structure
    p->ngroups = ngroups;
    return 0;
}

int ust_plan_set_gradient(ust_plan* p, int mode) {
    UST_TRY(check_plan(p));
    if (mode != UST_GRAD_REFERENCE && mode != UST_GRAD_DISCRETE) {
        set_error("ust_plan_set_gradient: mode must be UST_GRAD_REFERENCE (0) or UST_GRAD_DISCRETE (1)");
        return 1;
    }
    p->grad_mode = mode;  // the graphs of both modes stay: their keys differ (grad_key_offset)
    return 0;
}

int ust_plan_set_grid(ust_plan* p, const double* x, const double* y, double a0, double L) {
    UST_TRY(check_plan(p));
    if (!x || !y || !(L > 0)) { set_error("ust_plan_set_grid: bad arguments"); return 1; }
    UST_CUDA(cudaSetDevice(p->d.device));
    UST_CUDA(cudaDeviceSynchronize());
    drop_graphs(p);
    return p->d.dtype == UST_C64 ? set_grid_impl<float>(p, x, y, a0, L) : set_grid_impl<double>(p, x, y, a0, L);
}

int ust_plan_set_acquisition(ust_plan* p, int nt, const int32_t* src_lin, int nelem, const int32_t* rx_lin, int nm,
                             const int32_t* mask) {
    UST_TRY(check_plan(p));
    if (nt < 1 || nelem < 1 || nm < 1 || !src_lin || !rx_lin || !mask) { set_error("ust_plan_set_acquisition: bad arguments"); return 1; }
    const Geom& g = p->g;
    auto interior = [&](int lin) {
        int y = lin / g.Nx, x = lin % g.Nx;
        return lin >= 0 && lin < g.N && x > 0 && y > 0 && x < g.Nx - 1 && y < g.Ny - 1;
    };
    for (int i = 0; i < nt; ++i)
        if (!interior(src_lin[i])) { set_error("ust_plan_set_acquisition: a source lies on or outside the Dirichlet ring"); return 1; }
    for (int i = 0; i < nelem; ++i)
        if (!interior(rx_lin[i])) { set_error("ust_plan_set_acquisition: a receiver lies on or outside the Dirichlet ring"); return 1; }
    for (long long i = 0; i < (long long)nt * nm; ++i)
        if (mask[i] < 0 || mask[i] >= nelem) { set_error("ust_plan_set_acquisition: mask index out of range"); return 1; }
    UST_CUDA(cudaSetDevice(p->d.device));
    UST_CUDA(cudaDeviceSynchronize());
    drop_graphs(p);
    p->eval_kind = ust_plan::EVAL_NONE;
    for (int** q : {&p->src_lin, &p->rx_lin, &p->mask, &p->rx_next})
        if (*q) { cudaFree(*q); *q = nullptr; }
    if (p->rec_in) { cudaFree(p->rec_in); p->rec_in = nullptr; }
    if (p->rec_h2d) { cudaFree(p->rec_h2d); p->rec_h2d = nullptr; }  // sized by nt * nelem: regrown by the next host call
    if (p->drec) { cudaFree(p->drec); p->drec = nullptr; }
    if (p->d.fwi_buffers) UST_CUDA(cudaMalloc(&p->rec_in, (size_t)p->d.max_freq * nt * nelem * p->csz));
    if (p->d.fwi_buffers) UST_CUDA(cudaMalloc(&p->drec, (size_t)p->d.max_freq * nt * nm * p->csz));
    UST_CUDA(cudaMalloc((void**)&p->src_lin, nt * sizeof(int)));
    UST_CUDA(cudaMalloc((void**)&p->rx_lin, nelem * sizeof(int)));
    UST_CUDA(cudaMalloc((void**)&p->mask, (size_t)nt * nm * sizeof(int)));
    UST_CUDA(cudaMemcpy(p->src_lin, src_lin, nt * sizeof(int), cudaMemcpyHostToDevice));
    UST_CUDA(cudaMemcpy(p->rx_lin, rx_lin, nelem * sizeof(int), cudaMemcpyHostToDevice));
    UST_CUDA(cudaMemcpy(p->mask, mask, (size_t)nt * nm * sizeof(int), cudaMemcpyHostToDevice));
    // Kept receivers of one transmitter that snap to the same node: the adjoint source there is the sum of their residuals,
    // added in mask order by the first of them (receiver_kernel, gn_scatter_kernel).  Entry j holds the next such receiver
    // (nm: none), stored as -1 - next when j is not the first on its node.
    {
        std::vector<int> next((size_t)nt * nm, nm);
        std::unordered_map<int, int> last;  // node -> last kept receiver seen on it
        for (int t = 0; t < nt; ++t) {
            int* nx = next.data() + (size_t)t * nm;
            const int* mk = mask + (size_t)t * nm;
            last.clear();
            for (int j = 0; j < nm; ++j) {
                auto it = last.find(rx_lin[mk[j]]);
                if (it == last.end()) { last.emplace(rx_lin[mk[j]], j); continue; }
                const int i = it->second;  // previous receiver on this node: link it to j, keep its own first / not-first sign
                nx[i] = nx[i] >= 0 ? j : -1 - j;
                nx[j] = -1 - nm;
                it->second = j;
            }
        }
        UST_CUDA(cudaMalloc((void**)&p->rx_next, next.size() * sizeof(int)));
        UST_CUDA(cudaMemcpy(p->rx_next, next.data(), next.size() * sizeof(int), cudaMemcpyHostToDevice));
    }
    p->nt = nt; p->nelem = nelem; p->nm = nm; p->acq_set = true;
    p->onehot_ok = cdiv_i(nt, 128) <= 8;
    for (int i = 0; i < 8; ++i) { p->first_row[i] = 32767; p->last_row[i] = -1; }
    if (p->onehot_ok)
        for (int i = 0; i < nt; ++i) {
            const short r = (short)(src_lin[i] / g.Nx - 1);  // interior block row of the source node
            short& lo = p->first_row[i / 128]; short& hi = p->last_row[i / 128];
            lo = std::min(lo, r); hi = std::max(hi, r);
        }
    return 0;
}

int ust_factor(ust_plan* p, const void* vel_dev, int nfreq, const double* freqs, const double* bde, void* stream) {
    UST_TRY(check_plan(p));
    if (!vel_dev || !freqs) { set_error("ust_factor: null argument"); return 1; }
    UST_CUDA(cudaSetDevice(p->d.device));
    const int rc = DISPATCH(p, factor_impl, p, vel_dev, nfreq, freqs, bde, (cudaStream_t)stream);
    if (!rc && p->trace) return dump_update_trace(p, (cudaStream_t)stream);
    return rc;
}

int ust_factor_lossy(ust_plan* p, const void* vel_dev, const void* kappa_dev, int nfreq, const double* freqs, const double* bde, void* stream) {
    UST_TRY(check_plan(p));
    if (!vel_dev || !kappa_dev || !freqs) { set_error("ust_factor_lossy: null argument (kappa_dev is required)"); return 1; }
    UST_CUDA(cudaSetDevice(p->d.device));
    return DISPATCH(p, factor_impl, p, vel_dev, nfreq, freqs, bde, (cudaStream_t)stream, kappa_dev);
}

int ust_solve(ust_plan* p, int ifreq, void* X, int nrhs, int adjoint, void* stream) {
    UST_TRY(check_plan(p));
    if (!X) { set_error("ust_solve: null argument"); return 1; }
    UST_CUDA(cudaSetDevice(p->d.device));
    return DISPATCH(p, solve_impl, p, ifreq, X, nrhs, adjoint, (cudaStream_t)stream);
}

int ust_solve_helmholtz_host(ust_plan* p, const void* vel_host, const void* src_host, void* out_host, int nrhs, double f,
                             const double* bde, int adjoint, int refactor) {
    UST_TRY(check_plan(p));
    if (!src_host || !out_host) { set_error("ust_solve_helmholtz_host: null argument"); return 1; }
    if (nrhs < 1 || nrhs > p->d.max_nrhs) { set_error("ust_solve_helmholtz_host: nrhs exceeds plan max_nrhs"); return 1; }
    UST_CUDA(cudaSetDevice(p->d.device));
    const Geom& g = p->g;
    cudaStream_t st = p->own_stream;
    if (!p->Xh) UST_TRY(dev_alloc(p, &p->Xh, (size_t)g.N * p->d.max_nrhs * p->csz));
    if (refactor || !p->factored) {
        if (!vel_host) { set_error("ust_solve_helmholtz_host: vel required to factorise"); return 1; }
        UST_CUDA(cudaMemcpyAsync(p->vel, vel_host, g.N * p->rsz, cudaMemcpyHostToDevice, st));
        UST_TRY(DISPATCH(p, factor_impl, p, p->vel, 1, &f, bde, st));
    }
    const size_t bytes = (size_t)g.N * nrhs * p->csz;
    UST_CUDA(cudaMemcpyAsync(p->Xh, src_host, bytes, cudaMemcpyHostToDevice, st));
    UST_TRY(DISPATCH(p, solve_impl, p, 0, p->Xh, nrhs, adjoint, st));
    UST_CUDA(cudaMemcpyAsync(out_host, p->Xh, bytes, cudaMemcpyDeviceToHost, st));
    int status = 0;
    UST_CUDA(cudaMemcpyAsync(&status, p->d_status, sizeof(int), cudaMemcpyDeviceToHost, st));
    UST_CUDA(cudaStreamSynchronize(st));
    if (status) { set_error("ust_solve_helmholtz_host: a block inversion met a zero / non-finite pivot (singular operator)"); return 2; }
    return 0;
}

int ust_fwi_loss_grad(ust_plan* p, const void* slow, const void* rec, int nfreq, const double* freqs, const double* bde,
                      double* loss_dev, void* grad_dev, void* stream) {
    UST_TRY(check_plan(p));
    if (!slow || !rec || !freqs || !loss_dev || !grad_dev) { set_error("ust_fwi_loss_grad: null argument"); return 1; }
    UST_CUDA(cudaSetDevice(p->d.device));
    return DISPATCH(p, fwi_impl, p, slow, rec, nfreq, freqs, bde, loss_dev, grad_dev, (cudaStream_t)stream);
}

// host twins of ust_fwi_loss_grad (kappa_host == nullptr) and ust_fwi_loss_grad_lossy: staging buffers allocated on first use
static int fwi_host(ust_plan* p, const char* name, const void* slow_host, const void* kappa_host, const void* rec_host, int nfreq,
                    const double* freqs, const double* bde, double* loss_host, void* grad_host, void* grad_kappa_host) {
    if (!p->acq_set) { set_error(std::string(name) + ": ust_plan_set_acquisition has not been called"); return 1; }
    UST_CUDA(cudaSetDevice(p->d.device));
    const Geom& g = p->g;
    cudaStream_t st = p->own_stream;
    if (nfreq < 1 || nfreq > p->d.max_freq) { set_error(std::string(name) + ": nfreq out of range"); return 1; }
    const size_t rec_bytes = (size_t)p->d.max_freq * p->nt * p->nelem * p->csz;
    if (!p->slow_h2d) UST_TRY(dev_alloc(p, &p->slow_h2d, g.N * p->rsz));
    if (!p->grad_d2h) UST_TRY(dev_alloc(p, &p->grad_d2h, g.N * p->rsz));
    if (!p->rec_h2d) UST_CUDA(cudaMalloc(&p->rec_h2d, rec_bytes));
    if (kappa_host && !p->kappa_h2d) UST_TRY(dev_alloc(p, &p->kappa_h2d, g.N * p->rsz));
    if (kappa_host && !p->grad_kappa_d2h) UST_TRY(dev_alloc(p, &p->grad_kappa_d2h, g.N * p->rsz));
    UST_CUDA(cudaMemcpyAsync(p->slow_h2d, slow_host, g.N * p->rsz, cudaMemcpyHostToDevice, st));
    UST_CUDA(cudaMemcpyAsync(p->rec_h2d, rec_host, (size_t)nfreq * p->nt * p->nelem * p->csz, cudaMemcpyHostToDevice, st));
    if (kappa_host) UST_CUDA(cudaMemcpyAsync(p->kappa_h2d, kappa_host, g.N * p->rsz, cudaMemcpyHostToDevice, st));
    UST_TRY(DISPATCH(p, fwi_impl, p, p->slow_h2d, p->rec_h2d, nfreq, freqs, bde, p->d_scal, p->grad_d2h, st,
                     kappa_host ? p->kappa_h2d : nullptr, p->grad_kappa_d2h));
    UST_CUDA(cudaMemcpyAsync(loss_host, p->d_scal, sizeof(double), cudaMemcpyDeviceToHost, st));
    UST_CUDA(cudaMemcpyAsync(grad_host, p->grad_d2h, g.N * p->rsz, cudaMemcpyDeviceToHost, st));
    if (kappa_host) UST_CUDA(cudaMemcpyAsync(grad_kappa_host, p->grad_kappa_d2h, g.N * p->rsz, cudaMemcpyDeviceToHost, st));
    int status = 0;
    UST_CUDA(cudaMemcpyAsync(&status, p->d_status, sizeof(int), cudaMemcpyDeviceToHost, st));
    UST_CUDA(cudaStreamSynchronize(st));
    if (status) {  // SciPy's analogue is MatrixRankWarning + NaN output; here it is an error, never a silent garbage gradient
        set_error(std::string(name) + ": a block inversion met a zero / non-finite pivot (singular or ill-posed operator for this model and frequency)");
        return 2;
    }
    return 0;
}

int ust_fwi_loss_grad_host(ust_plan* p, const void* slow_host, const void* rec_host, int nfreq, const double* freqs,
                           const double* bde, double* loss_host, void* grad_host) {
    UST_TRY(check_plan(p));
    if (!slow_host || !rec_host || !freqs || !loss_host || !grad_host) { set_error("ust_fwi_loss_grad_host: null argument"); return 1; }
    return fwi_host(p, "ust_fwi_loss_grad_host", slow_host, nullptr, rec_host, nfreq, freqs, bde, loss_host, grad_host, nullptr);
}

int ust_fwi_loss_grad_lossy(ust_plan* p, const void* slow, const void* kappa, const void* rec, int nfreq, const double* freqs,
                            const double* bde, double* loss_dev, void* grad_s_dev, void* grad_kappa_dev, void* stream) {
    UST_TRY(check_plan(p));
    if (!slow || !kappa || !rec || !freqs || !loss_dev || !grad_s_dev || !grad_kappa_dev) {
        set_error("ust_fwi_loss_grad_lossy: null argument (kappa_dev is required)");
        return 1;
    }
    UST_CUDA(cudaSetDevice(p->d.device));
    return DISPATCH(p, fwi_impl, p, slow, rec, nfreq, freqs, bde, loss_dev, grad_s_dev, (cudaStream_t)stream, kappa, grad_kappa_dev);
}

int ust_fwi_loss_grad_lossy_host(ust_plan* p, const void* slow_host, const void* kappa_host, const void* rec_host, int nfreq,
                                 const double* freqs, const double* bde, double* loss_host, void* grad_s_host, void* grad_kappa_host) {
    UST_TRY(check_plan(p));
    if (!slow_host || !kappa_host || !rec_host || !freqs || !loss_host || !grad_s_host || !grad_kappa_host) {
        set_error("ust_fwi_loss_grad_lossy_host: null argument (kappa_host is required)");
        return 1;
    }
    return fwi_host(p, "ust_fwi_loss_grad_lossy_host", slow_host, kappa_host, rec_host, nfreq, freqs, bde, loss_host, grad_s_host,
                    grad_kappa_host);
}

int ust_ncg_linesearch(ust_plan* p, const void* sd_dev, double* out2_dev, void* stream) {
    UST_TRY(check_plan(p));
    if (!sd_dev || !out2_dev) { set_error("ust_ncg_linesearch: null argument"); return 1; }
    UST_CUDA(cudaSetDevice(p->d.device));
    return DISPATCH(p, linesearch_impl, p, sd_dev, nullptr, out2_dev, (cudaStream_t)stream);
}

int ust_fwi_gn_hvp(ust_plan* p, const void* v_dev, void* hv_dev, double* jv2_dev, void* jv_dev, void* stream) {
    UST_TRY(check_plan(p));
    if (!v_dev || !hv_dev || !jv2_dev) { set_error("ust_fwi_gn_hvp: null argument"); return 1; }
    UST_CUDA(cudaSetDevice(p->d.device));
    return DISPATCH(p, gn_hvp_impl, p, v_dev, nullptr, hv_dev, nullptr, jv2_dev, jv_dev, (cudaStream_t)stream);
}

int ust_ncg_linesearch_lossy(ust_plan* p, const void* sd_s_dev, const void* sd_kappa_dev, double* out2_dev, void* stream) {
    UST_TRY(check_plan(p));
    if (!sd_s_dev || !sd_kappa_dev || !out2_dev) {
        set_error("ust_ncg_linesearch_lossy: null argument (sd_kappa_dev is required)");
        return 1;
    }
    UST_CUDA(cudaSetDevice(p->d.device));
    return DISPATCH(p, linesearch_impl, p, sd_s_dev, sd_kappa_dev, out2_dev, (cudaStream_t)stream);
}

int ust_fwi_gn_hvp_lossy(ust_plan* p, const void* v_s_dev, const void* v_kappa_dev, void* hv_s_dev, void* hv_kappa_dev,
                         double* jv2_dev, void* jv_dev, void* stream) {
    UST_TRY(check_plan(p));
    if (!v_s_dev || !v_kappa_dev || !hv_s_dev || !hv_kappa_dev || !jv2_dev) {
        set_error("ust_fwi_gn_hvp_lossy: null argument (v_kappa_dev and hv_kappa_dev are required)");
        return 1;
    }
    UST_CUDA(cudaSetDevice(p->d.device));
    return DISPATCH(p, gn_hvp_impl, p, v_s_dev, v_kappa_dev, hv_s_dev, hv_kappa_dev, jv2_dev, jv_dev, (cudaStream_t)stream);
}

int ust_get_bde(ust_plan* p, double* out) {
    UST_TRY(check_plan(p));
    UST_CUDA(cudaSetDevice(p->d.device));
    UST_CUDA(cudaDeviceSynchronize());
    UST_CUDA(cudaMemcpy(out, p->d_bde, 3 * p->d.max_freq * sizeof(double), cudaMemcpyDeviceToHost));
    return 0;
}

int ust_get_planes(ust_plan* p, int ifreq, void* out_dev, void* stream) {
    UST_TRY(check_plan(p));
    if (ifreq < 0 || ifreq >= p->d.max_freq) { set_error("ust_get_planes: ifreq out of range"); return 1; }
    UST_CUDA(cudaSetDevice(p->d.device));
    const size_t bytes = (size_t)9 * p->g.N * p->csz;
    UST_CUDA(cudaMemcpyAsync(out_dev, (const char*)p->planes + (size_t)ifreq * bytes, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return 0;
}

int ust_get_src_est(ust_plan* p, int ifreq, void* out_host) {
    UST_TRY(check_plan(p));
    if (!p->src_est || ifreq < 0 || ifreq >= p->d.max_freq) { set_error("ust_get_src_est: unavailable"); return 1; }
    UST_CUDA(cudaSetDevice(p->d.device));
    UST_CUDA(cudaDeviceSynchronize());
    UST_CUDA(cudaMemcpy(out_host, (const char*)p->src_est + (size_t)ifreq * p->nt * p->csz, p->nt * p->csz, cudaMemcpyDeviceToHost));
    return 0;
}

int ust_residual_onehot(ust_plan* p, int ifreq, int t, double* out2_host) {
    UST_TRY(check_plan(p));
    if (p->eval_kind == ust_plan::EVAL_NONE || !p->U) { set_error("ust_residual_onehot: call ust_fwi_loss_grad first"); return 1; }
    if (ifreq < 0 || ifreq >= p->nfreq_cur || t < 0 || t >= p->nt || !out2_host) { set_error("ust_residual_onehot: bad arguments"); return 1; }
    UST_CUDA(cudaSetDevice(p->d.device));
    UST_CUDA(cudaDeviceSynchronize());
    const Geom& g = p->g;
    std::vector<int> src(p->nt);
    UST_CUDA(cudaMemcpy(src.data(), p->src_lin, p->nt * sizeof(int), cudaMemcpyDeviceToHost));
    double* acc = p->d_scal + 4;
    UST_CUDA(cudaMemset(acc, 0, 2 * sizeof(double)));
    const unsigned blocks = (unsigned)((g.N + 255) / 256);
    const size_t uoff = (size_t)ifreq * g.N * p->nt, poff = (size_t)ifreq * 9 * g.N;
    if (p->d.dtype == UST_C64)
        residual_onehot_kernel<float><<<blocks, 256>>>(g, (const cx<float>*)p->planes + poff, (const cx<float>*)p->U + uoff, p->nt, t, src[t], acc);
    else
        residual_onehot_kernel<double><<<blocks, 256>>>(g, (const cx<double>*)p->planes + poff, (const cx<double>*)p->U + uoff, p->nt, t, src[t], acc);
    UST_LAUNCH_CHECK();
    double h[2];
    UST_CUDA(cudaMemcpy(h, acc, sizeof(h), cudaMemcpyDeviceToHost));
    out2_host[0] = sqrt(h[0]);
    out2_host[1] = sqrt(h[1]);
    return 0;
}

void* ust_get_wavefield(ust_plan* p, int ifreq) {
    if (!p || !p->U || ifreq < 0 || ifreq >= p->d.max_freq) return nullptr;
    return (char*)p->U + (size_t)ifreq * p->g.N * p->nt * p->csz;
}

void* ust_get_adjoint_wavefield(ust_plan* p, int ifreq) {
    if (!p || !p->Lam || ifreq < 0 || ifreq >= p->d.max_freq) return nullptr;
    return (char*)p->Lam + (size_t)ifreq * p->g.N * p->nt * p->csz;
}

int ust_test_cgemm(int engine, int ta, int M, int N, int K, const void* A, int lda, const void* B, int ldb, const void* Cin,
                   int ldcin, void* Cout, int ldc, float sgn, int mask_lo, int mask_hi, int skip_lo, int skip_hi, void* stream) {
    static bool attrs = false;
    if (!attrs) { UST_TRY(set_kernel_attrs<float>()); attrs = true; }
    GemmTile<float> t;
    t.A = (const cx<float>*)A; t.lda = lda; t.B = (const cx<float>*)B; t.ldb = ldb;
    t.Cin = (const cx<float>*)Cin; t.ldcin = ldcin; t.Cout = (cx<float>*)Cout; t.ldc = ldc;
    t.M = M; t.N = N; t.K = K; t.Mstore = M; t.m0 = 0; t.n0 = 0; t.mask_lo = mask_lo; t.mask_hi = mask_hi; t.sgn = sgn;
    cudaStream_t st = (cudaStream_t)stream;
    if (engine == UST_ENGINE_TC2H && ta) { set_error("ust_test_cgemm: the 128 x 64 engine has no conj(A)^T form"); return 1; }
    if (engine == UST_ENGINE_TC2 || engine == UST_ENGINE_TC2H) {
        // operands are split into bf16 planes first (what the Gauss-Jordan epilogues / tri_apply2_kernel do for the sweeps)
        const int arows = ta ? K : M, acols = ta ? M : K;
        const int nPa = ((std::max(arows, acols) + 63) / 64) * 64;
        const int kpad = ((K + tc2::KC - 1) / tc2::KC) * tc2::KC;
        uint16_t *Ap = nullptr, *Bp = nullptr;
        const size_t ab = (size_t)tc2::NPL_A * nPa * nPa * sizeof(uint16_t), bb = tc2::bplanes_elems(kpad, N) * sizeof(uint16_t);
        UST_CUDA(cudaMalloc((void**)&Ap, ab));
        UST_CUDA(cudaMalloc((void**)&Bp, bb));
        CUtensorMap maps[2];
        unsigned long long* trace_dev = nullptr;
        int rc = tc2::make_aplane_maps(Ap, nPa, 1, maps);
        if (!rc) {
            tc2::ASplitArgs sa;
            sa.src0 = (const cx<float>*)A; sa.src_stride = 0; sa.ld = lda; sa.rows = arows; sa.cols = acols;
            sa.planes = Ap; sa.nP = nPa; sa.mat0 = 0; sa.mat_step = 0;
            tc2::a_split_kernel<<<dim3(cdiv_i(nPa, 256), nPa / 8, 1), 256, 0, st>>>(sa);
            tc2::b_split_kernel<<<dim3(kpad / 8, cdiv_i(N, tc2::TN)), 128, 0, st>>>((const cx<float>*)B, ldb, K, N, kpad, Bp);
            tc2::Tc2Tile tt;
            tc2::tile_no_emit(tt);
            tt.bplanes = Bp; tt.amat = 0; tt.Cin = t.Cin; tt.ldcin = ldcin; tt.Cout = t.Cout; tt.ldc = ldc;
            tt.M = M; tt.N = N; tt.K = K; tt.Mstore = M; tt.m0 = 0; tt.n0 = 0; tt.mask_lo = mask_lo; tt.mask_hi = mask_hi;
            tt.skip_lo = skip_lo; tt.skip_hi = skip_hi; tt.sgn = sgn;
            if (getenv("UST_TC2_TRACE")) { cudaMalloc((void**)&trace_dev, 16 * sizeof(unsigned long long)); cudaMemset(trace_dev, 0, 16 * sizeof(unsigned long long)); }
            tt.trace = trace_dev;
            tt.drain_every = getenv("UST_TC2_TEST_DRAIN") ? atoi(getenv("UST_TC2_TEST_DRAIN")) : 1;
            tt.bias_fix = getenv("UST_TC2_BIAS_FIX") ? (float)atof(getenv("UST_TC2_BIAS_FIX")) : 2.5e-8f;
            dim3 grid(cdiv_i(N, tc2::TN), cdiv_i(M, tc2::TM));
            if (engine == UST_ENGINE_TC2H) tc2h_test_gemm_kernel<<<dim3(cdiv_i(N, tc2::TNH), cdiv_i(M, tc2::TM)), tc2::NUM_THREADS_H, tc2::SMEM_BYTES_H, st>>>(tt, maps[0]);
            else if (ta) tc2_test_gemm_kernel<true><<<grid, tc2::NUM_THREADS, tc2::SMEM_BYTES, st>>>(tt, maps[1]);
            else tc2_test_gemm_kernel<false><<<grid, tc2::NUM_THREADS, tc2::SMEM_BYTES, st>>>(tt, maps[0]);
            if (cudaGetLastError() != cudaSuccess) { set_error("tc2 test gemm launch failed"); rc = 1; }
        }
        cudaError_t e = cudaStreamSynchronize(st);
        if (trace_dev) {
            // phase timestamps of CTA (0,0,0) in ns relative to kernel entry (tools/exp_tc2_trace.py)
            unsigned long long h[16];
            cudaMemcpy(h, trace_dev, sizeof(h), cudaMemcpyDeviceToHost);
            fprintf(stderr, "tc2 trace M=%d N=%d K=%d:", M, N, K);
            for (int i = 1; i < 16; ++i) fprintf(stderr, " [%d]%lld", i, h[i] ? (long long)(h[i] - h[0]) : -1LL);
            fprintf(stderr, "\n");
            cudaFree(trace_dev);
        }
        cudaFree(Ap); cudaFree(Bp);
        if (e != cudaSuccess) { set_error(std::string("tc2 test gemm failed: ") + cudaGetErrorString(e)); return 1; }
        return rc;
    }
    if (engine != UST_ENGINE_SIMT) { set_error("ust_test_cgemm: unknown engine (the first tcgen05 engine, value 2, was removed)"); return 1; }
    if (skip_hi > skip_lo) { set_error("ust_test_cgemm: row skipping is a tensor-core engine feature"); return 1; }
    {
        dim3 grid(cdiv_i(N, 64), cdiv_i(M, 64));
        if (ta) simt_test_gemm_kernel<true><<<grid, 256, 0, st>>>(t);
        else simt_test_gemm_kernel<false><<<grid, 256, 0, st>>>(t);
    }
    UST_LAUNCH_CHECK();
    return 0;
}

int ust_profile(ust_plan* p, int enable) {
    UST_TRY(check_plan(p));
    UST_CUDA(cudaSetDevice(p->d.device));
    if (enable && p->ev.empty()) {
        const size_t npairs = 65536;
        p->ev.resize(2 * npairs);
        p->ev_cls.resize(npairs);
        for (auto& e : p->ev) UST_CUDA(cudaEventCreate(&e));
    }
    p->prof = enable != 0;
    p->ev_used = 0;
    return 0;
}

int ust_get_profile(ust_plan* p, double* ms_out, long long* count_out) {
    UST_TRY(check_plan(p));
    UST_CUDA(cudaSetDevice(p->d.device));
    UST_CUDA(cudaDeviceSynchronize());
    for (int c = 0; c < 16; ++c) { ms_out[c] = 0; count_out[c] = 0; }
    for (size_t i = 0; i + 1 < p->ev_used; i += 2) {
        float ms = 0;
        UST_CUDA(cudaEventElapsedTime(&ms, p->ev[i], p->ev[i + 1]));
        int c = p->ev_cls[i / 2];
        ms_out[c] += ms; count_out[c] += 1;
    }
    p->ev_used = 0;
    return 0;
}

int ust_get_status(ust_plan* p, int* status_host) {
    UST_TRY(check_plan(p));
    UST_CUDA(cudaSetDevice(p->d.device));
    UST_CUDA(cudaDeviceSynchronize());
    UST_CUDA(cudaMemcpy(status_host, p->d_status, sizeof(int), cudaMemcpyDeviceToHost));
    return 0;
}

}  // extern "C"
