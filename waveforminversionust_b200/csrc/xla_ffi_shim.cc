// xla_ffi_shim.cc -- XLA FFI custom-call handlers over the C ABI of libustfwi.so (include/ustfwi.h).
//
// Replaces the jax.pure_callback(scipy_solve, ...) seam of the reference (Final_python/solve_helmholtz.py:85-93)
// so that solve_helmholtz / fwi_loss_function stay traceable inside jax.jit / lax.scan / jaxopt.LBFGS.
// NOT part of libustfwi.so: it needs the XLA FFI headers that ship with jaxlib (jax.ffi.include_dir()), which
// are absent from the build image; waveforminversionust_b200/jax_frontend.py compiles it against them when they are
// present.  In this image it is compiled against a TEST DOUBLE of that header (tests/xla_ffi_stub/) and its handlers are
// driven on the GPU by tests/test_ffi_shim.py, so the code below has met a compiler and run -- but not inside XLA.
// Every handler only forwards device pointers + XLA's stream to the C ABI; there is no numerical code here.
// Its plans keep the default gradient mode, UST_GRAD_REFERENCE: the discrete mode (ust_plan_set_gradient) is not exposed here.
// The loss is returned as two float32 words (hi, lo with hi + lo = the float64 loss to ~1e-14): the reference runs JAX
// with x64 disabled, where a float64 result buffer cannot exist.
#include <cuda_runtime.h>

#include <map>
#include <mutex>
#include <tuple>
#include <vector>

#include "../../include/ustfwi.h"
#include "xla/ffi/api/ffi.h"

namespace ffi = xla::ffi;

namespace {

struct PlanKey {
    int nx, ny, device, max_freq, max_nrhs, fwi;
    bool operator<(const PlanKey& o) const {
        return std::tie(nx, ny, device, max_freq, max_nrhs, fwi) < std::tie(o.nx, o.ny, o.device, o.max_freq, o.max_nrhs, o.fwi);
    }
};
std::mutex g_mu;
std::map<PlanKey, ust_plan*> g_plans;
std::map<int, double*> g_loss_scratch;  // one device double per GPU for ust_fwi_loss_grad's loss

double* loss_scratch(int dev) {
    auto it = g_loss_scratch.find(dev);
    if (it != g_loss_scratch.end()) return it->second;
    double* d = nullptr;
    if (cudaMalloc((void**)&d, sizeof(double)) != cudaSuccess) return nullptr;
    g_loss_scratch[dev] = d;
    return d;
}

ust_plan* get_plan(const PlanKey& k) {
    auto it = g_plans.find(k);
    if (it != g_plans.end()) return it->second;
    ust_plan_desc d{k.nx, k.ny, UST_C64, k.max_freq, k.max_nrhs, k.device, UST_STENCIL_PYTHON, UST_ENGINE_AUTO, k.fwi};
    ust_plan* p = nullptr;
    if (ust_plan_create(&d, &p)) return nullptr;
    g_plans[k] = p;
    return p;
}

ffi::Error fail(const char* what) { return ffi::Error(ffi::ErrorCode::kInternal, std::string(what) + ": " + ust_last_error()); }

// small host copies of x / y (grid coordinates) and scalar operands: they are device buffers under XLA
template <typename T>
std::vector<double> to_host(cudaStream_t st, const T* dev, size_t n) {
    std::vector<T> tmp(n);
    cudaMemcpyAsync(tmp.data(), dev, n * sizeof(T), cudaMemcpyDeviceToHost, st);
    cudaStreamSynchronize(st);
    return std::vector<double>(tmp.begin(), tmp.end());
}

// solve_helmholtz(x, y, vel, rhs, f, adjoint; a0, L_PML) -> (Ny*Nx, nrhs) complex64   (solve_helmholtz.py:21-101)
ffi::Error SolveImpl(cudaStream_t st, ffi::Buffer<ffi::F32> x, ffi::Buffer<ffi::F32> y, ffi::Buffer<ffi::F32> vel,
                     ffi::Buffer<ffi::C64> rhs, ffi::Buffer<ffi::F32> f, ffi::Buffer<ffi::S32> adjoint, double a0, double L_PML,
                     ffi::ResultBuffer<ffi::C64> out) {
    const int nx = (int)x.element_count(), ny = (int)y.element_count();
    const int nrhs = (int)(rhs.element_count() / ((size_t)nx * ny));
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lk(g_mu);
    ust_plan* p = get_plan({nx, ny, dev, 1, nrhs, 0});
    if (!p) return fail("ust_plan_create");
    std::vector<double> xh = to_host(st, x.typed_data(), nx), yh = to_host(st, y.typed_data(), ny);
    std::vector<double> fh = to_host(st, f.typed_data(), 1);
    int adj = 0;
    cudaMemcpyAsync(&adj, adjoint.typed_data(), sizeof(int), cudaMemcpyDeviceToHost, st);
    cudaStreamSynchronize(st);
    if (ust_plan_set_grid(p, xh.data(), yh.data(), a0, L_PML)) return fail("ust_plan_set_grid");
    if (ust_factor(p, vel.typed_data(), 1, fh.data(), nullptr, st)) return fail("ust_factor");
    cudaMemcpyAsync(out->typed_data(), rhs.typed_data(), rhs.size_bytes(), cudaMemcpyDeviceToDevice, st);
    if (ust_solve(p, 0, out->typed_data(), nrhs, adj, st)) return fail("ust_solve");
    return ffi::Error::Success();
}

// fwi_loss_function(params, REC_DATA, src_lin, rx_lin, mask, x, y, f; a0, L_PML) -> (loss f32[2] = (hi, lo), grad f32[Ny,Nx])
// (fwi_loss_function.py:29-103 + nonlinearcg.py:243-265)
ffi::Error LossGradImpl(cudaStream_t st, ffi::Buffer<ffi::F32> slow, ffi::Buffer<ffi::C64> rec, ffi::Buffer<ffi::S32> src_lin,
                        ffi::Buffer<ffi::S32> rx_lin, ffi::Buffer<ffi::S32> mask, ffi::Buffer<ffi::F32> x, ffi::Buffer<ffi::F32> y,
                        ffi::Buffer<ffi::F32> f, double a0, double L_PML, ffi::ResultBuffer<ffi::F32> loss,
                        ffi::ResultBuffer<ffi::F32> grad) {
    const int nx = (int)x.element_count(), ny = (int)y.element_count();
    const int nt = (int)src_lin.element_count(), nelem = (int)rx_lin.element_count();
    const int nm = (int)(mask.element_count() / nt), nfreq = (int)f.element_count();
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lk(g_mu);
    ust_plan* p = get_plan({nx, ny, dev, nfreq, nt, 1});
    if (!p) return fail("ust_plan_create");
    std::vector<double> xh = to_host(st, x.typed_data(), nx), yh = to_host(st, y.typed_data(), ny);
    std::vector<double> fh = to_host(st, f.typed_data(), nfreq);
    std::vector<int32_t> s(nt), r(nelem), m((size_t)nt * nm);
    cudaMemcpyAsync(s.data(), src_lin.typed_data(), s.size() * 4, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(r.data(), rx_lin.typed_data(), r.size() * 4, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(m.data(), mask.typed_data(), m.size() * 4, cudaMemcpyDeviceToHost, st);
    cudaStreamSynchronize(st);
    if (ust_plan_set_grid(p, xh.data(), yh.data(), a0, L_PML)) return fail("ust_plan_set_grid");
    if (ust_plan_set_acquisition(p, nt, s.data(), nelem, r.data(), nm, m.data())) return fail("ust_plan_set_acquisition");
    double* loss64 = loss_scratch(dev);
    if (!loss64) return ffi::Error(ffi::ErrorCode::kInternal, "cudaMalloc of the loss scratch failed");
    if (ust_fwi_loss_grad(p, slow.typed_data(), rec.typed_data(), nfreq, fh.data(), nullptr, loss64, grad->typed_data(), st))
        return fail("ust_fwi_loss_grad");
    if (ust_pack_f64_as_f32x2(loss64, loss->typed_data(), 1, st)) return fail("ust_pack_f64_as_f32x2");
    return ffi::Error::Success();
}

}  // namespace

XLA_FFI_DEFINE_HANDLER_SYMBOL(ust_solve_helmholtz_ffi, SolveImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()   // x
                                  .Arg<ffi::Buffer<ffi::F32>>()   // y
                                  .Arg<ffi::Buffer<ffi::F32>>()   // vel (Ny, Nx)
                                  .Arg<ffi::Buffer<ffi::C64>>()   // rhs (Ny*Nx, nrhs)
                                  .Arg<ffi::Buffer<ffi::F32>>()   // f (1,)
                                  .Arg<ffi::Buffer<ffi::S32>>()   // adjoint (1,) -- traced in the reference (lax.cond)
                                  .Attr<double>("a0")
                                  .Attr<double>("L_PML")
                                  .Ret<ffi::Buffer<ffi::C64>>());

XLA_FFI_DEFINE_HANDLER_SYMBOL(ust_fwi_loss_grad_ffi, LossGradImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()   // slowness params (Ny, Nx)
                                  .Arg<ffi::Buffer<ffi::C64>>()   // REC_DATA (nfreq, Nt, E)
                                  .Arg<ffi::Buffer<ffi::S32>>()   // one-hot source nodes (Nt,)
                                  .Arg<ffi::Buffer<ffi::S32>>()   // receiver nodes (E,)
                                  .Arg<ffi::Buffer<ffi::S32>>()   // mask_indices (Nt, Nm)
                                  .Arg<ffi::Buffer<ffi::F32>>()   // x
                                  .Arg<ffi::Buffer<ffi::F32>>()   // y
                                  .Arg<ffi::Buffer<ffi::F32>>()   // f (nfreq,)
                                  .Attr<double>("a0")
                                  .Attr<double>("L_PML")
                                  .Ret<ffi::Buffer<ffi::F32>>()   // loss (2,) = (hi, lo)
                                  .Ret<ffi::Buffer<ffi::F32>>()); // grad (Ny, Nx)
