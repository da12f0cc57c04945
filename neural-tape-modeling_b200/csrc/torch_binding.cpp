// PyTorch C++ extension over the C ABI of include/ntm_b200.h: registers torch.ops.ntm.* (SURVEY.md section 8b).
//
// The shim owns nothing and computes nothing.  Per call it validates shape / dtype / device / contiguity, selects the
// tensor's device (CUDAGuard), takes PyTorch's CURRENT stream of that device, forwards raw pointers to the extern "C"
// entry point in libntm_b200.so and turns a non-zero return code into a TORCH_CHECK failure (Python RuntimeError; the
// reference's own failures on this path are torch RuntimeErrors / AssertionErrors, code/model.py:81,284).  Launches are
// asynchronous and make no allocation of their own, so every op except ntm::delay_check can be captured in a CUDA Graph.
//
//   ntm::prepare / ntm::destroy            parameter blob of one module (RNN.__init__ / load_state_dict, code/model.py:44-45)
//   ntm::gru_forward[_out]                 RNN.forward, code/model.py:67-88
//   ntm::diffdel_forward                   DiffDelRNN.forward, code/model.py:393-424
//   ntm::delay_forward, ntm::delay_check   TimeVaryingDelayLine.forward, code/model.py:269-320 (assert :283)
//   ntm::esr_sums, ntm::esr_sums_rows      ESRLoss / DCPreESR, CoreAudioML/training.py:5-16, GreyBoxDRC/loss_funcs.py:6-52
//   ntm::mrstft_sums_rows                  auraloss MultiResolutionSTFTLoss (auraloss/freq.py), code/test-model.py:253
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/library.h>
#include <torch/types.h>

#include <tuple>
#include <vector>

#include "../../include/ntm_b200.h"

namespace {

using at::Tensor;

void check_rc(int rc, const char* what)
{
    if (rc == NTM_OK) return;
    // NTM_EDELAY is the reference's `assert self.max_delay >= torch.max(dt)`; the Python wrapper maps the message
    TORCH_CHECK(false, "ntm_b200: ", what, ": ", ntm_strerror(rc), " (code ", rc, ")");
}

// (B, 1, T) or (B, T) float32 CUDA tensor with unit stride in T -> row pointer, B, T, ld
struct Rows {
    const float* p;
    int64_t B, T, ld;
};
Rows rows(const Tensor& t, const char* name)
{
    TORCH_CHECK(t.is_cuda(), "ntm_b200: ", name, " must be a CUDA tensor (the engine has no CPU path)");
    TORCH_CHECK(t.scalar_type() == at::kFloat, "ntm_b200: ", name, " must be float32");
    TORCH_CHECK(t.dim() == 3 ? t.size(1) == 1 : t.dim() == 2, "ntm_b200: ", name,
                " must have shape (N_BATCHES, 1, N_SAMPLES), got ", t.sizes());
    const int64_t B = t.size(0), T = t.size(t.dim() - 1);
    TORCH_CHECK(T <= 1 || t.stride(t.dim() - 1) == 1, "ntm_b200: ", name, " must have unit stride along time");
    const int64_t ld = B > 1 ? t.stride(0) : std::max<int64_t>(T, 1);
    TORCH_CHECK(B <= 1 || ld >= T, "ntm_b200: ", name, " rows overlap (stride ", ld, " < ", T, ")");
    return {t.data_ptr<float>(), B, T, ld};
}
float* wptr(const Tensor& t) { return const_cast<float*>(t.data_ptr<float>()); }

void check_state(const Tensor& h, int64_t B, const Tensor& like, const char* name)
{
    TORCH_CHECK(h.is_cuda() && h.device() == like.device() && h.scalar_type() == at::kFloat && h.is_contiguous() &&
                    h.numel() == B * 64,
                "ntm_b200: ", name, " must be a contiguous float32 tensor of ", B, " x 64 values on ", like.device());
}

void* cur_stream(const Tensor& t) { return at::cuda::getCurrentCUDAStream(t.get_device()).stream(); }

int64_t prepare(const Tensor& w_ih, const Tensor& w_hh, const Tensor& b_ih, const Tensor& b_hh, const Tensor& w_out,
                const c10::optional<Tensor>& b_out, int64_t device)
{
    auto host = [](const Tensor& t) { return t.detach().to(at::kCPU, at::kFloat).contiguous(); };
    const Tensor a = host(w_ih), b = host(w_hh), c = host(b_ih), d = host(b_hh), e = host(w_out);
    TORCH_CHECK(b.dim() == 2 && b.size(0) == 3 * b.size(1), "ntm_b200: weight_hh_l0 must be (3H, H)");
    const int64_t H = b.size(1);
    TORCH_CHECK(a.numel() == 3 * H && c.numel() == 3 * H && d.numel() == 3 * H && e.numel() == H,
                "ntm_b200: only input_size=1, output_size=1 models are supported");
    Tensor f;
    if (b_out.has_value()) f = host(*b_out);
    void* handle = nullptr;
    check_rc(ntm_gru_prepare(a.data_ptr<float>(), b.data_ptr<float>(), c.data_ptr<float>(), d.data_ptr<float>(),
                             e.data_ptr<float>(), b_out.has_value() ? f.data_ptr<float>() : nullptr, (int)H, (int)device,
                             &handle),
             "prepare");
    return reinterpret_cast<int64_t>(handle);
}

void destroy(int64_t handle) { ntm_release(reinterpret_cast<void*>(handle)); }

// y and h_out are caller-owned (reused across calls, CUDA-Graph static buffers); h_out may alias h_in
void gru_forward_out(int64_t handle, int64_t mode, const Tensor& x, const c10::optional<Tensor>& h_in, Tensor y,
                     Tensor h_out, bool skip)
{
    const Rows xr = rows(x, "x"), yr = rows(y, "y");
    TORCH_CHECK(yr.B == xr.B && yr.T == xr.T && y.device() == x.device(), "ntm_b200: y must match x");
    check_state(h_out, xr.B, x, "h_out");
    if (h_in.has_value()) check_state(*h_in, xr.B, x, "h_in");
    const c10::cuda::CUDAGuard guard(x.device());
    check_rc(ntm_gru_forward(reinterpret_cast<void*>(handle), (int)mode, xr.p, xr.ld, wptr(y), yr.ld,
                             h_in.has_value() ? h_in->data_ptr<float>() : nullptr, wptr(h_out), xr.B, xr.T, skip ? 1 : 0,
                             cur_stream(x)),
             "gru_forward");
}

std::tuple<Tensor, Tensor> gru_forward(int64_t handle, int64_t mode, const Tensor& x, const c10::optional<Tensor>& h_in,
                                       bool skip)
{
    const Rows xr = rows(x, "x");
    Tensor y = at::empty({xr.B, 1, xr.T}, x.options());
    Tensor h_out = at::empty({1, xr.B, 64}, x.options());
    gru_forward_out(handle, mode, x, h_in, y, h_out, skip);
    return {y, h_out};
}

std::tuple<Tensor, Tensor, Tensor, Tensor> diffdel_forward(int64_t handle, int64_t mode, const Tensor& x, const Tensor& d,
                                                           const c10::optional<Tensor>& h_in, const Tensor& hist,
                                                           bool warmup, bool skip)
{
    const Rows xr = rows(x, "x"), dr = rows(d, "del_traj");
    TORCH_CHECK(dr.B == xr.B && dr.T == xr.T && d.device() == x.device(), "ntm_b200: x ", x.sizes(), " and del_traj ",
                d.sizes(), " must have the same shape and device");
    TORCH_CHECK(hist.is_cuda() && hist.device() == x.device() && hist.scalar_type() == at::kFloat && hist.is_contiguous() &&
                    hist.dim() == 3 && hist.size(0) == xr.B && hist.size(1) == 1,
                "ntm_b200: the delay history must be a contiguous float32 (", xr.B, ", 1, D) tensor on ", x.device());
    if (h_in.has_value()) check_state(*h_in, xr.B, x, "h_in");
    const int64_t D = hist.size(2);
    Tensor y = at::empty({xr.B, 1, xr.T}, x.options()), pre = at::empty({xr.B, 1, xr.T}, x.options());
    Tensor h_out = at::empty({1, xr.B, 64}, x.options()), hist_out = at::empty({xr.B, 1, D}, x.options());
    const int64_t ld = std::max<int64_t>(xr.T, 1);
    const c10::cuda::CUDAGuard guard(x.device());
    check_rc(ntm_diffdel_forward(reinterpret_cast<void*>(handle), (int)mode, xr.p, xr.ld, dr.p, dr.ld, wptr(y), ld,
                                 wptr(pre), ld, h_in.has_value() ? h_in->data_ptr<float>() : nullptr, wptr(h_out),
                                 hist.data_ptr<float>(), wptr(hist_out), xr.B, xr.T, D, warmup ? 1 : 0, skip ? 1 : 0,
                                 cur_stream(x)),
             "diffdel_forward");
    return {y, pre, h_out, hist_out};
}

std::tuple<Tensor, Tensor> delay_forward(const Tensor& x, const Tensor& d, const Tensor& hist, bool warmup)
{
    const Rows xr = rows(x, "x"), dr = rows(d, "dt");
    TORCH_CHECK(dr.B == xr.B && dr.T == xr.T && d.device() == x.device(), "ntm_b200: x ", x.sizes(), " and dt ", d.sizes(),
                " must have the same shape and device");
    TORCH_CHECK(hist.is_cuda() && hist.device() == x.device() && hist.scalar_type() == at::kFloat && hist.is_contiguous() &&
                    hist.dim() == 3 && hist.size(0) == xr.B && hist.size(1) == 1,
                "ntm_b200: the delay history must be a contiguous float32 (", xr.B, ", 1, D) tensor on ", x.device());
    const int64_t D = hist.size(2);
    Tensor y = at::empty({xr.B, 1, xr.T}, x.options()), hist_out = at::empty({xr.B, 1, D}, x.options());
    const c10::cuda::CUDAGuard guard(x.device());
    check_rc(ntm_delay_forward(xr.p, xr.ld, dr.p, dr.ld, wptr(y), std::max<int64_t>(xr.T, 1), hist.data_ptr<float>(),
                               wptr(hist_out), xr.B, xr.T, D, warmup ? 1 : 0, x.get_device(), cur_stream(x)),
             "delay_forward");
    return {y, hist_out};
}

// the reference's assert (code/model.py:283): true <=> every delay is <= max_delay.  Synchronises the stream.
bool delay_check(const Tensor& d, int64_t max_delay)
{
    const Rows dr = rows(d, "dt");
    const c10::cuda::CUDAGuard guard(d.device());
    const int rc = ntm_delay_check(dr.p, dr.ld, dr.B, dr.T, max_delay, d.get_device(), cur_stream(d));
    if (rc == NTM_EDELAY) return false;
    check_rc(rc, "delay_check");
    return true;
}

Tensor esr_sums(const Tensor& out, const Tensor& target, bool dc_pre)
{
    const Rows o = rows(out, "output"), t = rows(target, "target");
    TORCH_CHECK(o.B == t.B && o.T == t.T && out.device() == target.device(), "ntm_b200: output ", out.sizes(), " and target ",
                target.sizes(), " differ");
    Tensor sums = at::empty({2}, out.options().dtype(at::kDouble));
    const c10::cuda::CUDAGuard guard(out.device());
    check_rc(ntm_esr_sums(o.p, o.ld, t.p, t.ld, o.B, o.T, dc_pre ? 1 : 0, sums.data_ptr<double>(), out.get_device(),
                          cur_stream(out)),
             "esr_sums");
    return sums;
}

// first / count of the per-row ops: a contiguous int64 tensor of B values on the device of `like`, or None (nullptr)
const int64_t* row_index(const c10::optional<Tensor>& v, int64_t B, const Tensor& like, const char* name)
{
    if (!v.has_value()) return nullptr;
    TORCH_CHECK(v->is_cuda() && v->device() == like.device() && v->scalar_type() == at::kLong && v->is_contiguous() &&
                    v->numel() == B,
                "ntm_b200: ", name, " must be a contiguous int64 tensor of ", B, " values on ", like.device());
    return v->data_ptr<int64_t>();
}

// per-row sums over samples [first[b], first[b] + count[b]) of row b (int64 CUDA tensors of B values, or None = whole rows)
Tensor esr_sums_rows(const Tensor& out, const Tensor& target, const c10::optional<Tensor>& first,
                     const c10::optional<Tensor>& count, bool dc_pre)
{
    const Rows o = rows(out, "output"), t = rows(target, "target");
    TORCH_CHECK(o.B == t.B && o.T == t.T && out.device() == target.device(), "ntm_b200: output ", out.sizes(), " and target ",
                target.sizes(), " differ");
    Tensor sums = at::empty({o.B, 2}, out.options().dtype(at::kDouble));
    const c10::cuda::CUDAGuard guard(out.device());
    check_rc(ntm_esr_sums_rows(o.p, o.ld, t.p, t.ld, o.B, o.T, row_index(first, o.B, out, "first"),
                               row_index(count, o.B, out, "count"), dc_pre ? 1 : 0, sums.data_ptr<double>(),
                               out.get_device(), cur_stream(out)),
             "esr_sums_rows");
    return sums;
}

// per-row, per-resolution sums of the multi-resolution STFT loss: (B, n_res, 4) doubles, windows as esr_sums_rows
Tensor mrstft_sums_rows(const Tensor& out, const Tensor& target, const c10::optional<Tensor>& first,
                        const c10::optional<Tensor>& count, at::IntArrayRef fft_sizes, at::IntArrayRef hop_sizes,
                        at::IntArrayRef win_lengths)
{
    const Rows o = rows(out, "output"), t = rows(target, "target");
    TORCH_CHECK(o.B == t.B && o.T == t.T && out.device() == target.device(), "ntm_b200: output ", out.sizes(), " and target ",
                target.sizes(), " differ");
    const size_t n = fft_sizes.size();
    TORCH_CHECK(n > 0 && hop_sizes.size() == n && win_lengths.size() == n,
                "ntm_b200: fft_sizes, hop_sizes and win_lengths must have the same non-zero length");
    std::vector<int> fft(n), hop(n), win(n);
    for (size_t r = 0; r < n; ++r) {
        TORCH_CHECK(fft_sizes[r] >= 256 && fft_sizes[r] <= 4096 && (fft_sizes[r] & (fft_sizes[r] - 1)) == 0,
                    "ntm_b200: fft sizes must be powers of two from 256 to 4096, got ", fft_sizes[r]);
        TORCH_CHECK(win_lengths[r] >= 1 && win_lengths[r] <= fft_sizes[r], "ntm_b200: win_length ", win_lengths[r],
                    " must be in [1, fft_size = ", fft_sizes[r], "]");
        TORCH_CHECK(hop_sizes[r] >= 1 && hop_sizes[r] <= INT32_MAX, "ntm_b200: hop sizes must be >= 1, got ", hop_sizes[r]);
        fft[r] = (int)fft_sizes[r];
        hop[r] = (int)hop_sizes[r];
        win[r] = (int)win_lengths[r];
    }
    Tensor sums = at::empty({o.B, (int64_t)n, 4}, out.options().dtype(at::kDouble));
    const c10::cuda::CUDAGuard guard(out.device());
    check_rc(ntm_mrstft_sums_rows(o.p, o.ld, t.p, t.ld, o.B, o.T, row_index(first, o.B, out, "first"),
                                  row_index(count, o.B, out, "count"), (int)n, fft.data(), hop.data(), win.data(),
                                  sums.data_ptr<double>(), out.get_device(), cur_stream(out)),
             "mrstft_sums_rows");
    return sums;
}

}  // namespace

TORCH_LIBRARY(ntm, m)
{
    m.def("prepare(Tensor w_ih, Tensor w_hh, Tensor b_ih, Tensor b_hh, Tensor w_out, Tensor? b_out, int device) -> int", &prepare);
    m.def("destroy(int handle) -> ()", &destroy);
    m.def("gru_forward(int handle, int mode, Tensor x, Tensor? h_in, bool skip) -> (Tensor, Tensor)", &gru_forward);
    m.def("gru_forward_out(int handle, int mode, Tensor x, Tensor? h_in, Tensor(a!) y, Tensor(b!) h_out, bool skip) -> ()",
          &gru_forward_out);
    m.def("diffdel_forward(int handle, int mode, Tensor x, Tensor d, Tensor? h_in, Tensor hist, bool warmup, bool skip) -> "
          "(Tensor, Tensor, Tensor, Tensor)",
          &diffdel_forward);
    m.def("delay_forward(Tensor x, Tensor d, Tensor hist, bool warmup) -> (Tensor, Tensor)", &delay_forward);
    m.def("delay_check(Tensor d, int max_delay) -> bool", &delay_check);
    m.def("esr_sums(Tensor output, Tensor target, bool dc_pre) -> Tensor", &esr_sums);
    m.def("esr_sums_rows(Tensor output, Tensor target, Tensor? first, Tensor? count, bool dc_pre) -> Tensor", &esr_sums_rows);
    m.def("mrstft_sums_rows(Tensor output, Tensor target, Tensor? first, Tensor? count, int[] fft_sizes, int[] hop_sizes, "
          "int[] win_lengths) -> Tensor",
          &mrstft_sums_rows);
}
