// Python bindings of the gossipy_b200 sm_100a extension (module gossipy_b200._C).
//
// The kernels live in csrc/kernels/*.cu (plain CUDA, compiled by nvcc without torch headers); this
// file is the only translation unit that sees at::Tensor: it validates arguments, picks the current
// stream of the tensor's device and calls the launchers of kernels/kernels.h.
#include <torch/extension.h>
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <cuda_runtime.h>
#include <cstring>
#include <tuple>
#include <vector>

#include "kernels/kernels.h"
#include "exec/executor.h"
#include "sched/scheduler.h"

namespace gb {

#define GB_LAUNCH_CHECK() C10_CUDA_KERNEL_LAUNCH_CHECK()

static cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream(); }

// (ready flag address, generation, done counter address); zeros = no cross-GPU handshake
using Sync = std::tuple<int64_t, int64_t, int64_t>;
static PeerSync to_sync(const c10::optional<Sync>& s) {
    PeerSync p{nullptr, 0u, nullptr, nullptr};
    if (s.has_value()) {
        p.fault = device_fault_word();
        p.ready = reinterpret_cast<const uint32_t*>((uintptr_t)std::get<0>(*s));
        p.gen = (uint32_t)std::get<1>(*s);
        p.done = reinterpret_cast<uint32_t*>((uintptr_t)std::get<2>(*s));
    }
    return p;
}

static void check_row(const at::Tensor& t, const char* name) {
    TORCH_CHECK(t.is_cuda() && t.scalar_type() == at::kFloat && t.is_contiguous(), name,
                " must be a contiguous fp32 CUDA tensor");
}

// ---- merges --------------------------------------------------------------------------------------
void merge_pair(at::Tensor dst, at::Tensor src, double w_dst, double w_src, int64_t lo, int64_t hi,
                c10::optional<Sync> sync) {
    check_row(dst, "dst");
    TORCH_CHECK(src.is_cuda() && src.scalar_type() == at::kFloat && src.is_contiguous());
    TORCH_CHECK(0 <= lo && lo <= hi && hi <= dst.numel() && hi <= src.numel());
    c10::cuda::CUDAGuard guard(dst.device());
    launch_merge_pair(dst.data_ptr<float>(), src.data_ptr<float>(), (float)w_dst, (float)w_src, lo, hi,
                      to_sync(sync), cur_stream());
    GB_LAUNCH_CHECK();
}

void merge_segments(at::Tensor dst, at::Tensor src, at::Tensor seg, double w_dst, double w_src,
                    c10::optional<Sync> sync) {
    check_row(dst, "dst");
    TORCH_CHECK(seg.is_cuda() && seg.scalar_type() == at::kLong && seg.is_contiguous());
    TORCH_CHECK(seg.dim() == 2 && seg.size(1) == 4);
    c10::cuda::CUDAGuard guard(dst.device());
    launch_merge_segments(dst.data_ptr<float>(), src.data_ptr<float>(), seg.data_ptr<int64_t>(),
                          (int)seg.size(0), (float)w_dst, (float)w_src, to_sync(sync), cur_stream());
    GB_LAUNCH_CHECK();
}

void merge_indexed(at::Tensor dst, at::Tensor src, at::Tensor idx, double w_dst, double w_src,
                   c10::optional<Sync> sync) {
    check_row(dst, "dst");
    TORCH_CHECK(idx.is_cuda() && idx.scalar_type() == at::kLong && idx.is_contiguous());
    const int64_t n = idx.numel();
    if (n == 0) return;
    c10::cuda::CUDAGuard guard(dst.device());
    auto scratch = at::empty({n}, dst.options());
    launch_merge_indexed(dst.data_ptr<float>(), src.data_ptr<float>(), idx.data_ptr<int64_t>(), n,
                         (float)w_dst, (float)w_src, scratch.data_ptr<float>(), to_sync(sync), cur_stream());
    GB_LAUNCH_CHECK();
}

void merge_kway(at::Tensor dst, std::vector<at::Tensor> srcs, std::vector<double> weights,
                c10::optional<std::vector<Sync>> syncs) {
    check_row(dst, "dst");
    TORCH_CHECK(weights.size() == srcs.size() + 1, "need one weight per model incl. self");
    TORCH_CHECK((((uintptr_t)dst.data_ptr<float>()) & 15u) == 0, "row must be 16-byte aligned");
    TORCH_CHECK(!syncs.has_value() || syncs->size() == srcs.size());
    c10::cuda::CUDAGuard guard(dst.device());
    const int64_t n = dst.numel();
    if (srcs.empty()) { dst.mul_(weights[0]); return; }
    std::vector<const float*> ptrs; std::vector<float> w; std::vector<PeerSync> ps;
    w.push_back((float)weights[0]);
    for (size_t j = 0; j < srcs.size(); ++j) {
        const at::Tensor& s = srcs[j];
        TORCH_CHECK(s.is_cuda() && s.scalar_type() == at::kFloat && s.is_contiguous() && s.numel() >= n);
        TORCH_CHECK((((uintptr_t)s.data_ptr<float>()) & 15u) == 0);
        ptrs.push_back(s.data_ptr<float>());
        w.push_back((float)weights[1 + j]);
        if (syncs.has_value()) ps.push_back(to_sync((*syncs)[j]));
    }
    launch_merge_kway(dst.data_ptr<float>(), ptrs.data(), w.data(), (int)srcs.size(), n,
                      syncs.has_value() ? ps.data() : nullptr, cur_stream());
    GB_LAUNCH_CHECK();
}

// ---- optimizers ------------------------------------------------------------------------------------
void sgd_step(at::Tensor p, at::Tensor g, int64_t n, double lr, double wd, double momentum,
              c10::optional<at::Tensor> buf, double dampening, bool nesterov, bool first,
              c10::optional<at::Tensor> scale) {
    check_row(p, "p"); check_row(g, "g");
    TORCH_CHECK(n <= p.numel() && n <= g.numel());
    c10::cuda::CUDAGuard guard(p.device());
    launch_sgd(p.data_ptr<float>(), g.data_ptr<float>(), n, (float)lr, (float)wd, (float)momentum,
               buf.has_value() ? buf->data_ptr<float>() : nullptr, (float)dampening, nesterov, first,
               scale.has_value() ? scale->data_ptr<float>() : nullptr, cur_stream());
    GB_LAUNCH_CHECK();
}

at::Tensor keyed_perm(int64_t n, int64_t key, at::Device device) {
    TORCH_CHECK(device.is_cuda() && n >= 0 && n < (int64_t(1) << 31));
    c10::cuda::CUDAGuard guard(device);
    at::Tensor out = at::empty({n}, at::TensorOptions().device(device).dtype(at::kLong));
    launch_keyed_perm(out.data_ptr<int64_t>(), (int)n, (uint64_t)key, cur_stream());
    GB_LAUNCH_CHECK();
    return out;
}

at::Tensor keyed_randint(int64_t k, int64_t n, int64_t key, at::Device device) {
    TORCH_CHECK(device.is_cuda() && k >= 0 && n > 0);
    c10::cuda::CUDAGuard guard(device);
    at::Tensor out = at::empty({k}, at::TensorOptions().device(device).dtype(at::kLong));
    launch_keyed_randint(out.data_ptr<int64_t>(), k, n, (uint64_t)key, cur_stream());
    GB_LAUNCH_CHECK();
    return out;
}

void adam_step(at::Tensor p, at::Tensor g, int64_t n, at::Tensor m, at::Tensor v, int64_t step,
               double lr, double beta1, double beta2, double eps, double wd, bool decoupled) {
    check_row(p, "p"); check_row(g, "g"); check_row(m, "m"); check_row(v, "v");
    c10::cuda::CUDAGuard guard(p.device());
    launch_adam(p.data_ptr<float>(), g.data_ptr<float>(), n, m.data_ptr<float>(), v.data_ptr<float>(), step,
                (float)lr, (float)beta1, (float)beta2, (float)eps, (float)wd, decoupled, cur_stream());
    GB_LAUNCH_CHECK();
}

// ---- fused local updates -----------------------------------------------------------------------------
static thread_local float* g_debug_ptr = nullptr;

// partition ages: a device tensor is passed by pointer, a host tensor (<= 16 partitions) by value in the launch
// parameters -- no H2D copy, nothing for the host to wait for
template <class P> static void set_ages(P& p, const at::Tensor& ages) {
    p.n_parts = (int)ages.numel();
    if (ages.is_cuda()) { p.ages = ages.data_ptr<int64_t>(); return; }
    TORCH_CHECK(p.n_parts <= kMaxPartsByValue && ages.is_contiguous(), "host-side partition ages: at most 16 partitions");
    p.ages = nullptr; p.use_ages_val = true;
    for (int i = 0; i < p.n_parts; ++i) p.ages_val[i] = ages.data_ptr<int64_t>()[i];
}

static TrainImpl parse_train_impl(const std::string& impl) {
    const TrainImpl which = impl == "cluster" ? kTrainCluster : impl == "tc3" ? kTrainTc3
                            : impl == "tc8" ? kTrainTc8 : impl == "tc8-tf32" ? kTrainTc8Tf32 : kTrainAuto;
    TORCH_CHECK(which != kTrainAuto || impl.empty() || impl == "auto", "unknown training kernel '", impl,
                "' (cluster | tc8 | tc8-tf32 | tc3)");
    return which;
}
// what the automatic choice means for this process (also used by the C++ executor)
void set_train_impl(std::string impl) { set_default_train_impl(parse_train_impl(impl)); }

int64_t mlp1_train(at::Tensor row, at::Tensor X, at::Tensor y, std::tuple<int64_t, int64_t, int64_t> dims,
                   int64_t batch_size, int64_t local_epochs, double lr, double wd, int64_t key,
                   c10::optional<at::Tensor> part_id, c10::optional<at::Tensor> ages, std::string impl,
                   c10::optional<at::Tensor> peer, double w_self, double w_peer, c10::optional<Sync> sync,
                   double momentum = 0.0, double dampening = 0.0, bool nesterov = false,
                   c10::optional<at::Tensor> mom = c10::nullopt, bool mom_first = false) {
    check_row(row, "row"); check_row(X, "X");
    TORCH_CHECK(y.is_cuda() && y.scalar_type() == at::kLong && y.is_contiguous() && X.dim() == 2);
    TrainParams p{};
    p.IN = (int)std::get<0>(dims); p.H = (int)std::get<1>(dims); p.OUT = (int)std::get<2>(dims);
    p.n = (int)X.size(0);
    TORCH_CHECK(X.size(1) == p.IN && y.numel() == p.n && p.n > 0);
    const int64_t P = (int64_t)p.H * p.IN + p.H + (int64_t)p.OUT * p.H + p.OUT;
    TORCH_CHECK(row.numel() >= P);
    p.B = (int)(batch_size == 0 ? p.n : std::min<int64_t>(batch_size, p.n));
    p.epochs = (int)local_epochs;
    p.lr = (float)lr; p.wd = (float)wd; p.key = (uint64_t)key;
    p.row = row.data_ptr<float>(); p.X = X.data_ptr<float>(); p.y = y.data_ptr<int64_t>();
    p.dbg = g_debug_ptr;
    if (part_id.has_value() && ages.has_value()) {
        TORCH_CHECK(part_id->is_cuda() && part_id->scalar_type() == at::kLong && ages->scalar_type() == at::kLong);
        p.part_id = part_id->data_ptr<int64_t>();
        set_ages(p, *ages);
    }
    if (peer.has_value()) {
        TORCH_CHECK(peer->is_cuda() && peer->scalar_type() == at::kFloat && peer->numel() >= P);
        p.peer = peer->data_ptr<float>(); p.w_self = (float)w_self; p.w_peer = (float)w_peer;
        p.sync = to_sync(sync);
    }
    if (momentum != 0.0) {
        TORCH_CHECK(mom.has_value() && mom->is_cuda() && mom->scalar_type() == at::kFloat && mom->is_contiguous() &&
                    mom->numel() >= P, "momentum needs the momentum-buffer row");
        p.momentum = (float)momentum; p.dampening = (float)dampening; p.nesterov = nesterov;
        p.mom = mom->data_ptr<float>(); p.mom_first = mom_first;
    }
    c10::cuda::CUDAGuard guard(row.device());
    const TrainImpl which = parse_train_impl(impl);
    const char* why = "";
    const bool ok = launch_mlp1_train(p, which, cur_stream(), &why);
    TORCH_CHECK(ok, why, " (in=", p.IN, " hidden=", p.H, " out=", p.OUT, " batch=", p.B, ")");
    GB_LAUNCH_CHECK();
    const int spe = (p.n + p.B - 1) / p.B;
    return p.epochs > 0 ? (int64_t)p.epochs * spe : 1;
}

at::Tensor mlp1_train_tc_debug(at::Tensor row, at::Tensor X, at::Tensor y,
                               std::tuple<int64_t, int64_t, int64_t> dims, int64_t batch_size,
                               int64_t local_epochs, double lr, double wd, int64_t key, std::string impl) {
    // runs a tcgen05 kernel with its debug buffer attached: lr == 0 -> relu(z1) [128, 32] of the first
    // step (bring-up test); lr != 0 -> average cycles per step of each phase in the first 6 floats
    auto dbg = at::zeros({128, 32}, row.options());
    g_debug_ptr = dbg.data_ptr<float>();
    mlp1_train(row, X, y, dims, batch_size, local_epochs, lr, wd, key, c10::nullopt, c10::nullopt, impl,
               c10::nullopt, 1.0, 0.0, c10::nullopt);
    g_debug_ptr = nullptr;
    return dbg;
}

std::tuple<at::Tensor, at::Tensor, at::Tensor, int64_t> mlp1_stage_debug(at::Tensor X, at::Tensor y,
                                                                         int64_t batch_size, int64_t local_epochs,
                                                                         int64_t key) {
    // runs the device-side loader of the tc3 training kernel and returns (XF, XT, YS, FP)
    check_row(X, "X");
    TORCH_CHECK(y.is_cuda() && y.scalar_type() == at::kLong && y.is_contiguous());
    const int n = (int)X.size(0), IN = (int)X.size(1);
    const int B = (int)std::min<int64_t>(batch_size, n);
    int FPC, FP, steps;
    const size_t bytes = mlp1_stage_bytes(n, IN, B, (int)local_epochs, &FPC, &FP, &steps);
    c10::cuda::CUDAGuard guard(X.device());
    auto buf = at::empty({(int64_t)(bytes / 4)}, X.options());
    TORCH_CHECK(launch_mlp1_stage(X.data_ptr<float>(), y.data_ptr<int64_t>(), n, IN, B, (int)local_epochs,
                                  (uint64_t)key, buf.data_ptr<float>(), cur_stream()), "unsupported shape");
    GB_LAUNCH_CHECK();
    const int64_t tile = 32 * (int64_t)FP;
    auto xf = buf.narrow(0, 0, steps * 2 * tile).view({steps, 2, tile});
    auto xt = buf.narrow(0, steps * 2 * tile, steps * 2 * tile).view({steps, 2, tile});
    auto ys = buf.narrow(0, steps * 4 * tile, steps * 32).view(at::kInt).view({steps, 32});
    return {xf, xt, ys, (int64_t)FP};
}

std::tuple<at::Tensor, c10::optional<at::Tensor>> mlp1_eval(at::Tensor row, at::Tensor X, at::Tensor y,
                                                            std::tuple<int64_t, int64_t, int64_t> dims, int64_t n_classes,
                                                            c10::optional<at::Tensor> X_lp, bool want_score1) {
    // confusion matrix [C, C] (int32) and, on request, the class-1 logit of every sample (AUC of 2-output networks)
    check_row(row, "row"); check_row(X, "X");
    TORCH_CHECK(y.is_cuda() && y.scalar_type() == at::kLong && y.is_contiguous());
    const int IN = (int)std::get<0>(dims), H = (int)std::get<1>(dims), OUT = (int)std::get<2>(dims);
    const int n = (int)X.size(0);
    TORCH_CHECK(X.size(1) == IN && y.numel() == n);
    c10::cuda::CUDAGuard guard(row.device());
    auto cm = at::zeros({n_classes, n_classes}, row.options().dtype(at::kInt));
    c10::optional<at::Tensor> sc;
    float* scp = nullptr;
    if (want_score1) { sc = at::empty({n}, row.options()); scp = sc->data_ptr<float>(); }
    if (X_lp.has_value()) {      // pre-tiled test set -> tensor-core kernel
        TORCH_CHECK(X_lp->is_cuda() && X_lp->scalar_type() == at::kFloat && X_lp->is_contiguous() &&
                    X_lp->numel() == mlp1_eval_pretile_floats(n, IN), "X_lp must come from mlp1_eval_pretile(X)");
        if (launch_mlp1_eval_tc(row.data_ptr<float>(), X_lp->data_ptr<float>(), y.data_ptr<int64_t>(), n, IN, H,
                                OUT, (int)n_classes, cm.data_ptr<int>(), scp, cur_stream())) {
            GB_LAUNCH_CHECK();
            return {cm, sc};
        }
    }
    TORCH_CHECK(launch_mlp1_eval(row.data_ptr<float>(), X.data_ptr<float>(), y.data_ptr<int64_t>(), n, IN, H,
                                 OUT, (int)n_classes, cm.data_ptr<int>(), scp, cur_stream()),
                "mlp1_eval: hidden <= 128 and out <= 16 supported");
    GB_LAUNCH_CHECK();
    return {cm, sc};
}

at::Tensor mlp1_eval_pretile(at::Tensor X) {
    // the test set in the operand image of the tensor-core evaluation kernel (done once per data set)
    check_row(X, "X");
    TORCH_CHECK(X.dim() == 2);
    const int n = (int)X.size(0), IN = (int)X.size(1);
    c10::cuda::CUDAGuard guard(X.device());
    auto out = at::empty({mlp1_eval_pretile_floats(n, IN)}, X.options());
    launch_mlp1_eval_pretile(X.data_ptr<float>(), n, IN, out.data_ptr<float>(), cur_stream());
    GB_LAUNCH_CHECK();
    return out;
}

int64_t logreg_train(at::Tensor row, at::Tensor X, at::Tensor y, std::tuple<int64_t, int64_t> dims,
                     int64_t batch_size, int64_t local_epochs, double lr, double wd, int64_t key,
                     c10::optional<at::Tensor> part_id, c10::optional<at::Tensor> ages,
                     c10::optional<at::Tensor> peer, double w_self, double w_peer, c10::optional<Sync> sync) {
    check_row(row, "row"); check_row(X, "X");
    TORCH_CHECK(y.is_cuda() && y.scalar_type() == at::kLong && y.is_contiguous());
    LogregParams p{};
    p.IN = (int)std::get<0>(dims); p.OUT = (int)std::get<1>(dims);
    p.n = (int)X.size(0);
    TORCH_CHECK(X.dim() == 2 && X.size(1) == p.IN && p.n > 0);
    p.B = (int)(batch_size == 0 ? p.n : std::min<int64_t>(batch_size, p.n));
    p.epochs = (int)local_epochs; p.lr = (float)lr; p.wd = (float)wd; p.key = (uint64_t)key;
    p.row = row.data_ptr<float>(); p.X = X.data_ptr<float>(); p.y = y.data_ptr<int64_t>();
    if (part_id.has_value() && ages.has_value()) {
        p.part_id = part_id->data_ptr<int64_t>();
        set_ages(p, *ages);
    }
    if (peer.has_value()) {
        TORCH_CHECK(peer->is_cuda() && peer->scalar_type() == at::kFloat);
        p.peer = peer->data_ptr<float>(); p.w_self = (float)w_self; p.w_peer = (float)w_peer;
        p.sync = to_sync(sync);
    }
    c10::cuda::CUDAGuard guard(row.device());
    TORCH_CHECK(launch_logreg_train(p, cur_stream()), "logreg_train: unsupported shape for the fused kernel");
    GB_LAUNCH_CHECK();
    const int spe = (p.n + p.B - 1) / p.B;
    return p.epochs > 0 ? (int64_t)p.epochs * spe : 1;
}

at::Tensor logreg_scores(at::Tensor row, at::Tensor X, std::tuple<int64_t, int64_t> dims) {
    check_row(row, "row"); check_row(X, "X");
    const int IN = (int)std::get<0>(dims), OUT = (int)std::get<1>(dims), n = (int)X.size(0);
    c10::cuda::CUDAGuard guard(row.device());
    auto out = at::empty({n, OUT}, X.options());
    launch_logreg_scores(row.data_ptr<float>(), X.data_ptr<float>(), n, IN, OUT, out.data_ptr<float>(), cur_stream());
    GB_LAUNCH_CHECK();
    return out;
}

void linear_seq_update(at::Tensor w, at::Tensor X, at::Tensor y, int64_t kind, double lr, int64_t n_updates) {
    TORCH_CHECK(w.is_cuda() && X.is_cuda() && y.is_cuda());
    auto Xc = X.to(at::kFloat).contiguous();
    auto yc = y.to(at::kFloat).contiguous();
    const int dim = (int)w.numel(), n = (int)Xc.size(0);
    TORCH_CHECK(dim <= 1024 && Xc.numel() == (int64_t)n * dim && yc.numel() == n);
    c10::cuda::CUDAGuard guard(w.device());
    launch_linear_seq(w.data_ptr<float>(), Xc.data_ptr<float>(), yc.data_ptr<float>(), n, dim, (int)kind,
                      (float)lr, (long long)n_updates, cur_stream());
    GB_LAUNCH_CHECK();
}

at::Tensor kmeans_assign(at::Tensor C, at::Tensor X) {
    TORCH_CHECK(C.is_cuda() && X.is_cuda() && C.dim() == 2);
    auto Xc = X.to(at::kFloat).contiguous();
    auto Cc = C.contiguous();
    const int k = (int)C.size(0), dim = (int)C.size(1), n = (int)Xc.size(0);
    c10::cuda::CUDAGuard guard(C.device());
    auto out = at::empty({n}, Xc.options().dtype(at::kLong));
    launch_kmeans_assign(Cc.data_ptr<float>(), Xc.data_ptr<float>(), n, k, dim, out.data_ptr<int64_t>(), cur_stream());
    GB_LAUNCH_CHECK();
    return out;
}

void kmeans_update(at::Tensor C, at::Tensor X, double alpha) {
    TORCH_CHECK(C.is_cuda() && C.is_contiguous() && C.dim() == 2);
    auto Xc = X.to(at::kFloat).contiguous();
    const int k = (int)C.size(0), dim = (int)C.size(1), n = (int)Xc.size(0);
    if (n == 0) return;
    auto asg = kmeans_assign(C, Xc);
    c10::cuda::CUDAGuard guard(C.device());
    launch_kmeans_apply(C.data_ptr<float>(), Xc.data_ptr<float>(), asg.data_ptr<int64_t>(), n, k, dim,
                        (float)alpha, cur_stream());
    GB_LAUNCH_CHECK();
}

void mf_update(at::Tensor X, at::Tensor b, at::Tensor Y, at::Tensor c, at::Tensor ratings, double reg, double lr) {
    TORCH_CHECK(Y.is_cuda() && ratings.is_cuda() && Y.dim() == 2);
    auto rc = ratings.to(at::kFloat).contiguous();
    const int m = (int)rc.size(0), k = (int)Y.size(1);
    TORCH_CHECK(k <= 128, "mf_update: rank <= 128 supported");
    c10::cuda::CUDAGuard guard(Y.device());
    launch_mf_update(X.data_ptr<float>(), b.data_ptr<float>(), Y.data_ptr<float>(), c.data_ptr<float>(),
                     rc.data_ptr<float>(), m, k, (float)reg, (float)lr, cur_stream());
    GB_LAUNCH_CHECK();
}

at::Tensor kmeans_match_merge(at::Tensor C, at::Tensor P, int64_t k, int64_t dim, double w_own, double w_peer,
                              c10::optional<Sync> sync) {
    // C[:k*dim] = w_own * C + w_peer * P[perm] with the optimal (min total distance) matching, k <= 8; returns perm
    check_row(C, "C");
    TORCH_CHECK(P.is_cuda() && P.scalar_type() == at::kFloat && C.numel() >= k * dim && P.numel() >= k * dim);
    c10::cuda::CUDAGuard guard(C.device());
    auto perm = at::empty({k}, C.options().dtype(at::kLong));
    TORCH_CHECK(launch_kmeans_match_merge(C.data_ptr<float>(), P.data_ptr<float>(), (int)k, (int)dim, (float)w_own,
                                          (float)w_peer, to_sync(sync), perm.data_ptr<int64_t>(), cur_stream()),
                "kmeans_match_merge: 1 <= k <= 8");
    GB_LAUNCH_CHECK();
    return perm;
}

// ---- bank of linear learners ----------------------------------------------------------------------------
static BankView bank_view(at::Tensor W, at::Tensor age, at::Tensor S, at::Tensor slot_age, at::Tensor X, at::Tensor y,
                          at::Tensor off, at::Tensor cnt, int64_t D, int64_t kind, int64_t mode, double lr) {
    TORCH_CHECK(W.is_cuda() && W.scalar_type() == at::kFloat && W.is_contiguous() && W.dim() == 2);
    TORCH_CHECK(S.is_cuda() && S.scalar_type() == at::kFloat && S.is_contiguous() && S.dim() == 2 && S.size(1) == W.size(1));
    TORCH_CHECK(age.scalar_type() == at::kLong && slot_age.scalar_type() == at::kLong && off.scalar_type() == at::kLong &&
                cnt.scalar_type() == at::kInt && X.scalar_type() == at::kFloat && y.scalar_type() == at::kFloat);
    TORCH_CHECK(X.is_contiguous() && y.is_contiguous() && age.numel() == W.size(0) && slot_age.numel() == S.size(0));
    BankView b{};
    b.W = W.data_ptr<float>(); b.age = reinterpret_cast<long long*>(age.data_ptr<int64_t>());
    b.S = S.data_ptr<float>(); b.slot_age = reinterpret_cast<long long*>(slot_age.data_ptr<int64_t>());
    b.D = (int)D; b.Dp = (int)W.size(1);
    b.X = X.data_ptr<float>(); b.y = y.data_ptr<float>();
    b.off = off.data_ptr<int64_t>(); b.cnt = cnt.data_ptr<int>();
    b.kind = (int)kind; b.mode = (int)mode; b.lr = (float)lr;
    return b;
}
#define BANK_ARGS at::Tensor W, at::Tensor age, at::Tensor S, at::Tensor slot_age, at::Tensor X, at::Tensor y, \
                  at::Tensor off, at::Tensor cnt, int64_t D, int64_t kind, int64_t mode, double lr
#define BANK_PASS W, age, S, slot_age, X, y, off, cnt, D, kind, mode, lr
static void check_idx(const at::Tensor& t) { TORCH_CHECK(t.is_cuda() && t.scalar_type() == at::kInt && t.is_contiguous()); }
void bank_snapshot(BANK_ARGS, at::Tensor sender, at::Tensor slot) {
    check_idx(sender); check_idx(slot);
    c10::cuda::CUDAGuard guard(W.device());
    launch_bank_snapshot(bank_view(BANK_PASS), sender.data_ptr<int>(), slot.data_ptr<int>(), (int)sender.numel(), cur_stream());
    GB_LAUNCH_CHECK();
}
void bank_snapshot_push(BANK_ARGS, std::vector<int64_t> peer_S, std::vector<int64_t> peer_age, at::Tensor sender,
                        at::Tensor slot, at::Tensor dst_rank) {
    check_idx(sender); check_idx(slot); check_idx(dst_rank);
    TORCH_CHECK(peer_S.size() == peer_age.size() && (int)peer_S.size() <= kMaxRanks && sender.numel() == dst_rank.numel());
    BankPeers pr{};
    for (size_t r = 0; r < peer_S.size(); ++r) {
        pr.S[r] = reinterpret_cast<float*>((uintptr_t)peer_S[r]);
        pr.slot_age[r] = reinterpret_cast<long long*>((uintptr_t)peer_age[r]);
    }
    c10::cuda::CUDAGuard guard(W.device());
    launch_bank_snapshot_push(bank_view(BANK_PASS), pr, sender.data_ptr<int>(), slot.data_ptr<int>(), dst_rank.data_ptr<int>(),
                              (int)sender.numel(), cur_stream());
    GB_LAUNCH_CHECK();
}
void rank_barrier(std::vector<int64_t> flags, int64_t rank, int64_t gen) {
    TORCH_CHECK((int)flags.size() <= kMaxRanks && rank >= 0 && rank < (int64_t)flags.size());
    RankBarrier rb{};
    for (size_t r = 0; r < flags.size(); ++r) rb.flags[r] = reinterpret_cast<uint32_t*>((uintptr_t)flags[r]);
    rb.rank = (int)rank; rb.world = (int)flags.size(); rb.gen = (uint32_t)gen;
    launch_rank_barrier(rb, cur_stream());
    GB_LAUNCH_CHECK();
}
void bank_deliver(BANK_ARGS, at::Tensor recv, at::Tensor slot, c10::optional<at::Tensor> item_mode) {
    check_idx(recv); check_idx(slot);
    if (item_mode.has_value()) { check_idx(*item_mode); TORCH_CHECK(item_mode->numel() == recv.numel()); }
    c10::cuda::CUDAGuard guard(W.device());
    TORCH_CHECK(launch_bank_deliver(bank_view(BANK_PASS), recv.data_ptr<int>(), slot.data_ptr<int>(),
                                    item_mode.has_value() ? item_mode->data_ptr<int>() : nullptr, (int)recv.numel(),
                                    cur_stream()), "bank: dim <= 1024 supported");
    GB_LAUNCH_CHECK();
}
void bank_update(BANK_ARGS, at::Tensor nodes) {
    check_idx(nodes);
    c10::cuda::CUDAGuard guard(W.device());
    TORCH_CHECK(launch_bank_update(bank_view(BANK_PASS), nodes.data_ptr<int>(), (int)nodes.numel(), cur_stream()),
                "bank: dim <= 1024 supported");
    GB_LAUNCH_CHECK();
}
at::Tensor bank_scores(BANK_ARGS, at::Tensor nodes, at::Tensor Xte) {
    check_idx(nodes); check_row(Xte, "Xte");
    c10::cuda::CUDAGuard guard(W.device());
    auto out = at::empty({nodes.numel(), Xte.size(0)}, W.options());
    launch_bank_scores(bank_view(BANK_PASS), nodes.data_ptr<int>(), (int)nodes.numel(), Xte.data_ptr<float>(),
                       (int)Xte.size(0), out.data_ptr<float>(), cur_stream());
    GB_LAUNCH_CHECK();
    return out;
}

// ---- banks of k-means / matrix-factorisation models --------------------------------------------------------
static FamilyBankView family_view(at::Tensor W, at::Tensor age, at::Tensor S, at::Tensor slot_age, at::Tensor data,
                                  at::Tensor off, at::Tensor cnt, int64_t k, int64_t dim, int64_t mode, bool hungarian,
                                  double alpha, double reg, double lr) {
    TORCH_CHECK(W.is_cuda() && W.scalar_type() == at::kFloat && W.is_contiguous() && W.dim() == 2 && W.size(1) % 32 == 0);
    TORCH_CHECK(S.is_cuda() && S.scalar_type() == at::kFloat && S.is_contiguous() && S.dim() == 2 && S.size(1) == W.size(1));
    TORCH_CHECK(age.scalar_type() == at::kLong && slot_age.scalar_type() == at::kLong && off.scalar_type() == at::kLong &&
                cnt.scalar_type() == at::kInt && data.scalar_type() == at::kFloat);
    TORCH_CHECK(data.is_contiguous() && off.numel() == W.size(0) && cnt.numel() == W.size(0) &&
                age.numel() == W.size(0) && slot_age.numel() == S.size(0));
    FamilyBankView b{};
    b.W = W.data_ptr<float>(); b.age = reinterpret_cast<long long*>(age.data_ptr<int64_t>());
    b.S = S.data_ptr<float>(); b.slot_age = reinterpret_cast<long long*>(slot_age.data_ptr<int64_t>());
    b.Dp = (int)W.size(1);
    b.data = data.data_ptr<float>(); b.off = off.data_ptr<int64_t>(); b.cnt = cnt.data_ptr<int>();
    b.k = (int)k; b.dim = (int)dim; b.mode = (int)mode; b.hungarian = hungarian ? 1 : 0;
    b.alpha = (float)alpha; b.reg = (float)reg; b.lr = (float)lr;
    return b;
}
#define FAMILY_ARGS at::Tensor W, at::Tensor age, at::Tensor S, at::Tensor slot_age, at::Tensor data, at::Tensor off, \
                    at::Tensor cnt, int64_t k, int64_t dim, int64_t mode, bool hungarian, double alpha, double reg, double lr
#define FAMILY_PASS W, age, S, slot_age, data, off, cnt, k, dim, mode, hungarian, alpha, reg, lr
void family_snapshot(FAMILY_ARGS, at::Tensor sender, at::Tensor slot) {
    check_idx(sender); check_idx(slot);
    c10::cuda::CUDAGuard guard(W.device());
    launch_family_snapshot(family_view(FAMILY_PASS), sender.data_ptr<int>(), slot.data_ptr<int>(), (int)sender.numel(),
                           cur_stream());
    GB_LAUNCH_CHECK();
}
void kmeans_bank_deliver(FAMILY_ARGS, at::Tensor recv, at::Tensor slot) {
    check_idx(recv); check_idx(slot);
    TORCH_CHECK(k * dim <= W.size(1), "kmeans bank: row narrower than k * dim");
    c10::cuda::CUDAGuard guard(W.device());
    TORCH_CHECK(launch_kmeans_bank_deliver(family_view(FAMILY_PASS), recv.data_ptr<int>(), slot.data_ptr<int>(),
                                           (int)recv.numel(), cur_stream()),
                "kmeans bank: 1 <= k <= ", kFamilyMaxK, " (hungarian matching: k <= 8)");
    GB_LAUNCH_CHECK();
}
at::Tensor kmeans_bank_eval(FAMILY_ARGS, at::Tensor nodes, at::Tensor Xte, at::Tensor yte, int64_t n_true) {
    check_idx(nodes); check_row(Xte, "Xte");
    TORCH_CHECK(yte.is_cuda() && yte.scalar_type() == at::kLong && yte.is_contiguous() && yte.numel() == Xte.size(0));
    TORCH_CHECK(Xte.numel() == Xte.size(0) * dim);
    c10::cuda::CUDAGuard guard(W.device());
    auto ct = at::zeros({nodes.numel(), n_true, k}, W.options().dtype(at::kInt));
    launch_kmeans_bank_eval(family_view(FAMILY_PASS), nodes.data_ptr<int>(), (int)nodes.numel(), Xte.data_ptr<float>(),
                            yte.data_ptr<int64_t>(), (int)Xte.size(0), (int)n_true, ct.data_ptr<int>(), cur_stream());
    GB_LAUNCH_CHECK();
    return ct;
}
void mf_bank_deliver(FAMILY_ARGS, at::Tensor recv, at::Tensor slot) {
    check_idx(recv); check_idx(slot);
    TORCH_CHECK(dim * k + dim + k + 1 <= W.size(1), "mf bank: row narrower than [Y | c | X | b]");
    c10::cuda::CUDAGuard guard(W.device());
    TORCH_CHECK(launch_mf_bank_deliver(family_view(FAMILY_PASS), recv.data_ptr<int>(), slot.data_ptr<int>(),
                                       (int)recv.numel(), cur_stream()), "mf bank: rank <= 128 supported");
    GB_LAUNCH_CHECK();
}
at::Tensor mf_bank_eval(FAMILY_ARGS, at::Tensor nodes, at::Tensor te, at::Tensor te_off, at::Tensor te_cnt) {
    check_idx(nodes); check_idx(te_cnt);
    TORCH_CHECK(te.is_cuda() && te.scalar_type() == at::kFloat && te.is_contiguous());
    TORCH_CHECK(te_off.is_cuda() && te_off.scalar_type() == at::kLong && te_off.numel() == W.size(0) &&
                te_cnt.numel() == W.size(0));
    c10::cuda::CUDAGuard guard(W.device());
    auto sse = at::empty({nodes.numel()}, W.options());
    launch_mf_bank_eval(family_view(FAMILY_PASS), nodes.data_ptr<int>(), (int)nodes.numel(), te.data_ptr<float>(),
                        te_off.data_ptr<int64_t>(), te_cnt.data_ptr<int>(), sse.data_ptr<float>(), cur_stream());
    GB_LAUNCH_CHECK();
    return sse;
}

// ---- multi-process runtime: CUDA-IPC arenas and cross-GPU flags -----------------------------------------
// One process per GPU (torch.distributed only exchanges the 64-byte IPC handles).  Each rank
// cudaMalloc's its arena, exports it and maps every peer's arena; a peer row is then a device
// pointer that the merge / train kernels dereference (loads travel over NVLink / NVSwitch).
int64_t ipc_alloc(int64_t nbytes) {
    void* p = nullptr;
    C10_CUDA_CHECK(cudaMalloc(&p, (size_t)nbytes));
    C10_CUDA_CHECK(cudaMemset(p, 0, (size_t)nbytes));
    C10_CUDA_CHECK(cudaDeviceSynchronize());
    return (int64_t)(uintptr_t)p;
}
void ipc_free(int64_t ptr) { C10_CUDA_CHECK(cudaFree((void*)(uintptr_t)ptr)); }
pybind11::bytes ipc_get_handle(int64_t ptr) {
    cudaIpcMemHandle_t h;
    C10_CUDA_CHECK(cudaIpcGetMemHandle(&h, (void*)(uintptr_t)ptr));
    return pybind11::bytes(reinterpret_cast<const char*>(&h), sizeof(h));
}
int64_t ipc_open_handle(pybind11::bytes handle) {
    std::string s = handle;
    TORCH_CHECK(s.size() == sizeof(cudaIpcMemHandle_t), "bad IPC handle size");
    cudaIpcMemHandle_t h;
    memcpy(&h, s.data(), sizeof(h));
    void* p = nullptr;
    C10_CUDA_CHECK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    return (int64_t)(uintptr_t)p;
}
// one process, several visible GPUs (benchmarks / ncu captures of the peer kernels): let kernels on `dev` dereference
// cudaMalloc'ed memory of `peer`
void enable_peer_access(int64_t dev, int64_t peer) {
    c10::cuda::CUDAGuard guard((c10::DeviceIndex)dev);
    int can = 0;
    C10_CUDA_CHECK(cudaDeviceCanAccessPeer(&can, (int)dev, (int)peer));
    TORCH_CHECK(can, "device ", dev, " cannot access device ", peer);
    cudaError_t e = cudaDeviceEnablePeerAccess((int)peer, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
    else C10_CUDA_CHECK(e);
}
void ipc_close_handle(int64_t ptr) { C10_CUDA_CHECK(cudaIpcCloseMemHandle((void*)(uintptr_t)ptr)); }
at::Tensor tensor_from_ptr(int64_t ptr, std::vector<int64_t> sizes, int64_t device, bool as_int32) {
    auto opts = at::TensorOptions().device(at::kCUDA, (c10::DeviceIndex)device)
                    .dtype(as_int32 ? at::kInt : at::kFloat);
    return at::from_blob((void*)(uintptr_t)ptr, sizes, [](void*) {}, opts);
}
void flag_signal(int64_t flag_ptr, int64_t value) {
    launch_flag_signal((uint32_t*)(uintptr_t)flag_ptr, (uint32_t)value, cur_stream());
    GB_LAUNCH_CHECK();
}
void flag_wait(int64_t flag_ptr, int64_t value) {
    launch_flag_wait((const uint32_t*)(uintptr_t)flag_ptr, (uint32_t)value, cur_stream());
    GB_LAUNCH_CHECK();
}
void flag_add(int64_t flag_ptr, int64_t value) {
    launch_flag_add((uint32_t*)(uintptr_t)flag_ptr, (uint32_t)value, cur_stream());
    GB_LAUNCH_CHECK();
}
// one-shot all-reduce (mean) of symmetric buffers: NVLS multicast when mc_ptr != 0, P2P pull otherwise
void allreduce_mean(at::Tensor out, int64_t mc_ptr, std::vector<int64_t> buf_ptrs, std::vector<int64_t> flag_ptrs,
                    int64_t rank, int64_t epoch, double scale, int64_t n) {
    check_row(out, "out");
    const int world = (int)buf_ptrs.size();
    TORCH_CHECK(world >= 1 && world <= kMaxRanks && (int)flag_ptrs.size() == world && n <= out.numel());
    AllReduceArgs a{};
    a.mc = reinterpret_cast<const float*>((uintptr_t)mc_ptr);
    for (int r = 0; r < world; ++r) {
        a.bufs[r] = reinterpret_cast<const float*>((uintptr_t)buf_ptrs[r]);
        a.flags[r] = reinterpret_cast<uint32_t*>((uintptr_t)flag_ptrs[r]);
    }
    a.rank = (int)rank; a.world = world; a.epoch = (uint32_t)epoch; a.scale = (float)scale;
    c10::cuda::CUDAGuard guard(out.device());
    TORCH_CHECK(launch_allreduce_mean(out.data_ptr<float>(), a, n, cur_stream()), "allreduce_mean: bad arguments");
    GB_LAUNCH_CHECK();
}
int64_t device_sm_count() { return sm_count(); }
// the current device's fault word (bits: kernels.h) -- read (and cleared) with one small D2H copy; the simulator
// checks it whenever it reads a round's metrics
int64_t device_fault(bool clear) {
    uint32_t v = 0;
    uint32_t* w = device_fault_word();
    cudaMemcpy(&v, w, sizeof(v), cudaMemcpyDeviceToHost);
    if (clear && v != 0) cudaMemset(w, 0, sizeof(v));
    return (int64_t)v;
}
// pre-size the staging buffer of the CURRENT stream for the fused MLP training kernel (init_nodes)
bool reserve_mlp1_staging(int64_t n, int64_t in_dim, int64_t batch_size, int64_t local_epochs, std::string impl) {
    const int B = (int)(batch_size == 0 ? n : std::min<int64_t>(batch_size, n));
    const int nc = 8;
    const bool x3 = impl != "tc8-tf32";
    return reserve_train_staging((int)n, (int)in_dim, B, (int)local_epochs, nc, x3, cur_stream());
}
void preload() {
    preload_merge(); preload_optim(); preload_small(); preload_eval(); preload_train_cluster();
    preload_train_tc3(); preload_train_tc4(); preload_stage(); preload_nvls(); preload_eval_tc(); preload_bank();
    cudaGetLastError();
}

}  // namespace gb

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
    namespace py = pybind11;
    m.doc() = "gossipy_b200 sm_100a kernels + native scheduler";
    m.def("merge_pair", &gb::merge_pair, py::arg("dst"), py::arg("src"), py::arg("w_dst"), py::arg("w_src"),
          py::arg("lo"), py::arg("hi"), py::arg("sync") = py::none());
    m.def("merge_segments", &gb::merge_segments, py::arg("dst"), py::arg("src"), py::arg("seg"),
          py::arg("w_dst"), py::arg("w_src"), py::arg("sync") = py::none());
    m.def("merge_indexed", &gb::merge_indexed, py::arg("dst"), py::arg("src"), py::arg("idx"),
          py::arg("w_dst"), py::arg("w_src"), py::arg("sync") = py::none());
    m.def("merge_kway", &gb::merge_kway, py::arg("dst"), py::arg("srcs"), py::arg("weights"),
          py::arg("syncs") = py::none());
    m.def("sgd_step", &gb::sgd_step);
    m.def("adam_step", &gb::adam_step);
    m.def("keyed_perm", &gb::keyed_perm);
    m.def("keyed_randint", &gb::keyed_randint);
    m.def("mlp1_train", &gb::mlp1_train, py::arg("row"), py::arg("X"), py::arg("y"), py::arg("dims"),
          py::arg("batch_size"), py::arg("local_epochs"), py::arg("lr"), py::arg("wd"), py::arg("key"),
          py::arg("part_id") = py::none(), py::arg("ages") = py::none(), py::arg("impl") = "",
          py::arg("peer") = py::none(), py::arg("w_self") = 1.0, py::arg("w_peer") = 0.0,
          py::arg("sync") = py::none(), py::arg("momentum") = 0.0, py::arg("dampening") = 0.0, py::arg("nesterov") = false,
          py::arg("mom") = py::none(), py::arg("mom_first") = false);
    m.def("mlp1_train_tc_debug", &gb::mlp1_train_tc_debug, py::arg("row"), py::arg("X"), py::arg("y"),
          py::arg("dims"), py::arg("batch_size"), py::arg("local_epochs"), py::arg("lr"), py::arg("wd"),
          py::arg("key"), py::arg("impl") = "tc");
    m.def("mlp1_stage_debug", &gb::mlp1_stage_debug);
    m.def("mlp1_eval", &gb::mlp1_eval, py::arg("row"), py::arg("X"), py::arg("y"), py::arg("dims"), py::arg("n_classes"),
          py::arg("X_lp") = py::none(), py::arg("want_score1") = false);
    m.def("mlp1_eval_pretile", &gb::mlp1_eval_pretile);
    m.def("logreg_train", &gb::logreg_train, py::arg("row"), py::arg("X"), py::arg("y"), py::arg("dims"),
          py::arg("batch_size"), py::arg("local_epochs"), py::arg("lr"), py::arg("wd"), py::arg("key"),
          py::arg("part_id") = py::none(), py::arg("ages") = py::none(), py::arg("peer") = py::none(),
          py::arg("w_self") = 1.0, py::arg("w_peer") = 0.0, py::arg("sync") = py::none());
    m.def("logreg_scores", &gb::logreg_scores);
    m.def("linear_seq_update", &gb::linear_seq_update);
    m.def("kmeans_update", &gb::kmeans_update);
    m.def("kmeans_assign", &gb::kmeans_assign);
    m.def("mf_update", &gb::mf_update);
    m.def("kmeans_match_merge", &gb::kmeans_match_merge, py::arg("C"), py::arg("P"), py::arg("k"), py::arg("dim"),
          py::arg("w_own"), py::arg("w_peer"), py::arg("sync") = py::none());
    m.def("bank_snapshot", &gb::bank_snapshot);
    m.def("bank_deliver", &gb::bank_deliver, py::arg("W"), py::arg("age"), py::arg("S"), py::arg("slot_age"), py::arg("X"), py::arg("y"),
          py::arg("off"), py::arg("cnt"), py::arg("D"), py::arg("kind"), py::arg("mode"), py::arg("lr"), py::arg("recv"), py::arg("slot"),
          py::arg("item_mode") = py::none());
    m.def("bank_update", &gb::bank_update);
    m.def("bank_scores", &gb::bank_scores);
    m.def("family_snapshot", &gb::family_snapshot);
    m.def("kmeans_bank_deliver", &gb::kmeans_bank_deliver);
    m.def("kmeans_bank_eval", &gb::kmeans_bank_eval);
    m.def("mf_bank_deliver", &gb::mf_bank_deliver);
    m.def("mf_bank_eval", &gb::mf_bank_eval);
    m.def("ipc_alloc", &gb::ipc_alloc);
    m.def("ipc_free", &gb::ipc_free);
    m.def("ipc_get_handle", &gb::ipc_get_handle);
    m.def("ipc_open_handle", &gb::ipc_open_handle);
    m.def("ipc_close_handle", &gb::ipc_close_handle);
    m.def("enable_peer_access", &gb::enable_peer_access);
    m.def("tensor_from_ptr", &gb::tensor_from_ptr);
    m.def("bank_snapshot_push", &gb::bank_snapshot_push);
    m.def("rank_barrier", &gb::rank_barrier);
    m.def("flag_signal", &gb::flag_signal);
    m.def("flag_wait", &gb::flag_wait);
    m.def("flag_add", &gb::flag_add);
    m.def("device_sm_count", &gb::device_sm_count);
    m.def("preload", &gb::preload);
    m.def("device_fault", &gb::device_fault, py::arg("clear") = true);
    m.def("set_train_impl", &gb::set_train_impl);
    m.def("set_eval_tf32", &gb::set_eval_tf32);
    m.def("reserve_mlp1_staging", &gb::reserve_mlp1_staging);
    m.def("allreduce_mean", &gb::allreduce_mean);
    gb::bind_scheduler(m);
    gb::bind_executor(m);
}
