// Batched kernels for the linear learners (AdaLine / Pegasos): MANY gossip nodes per launch.
//
// The reference's own experiment scripts for these models run one node per training sample
// (4 141 nodes for spambase, main_ormandi_2013.py / main_giaretta_2019.py); a node's model is a
// 57-float vector and its local update a handful of dot products -- per-node launches would be pure
// launch latency.  Here all nodes' models live in one bank W[N][Dp] (ages in age[N]), in-flight
// snapshots in a second bank S[slots][Dp], and every phase of a simulated tick is ONE launch over a
// work list produced by the native scheduler: one warp per work item, the model in registers,
// the node's samples streamed in order (the updates are strictly sequential in t).
// Semantics: gossipy/model/handler.py:117-136 (modes), :364-373 (AdaLine), :416-423 (Pegasos).
#include "common.cuh"
#include "kernels.h"

namespace gb {

constexpr int BK_WARPS = 4;

template <int KPL>
GB_DEVICE void bank_update(float (&w)[KPL], long long& age, const BankView& b, int node, int lane) {
    const int64_t o = b.off[node];
    const int c = b.cnt[node];
    for (int i = 0; i < c; ++i) {
        const float* x = b.X + (size_t)(o + i) * b.D;
        float xr[KPL];
        float acc = 0.f;
#pragma unroll
        for (int q = 0; q < KPL; ++q) {
            const int k = q * 32 + lane;
            xr[q] = k < b.D ? x[k] : 0.f;
            acc = fmaf(w[q], xr[q], acc);
        }
        const float yhat = gb_warp_sum(acc);
        const float ys = b.y[o + i];
        if (b.kind == 0) {                     // AdaLine: w += lr (y - w.x) x
            const float cf = b.lr * (ys - yhat);
#pragma unroll
            for (int q = 0; q < KPL; ++q) w[q] = fmaf(cf, xr[q], w[q]);
            age += 1;
        } else {                               // Pegasos: t = ++age; eta = 1/(t lam); w *= (1 - eta lam); hinge step
            age += 1;
            const float eta = 1.f / ((float)age * b.lr);
            const float sc = 1.f - eta * b.lr;
            const float cf = (yhat * ys - 1.f < 0.f) ? eta * ys : 0.f;
#pragma unroll
            for (int q = 0; q < KPL; ++q) w[q] = fmaf(cf, xr[q], w[q] * sc);
        }
    }
}

// snapshot: S[slot] = W[sender], slot_age = age[sender]
__global__ void __launch_bounds__(BK_WARPS * 32)
bank_snapshot_kernel(const BankView b, const int* __restrict__ sender, const int* __restrict__ slot, int n) {
    const int item = blockIdx.x * BK_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (item >= n) return;
    const int s = sender[item], d = slot[item];
    if (d < 0) return;                          // PULL request: nothing travels
    for (int k = lane; k < b.Dp; k += 32) b.S[(size_t)d * b.Dp + k] = b.W[(size_t)s * b.Dp + k];
    if (lane == 0) b.slot_age[d] = b.age[s];
}

// several ranks: S[slot] of the RECEIVER's rank = W[sender] (stores travel over NVLink / NVSwitch; the next
// rank_barrier_kernel publishes them)
__global__ void __launch_bounds__(BK_WARPS * 32)
bank_snapshot_push_kernel(const BankView b, const BankPeers peers, const int* __restrict__ sender,
                          const int* __restrict__ slot, const int* __restrict__ dst_rank, int n) {
    const int item = blockIdx.x * BK_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (item >= n) return;
    const int s = sender[item], d = slot[item];
    if (d < 0) return;
    float* S = peers.S[dst_rank[item]];
    for (int k = lane; k < b.Dp; k += 32) S[(size_t)d * b.Dp + k] = b.W[(size_t)s * b.Dp + k];
    if (lane == 0) peers.slot_age[dst_rank[item]][d] = b.age[s];
}

// barrier across the ranks of the job, stream ordered: everything this rank's earlier kernels wrote (also into peers'
// memory) is visible to every rank's later kernels.  One generation word per (rank, peer); bounded wait (fault bit 8).
__global__ void rank_barrier_kernel(const RankBarrier rb, uint32_t* fault) {
    const int t = threadIdx.x;
    __threadfence_system();
    if (t < rb.world) gb_st_release_sys(rb.flags[t] + rb.rank, rb.gen);
    if (t < rb.world) gb_wait_flag(rb.flags[rb.rank] + t, rb.gen, fault, 8u);
}

// deliver: node recv[i] consumes snapshot slot[i] according to the CreateModelMode
template <int KPL>
__global__ void __launch_bounds__(BK_WARPS * 32)
bank_deliver_kernel(const BankView b, const int* __restrict__ recv, const int* __restrict__ slot,
                    const int* __restrict__ item_mode, int n) {
    const int item = blockIdx.x * BK_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (item >= n) return;
    const int r = recv[item], s = slot[item];
    if (s < 0) return;                          // PULL request delivered: the receiver only replies
    // PassThroughNode: the receiver either merges (the bank's mode) or adopts the model untouched (PASS), decided per
    // message by a keyed draw on the host
    const int mode = item_mode != nullptr ? item_mode[item] : b.mode;
    float w[KPL], sv[KPL];
#pragma unroll
    for (int q = 0; q < KPL; ++q) {
        const int k = q * 32 + lane;
        w[q] = k < b.D ? b.W[(size_t)r * b.Dp + k] : 0.f;
        sv[q] = k < b.D ? b.S[(size_t)s * b.Dp + k] : 0.f;
    }
    long long aw = b.age[r], as = b.slot_age[s];
    switch (mode) {
        case 1:                                 // UPDATE: train the received model and adopt it
#pragma unroll
            for (int q = 0; q < KPL; ++q) w[q] = sv[q];
            aw = as;
            bank_update<KPL>(w, aw, b, r, lane);
            break;
        case 2:                                 // MERGE_UPDATE
#pragma unroll
            for (int q = 0; q < KPL; ++q) w[q] = 0.5f * (w[q] + sv[q]);
            aw = aw > as ? aw : as;
            bank_update<KPL>(w, aw, b, r, lane);
            break;
        case 3:                                 // UPDATE_MERGE: both models train on the local data, then merge
            bank_update<KPL>(w, aw, b, r, lane);
            bank_update<KPL>(sv, as, b, r, lane);
#pragma unroll
            for (int q = 0; q < KPL; ++q) w[q] = 0.5f * (w[q] + sv[q]);
            aw = aw > as ? aw : as;
            break;
        default:                                // PASS: adopt untouched, age unchanged
#pragma unroll
            for (int q = 0; q < KPL; ++q) w[q] = sv[q];
            break;
    }
#pragma unroll
    for (int q = 0; q < KPL; ++q) {
        const int k = q * 32 + lane;
        if (k < b.D) b.W[(size_t)r * b.Dp + k] = w[q];
    }
    if (lane == 0) b.age[r] = aw;
}

// local update of a list of nodes (init_nodes: every node trains once on its own data)
template <int KPL>
__global__ void __launch_bounds__(BK_WARPS * 32)
bank_update_kernel(const BankView b, const int* __restrict__ nodes, int n) {
    const int item = blockIdx.x * BK_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (item >= n) return;
    const int r = nodes[item];
    float w[KPL];
#pragma unroll
    for (int q = 0; q < KPL; ++q) { const int k = q * 32 + lane; w[q] = k < b.D ? b.W[(size_t)r * b.Dp + k] : 0.f; }
    long long aw = b.age[r];
    bank_update<KPL>(w, aw, b, r, lane);
#pragma unroll
    for (int q = 0; q < KPL; ++q) { const int k = q * 32 + lane; if (k < b.D) b.W[(size_t)r * b.Dp + k] = w[q]; }
    if (lane == 0) b.age[r] = aw;
}

// evaluation scores of a list of nodes on a shared test set: scores[e][t] = Xte[t] . W[nodes[e]]
__global__ void __launch_bounds__(256)
bank_scores_kernel(const BankView b, const int* __restrict__ nodes, int n_nodes, const float* __restrict__ Xte,
                   int n_te, float* __restrict__ scores) {
    extern __shared__ float wsh[];
    const int e = blockIdx.x;
    if (e >= n_nodes) return;
    const int node = nodes[e];
    for (int k = threadIdx.x; k < b.D; k += blockDim.x) wsh[k] = b.W[(size_t)node * b.Dp + k];
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int t = warp; t < n_te; t += nw) {
        float acc = 0.f;
        for (int k = lane; k < b.D; k += 32) acc = fmaf(wsh[k], Xte[(size_t)t * b.D + k], acc);
        acc = gb_warp_sum(acc);
        if (lane == 0) scores[(size_t)e * n_te + t] = acc;
    }
}

template <int KPL>
static void deliver_t(const BankView& b, const int* recv, const int* slot, const int* item_mode, int n, cudaStream_t st) {
    bank_deliver_kernel<KPL><<<(n + BK_WARPS - 1) / BK_WARPS, BK_WARPS * 32, 0, st>>>(b, recv, slot, item_mode, n);
}
template <int KPL>
static void update_t(const BankView& b, const int* nodes, int n, cudaStream_t st) {
    bank_update_kernel<KPL><<<(n + BK_WARPS - 1) / BK_WARPS, BK_WARPS * 32, 0, st>>>(b, nodes, n);
}

void launch_bank_snapshot(const BankView& b, const int* sender, const int* slot, int n, cudaStream_t st) {
    if (n <= 0) return;
    bank_snapshot_kernel<<<(n + BK_WARPS - 1) / BK_WARPS, BK_WARPS * 32, 0, st>>>(b, sender, slot, n);
}
void launch_bank_snapshot_push(const BankView& b, const BankPeers& peers, const int* sender, const int* slot,
                               const int* dst_rank, int n, cudaStream_t st) {
    if (n <= 0) return;
    bank_snapshot_push_kernel<<<(n + BK_WARPS - 1) / BK_WARPS, BK_WARPS * 32, 0, st>>>(b, peers, sender, slot, dst_rank, n);
}
void launch_rank_barrier(const RankBarrier& rb, cudaStream_t st) {
    rank_barrier_kernel<<<1, 32, 0, st>>>(rb, device_fault_word());
}
bool launch_bank_deliver(const BankView& b, const int* recv, const int* slot, const int* item_mode, int n, cudaStream_t st) {
    if (n <= 0) return true;
    if (b.D <= 64) deliver_t<2>(b, recv, slot, item_mode, n, st);
    else if (b.D <= 128) deliver_t<4>(b, recv, slot, item_mode, n, st);
    else if (b.D <= 256) deliver_t<8>(b, recv, slot, item_mode, n, st);
    else if (b.D <= 1024) deliver_t<32>(b, recv, slot, item_mode, n, st);
    else return false;
    return true;
}
bool launch_bank_update(const BankView& b, const int* nodes, int n, cudaStream_t st) {
    if (n <= 0) return true;
    if (b.D <= 64) update_t<2>(b, nodes, n, st);
    else if (b.D <= 128) update_t<4>(b, nodes, n, st);
    else if (b.D <= 256) update_t<8>(b, nodes, n, st);
    else if (b.D <= 1024) update_t<32>(b, nodes, n, st);
    else return false;
    return true;
}
void launch_bank_scores(const BankView& b, const int* nodes, int n_nodes, const float* Xte, int n_te, float* scores,
                        cudaStream_t st) {
    if (n_nodes <= 0 || n_te <= 0) return;
    bank_scores_kernel<<<n_nodes, 256, b.D * sizeof(float), st>>>(b, nodes, n_nodes, Xte, n_te, scores);
}

void preload_bank() {
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, bank_snapshot_kernel);
    cudaFuncGetAttributes(&a, bank_snapshot_push_kernel);
    cudaFuncGetAttributes(&a, rank_barrier_kernel);
    cudaFuncGetAttributes(&a, bank_deliver_kernel<2>); cudaFuncGetAttributes(&a, bank_deliver_kernel<4>);
    cudaFuncGetAttributes(&a, bank_deliver_kernel<8>); cudaFuncGetAttributes(&a, bank_deliver_kernel<32>);
    cudaFuncGetAttributes(&a, bank_update_kernel<2>); cudaFuncGetAttributes(&a, bank_update_kernel<4>);
    cudaFuncGetAttributes(&a, bank_update_kernel<8>); cudaFuncGetAttributes(&a, bank_update_kernel<32>);
    cudaFuncGetAttributes(&a, bank_scores_kernel);
    preload_bank_families();
}

}  // namespace gb
