// Batched kernels for the k-means and matrix-factorisation families: MANY gossip nodes per launch.
//
// Same scheme as bank.cu (all nodes' models in one bank W[N][Dp], in-flight snapshots in S[slots][Dp], one launch
// per phase of a simulated tick over a work list from the native scheduler), but one CTA per work item: an MF row
// is [Y (n_items*k) | c (n_items) | X (k) | b (1)], about 22 k floats at ml-1m, far past what a warp keeps in
// registers.  The merge is CTA-wide; the local update, which is sequential in the samples / ratings, runs on one
// warp (k-means: the assignments of all samples are independent and spread over the CTA's warps).
// Semantics: KMeansHandler / MFModelHandler (model/handler.py) and the per-node kernels of small.cu, whose
// arithmetic is reproduced operation for operation (distance order, tie rules, update order).
#include "common.cuh"
#include "kernels.h"
#include <algorithm>

namespace gb {

constexpr int FB_THREADS = 256;
constexpr int FB_WARPS = FB_THREADS / 32;

// ---- rows ------------------------------------------------------------------------------------------------
GB_DEVICE void fb_copy_row(float* __restrict__ dst, const float* __restrict__ src, int Dp) {
    // rows are Dp floats with Dp a multiple of 32: 128-byte aligned, whole float4s
    const float4* s4 = reinterpret_cast<const float4*>(src);
    float4* d4 = reinterpret_cast<float4*>(dst);
    for (int i = threadIdx.x; i < Dp / 4; i += FB_THREADS) d4[i] = s4[i];
}

// snapshot of rows wider than the warp-per-item kernel of bank.cu covers: S[slot] = W[sender], one CTA per item
__global__ void __launch_bounds__(FB_THREADS)
bank_snapshot_wide_kernel(const FamilyBankView b, const int* __restrict__ sender, const int* __restrict__ slot, int n) {
    const int item = blockIdx.x;
    if (item >= n) return;
    const int s = sender[item], d = slot[item];
    if (d < 0) return;                          // PULL request: nothing travels
    fb_copy_row(b.S + (size_t)d * b.Dp, b.W + (size_t)s * b.Dp, b.Dp);
    if (threadIdx.x == 0) b.slot_age[d] = b.age[s];
}

// ---- k-means -----------------------------------------------------------------------------------------------
// index of the first centroid with the strictly smallest squared distance (kmeans_assign_kernel's order: lanes
// stride the dimensions, fmaf accumulation, butterfly warp sum); called by a whole warp
GB_DEVICE int fb_nearest(const float* __restrict__ C, const float* __restrict__ x, int k, int dim, int lane) {
    int best = 0; float bd = 3.4e38f;
    for (int c = 0; c < k; ++c) {
        float acc = 0.f;
        for (int d = lane; d < dim; d += 32) { const float df = x[d] - C[c * dim + d]; acc = fmaf(df, df, acc); }
        acc = gb_warp_sum(acc);
        if (acc < bd) { bd = acc; best = c; }
    }
    return best;
}

// the node's local batch: all samples assigned against the incoming centroids, then for every centroid the
// highest-index sample assigned to it moves it by the EMA step (kmeans_assign_kernel + kmeans_apply_kernel)
GB_DEVICE void fb_kmeans_update(float* C, const FamilyBankView& b, int node, int* winner) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t o = b.off[node];
    const int n = b.cnt[node], k = b.k, dim = b.dim;
    for (int c = tid; c < k; c += FB_THREADS) winner[c] = -1;
    __syncthreads();
    for (int s = warp; s < n; s += FB_WARPS) {
        const int best = fb_nearest(C, b.data + (size_t)(o + s) * dim, k, dim, lane);
        if (lane == 0) atomicMax(&winner[best], s);
    }
    __syncthreads();
    for (int e = tid; e < k * dim; e += FB_THREADS) {
        const int c = e / dim, d = e - c * dim;
        const int s = winner[c];
        if (s >= 0) C[e] = C[e] * (1.f - b.alpha) + b.alpha * b.data[(size_t)(o + s) * dim + d];
    }
    __syncthreads();
}

struct FbMatch {                                // shared scratch of the optimal matching
    float cost[64];
    unsigned long long best;
    int perm[8];
};

// C = 0.5 C + 0.5 P, with P's centroids permuted by the optimal assignment when `hungarian` (k <= 8): the summed
// Euclidean distance of all k! permutations, ties to the lexicographically smallest (kmeans_match_merge_kernel)
GB_DEVICE void fb_kmeans_merge(float* C, const float* P, const FamilyBankView& b, FbMatch& m) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int k = b.k, dim = b.dim;
    if (!b.hungarian) {
        for (int e = tid; e < k * dim; e += FB_THREADS) C[e] = 0.5f * C[e] + 0.5f * P[e];
        __syncthreads();
        return;
    }
    if (tid == 0) m.best = ~0ull;
    for (int e = warp; e < k * k; e += FB_WARPS) {
        const int i = e / k, j = e % k;
        float acc = 0.f;
        for (int d = lane; d < dim; d += 32) { const float df = C[i * dim + d] - P[j * dim + d]; acc = fmaf(df, df, acc); }
        acc = gb_warp_sum(acc);
        if (lane == 0) m.cost[i * 8 + j] = sqrtf(acc);
    }
    __syncthreads();
    int nperm = 1;
    for (int i = 2; i <= k; ++i) nperm *= i;
    for (int pi = tid; pi < nperm; pi += FB_THREADS) {
        int avail[8], idx = pi, fact = nperm;
#pragma unroll
        for (int i = 0; i < 8; ++i) avail[i] = i;
        float total = 0.f;
        for (int i = 0; i < k; ++i) {            // factoradic digits, most significant first: lexicographic order
            fact /= (k - i);
            const int dgt = idx / fact; idx -= dgt * fact;
            const int col = avail[dgt];
            for (int t = dgt; t < k - i - 1; ++t) avail[t] = avail[t + 1];
            total += m.cost[i * 8 + col];
        }
        atomicMin(&m.best, ((unsigned long long)__float_as_uint(total) << 32) | (unsigned)pi);
    }
    __syncthreads();
    if (tid == 0) {
        int avail[8], idx = (int)(m.best & 0xffffffffull), fact = nperm;
        for (int i = 0; i < 8; ++i) avail[i] = i;
        for (int i = 0; i < k; ++i) {
            fact /= (k - i);
            const int dgt = idx / fact; idx -= dgt * fact;
            m.perm[i] = avail[dgt];
            for (int t = dgt; t < k - i - 1; ++t) avail[t] = avail[t + 1];
        }
    }
    __syncthreads();
    for (int e = tid; e < k * dim; e += FB_THREADS) {
        const int i = e / dim, d = e - i * dim;
        C[e] = 0.5f * C[e] + 0.5f * P[m.perm[i] * dim + d];
    }
    __syncthreads();
}

// deliver: node recv[i] consumes snapshot slot[i] according to the CreateModelMode.  Ages as KMeansHandler:
// a local update adds 1, the merge leaves them alone, UPDATE adopts the sender's.
__global__ void __launch_bounds__(FB_THREADS)
kmeans_bank_deliver_kernel(const FamilyBankView b, const int* __restrict__ recv, const int* __restrict__ slot, int n) {
    __shared__ int winner[kFamilyMaxK];
    __shared__ FbMatch match;
    const int item = blockIdx.x;
    if (item >= n) return;
    const int r = recv[item], s = slot[item];
    if (s < 0) return;                          // PULL request delivered: the receiver only replies
    float* w = b.W + (size_t)r * b.Dp;
    float* sv = b.S + (size_t)s * b.Dp;         // consumed by this delivery only: UPDATE_MERGE trains it in place
    long long aw = b.age[r];
    switch (b.mode) {
        case 1:                                 // UPDATE: adopt the received model and train it
            fb_copy_row(w, sv, b.Dp);
            __syncthreads();
            aw = b.slot_age[s] + 1;
            fb_kmeans_update(w, b, r, winner);
            break;
        case 2:                                 // MERGE_UPDATE
            fb_kmeans_merge(w, sv, b, match);
            fb_kmeans_update(w, b, r, winner);
            aw += 1;
            break;
        case 3:                                 // UPDATE_MERGE: both train on the local batch, then merge
            fb_kmeans_update(w, b, r, winner);
            fb_kmeans_update(sv, b, r, winner);
            fb_kmeans_merge(w, sv, b, match);
            aw += 1;
            break;
        default:                                // PASS: adopt untouched, age unchanged
            fb_copy_row(w, sv, b.Dp);
            break;
    }
    if (threadIdx.x == 0) b.age[r] = aw;
}

// evaluation: ct[e][y][c] += 1 for every sample of the shared set (label y, nearest centroid c of node nodes[e]);
// grid (sample chunks, evaluated nodes), one warp per sample
__global__ void __launch_bounds__(FB_THREADS)
kmeans_bank_eval_kernel(const FamilyBankView b, const int* __restrict__ nodes, const float* __restrict__ Xte,
                        const int64_t* __restrict__ yte, int n_te, int n_true, int* __restrict__ ct) {
    const int e = blockIdx.y, lane = threadIdx.x & 31;
    const float* C = b.W + (size_t)nodes[e] * b.Dp;
    int* cte = ct + (size_t)e * n_true * b.k;
    for (int t = blockIdx.x * FB_WARPS + (threadIdx.x >> 5); t < n_te; t += gridDim.x * FB_WARPS) {
        const int best = fb_nearest(C, Xte + (size_t)t * b.dim, b.k, b.dim, lane);
        if (lane == 0) atomicAdd(&cte[(int)yte[t] * b.k + best], 1);
    }
}

// ---- matrix factorisation ----------------------------------------------------------------------------------
// row layout [Y (m*k) | c (m) | X (k) | b (1)], m = b.dim items
// sequential rank-k SGD over the node's ratings, executed by ONE warp (mf_update_kernel: lanes = factors, the item
// factor is updated first and the user factor uses the new one)
GB_DEVICE void fb_mf_update(float* row, const FamilyBankView& b, int node, int lane) {
    const int k = b.k, m = b.dim;
    float* Y = row;
    float* c = row + (size_t)m * k;
    float* Xu = c + m;
    float* bu = Xu + k;
    const float* ratings = b.data + 2 * b.off[node];
    const int nr = b.cnt[node];
    const int kpl = (k + 31) / 32;              // k <= 128
    float x[4], bb = bu[0];
    for (int i = 0; i < 4; ++i) { const int f = i * 32 + lane; x[i] = (i < kpl && f < k) ? Xu[f] : 0.f; }
    const float decay = 1.f - b.reg * b.lr;
    for (int r = 0; r < nr; ++r) {
        const int item = (int)ratings[2 * r];
        const float rating = ratings[2 * r + 1];
        float yv[4], acc = 0.f;
        for (int i = 0; i < 4; ++i) {
            const int f = i * 32 + lane;
            yv[i] = (i < kpl && f < k) ? Y[(size_t)item * k + f] : 0.f;
            acc = fmaf(x[i], yv[i], acc);
        }
        const float ci = c[item];
        const float err = rating - gb_warp_sum(acc) - bb - ci;
        for (int i = 0; i < 4; ++i) {
            const int f = i * 32 + lane;
            if (i < kpl && f < k) {
                const float ynew = decay * yv[i] + b.lr * err * x[i];
                x[i] = decay * x[i] + b.lr * err * ynew;
                Y[(size_t)item * k + f] = ynew;
            }
        }
        bb += b.lr * err;
        if (lane == 0) c[item] = ci + b.lr * err;
        __syncwarp();
    }
    for (int i = 0; i < 4; ++i) { const int f = i * 32 + lane; if (i < kpl && f < k) Xu[f] = x[i]; }
    if (lane == 0) bu[0] = bb;
}

// shared prefix [Y | c] = wa * own + wb * peer, wa = a / (2 (a+b)), wb = b / (2 (a+b)) with the ages a, b
// (MFModelHandler._merge, whose weights the host computes in double before the fp32 merge)
GB_DEVICE void fb_mf_merge(float* __restrict__ w, const float* __restrict__ p, long long a, long long bage,
                           const FamilyBankView& b) {
    const double den = 2.0 * (double)(a + bage);
    const float wa = (float)((double)a / den), wb = (float)((double)bage / den);
    const int n_shared = b.dim * b.k + b.dim;
    const int nvec = n_shared / 4;
    float4* w4 = reinterpret_cast<float4*>(w);
    const float4* p4 = reinterpret_cast<const float4*>(p);
    for (int i = threadIdx.x; i < nvec; i += FB_THREADS) {
        const float4 d = w4[i], s = p4[i];
        float4 o;
        o.x = (wa == 0.f ? 0.f : wa * d.x) + wb * s.x; o.y = (wa == 0.f ? 0.f : wa * d.y) + wb * s.y;
        o.z = (wa == 0.f ? 0.f : wa * d.z) + wb * s.z; o.w = (wa == 0.f ? 0.f : wa * d.w) + wb * s.w;
        w4[i] = o;
    }
    for (int i = nvec * 4 + threadIdx.x; i < n_shared; i += FB_THREADS) w[i] = (wa == 0.f ? 0.f : wa * w[i]) + wb * p[i];
    __syncthreads();
}

// deliver: ages as MFModelHandler: a local update adds the number of ratings, the merge leaves them alone,
// UPDATE adopts the sender's
__global__ void __launch_bounds__(FB_THREADS)
mf_bank_deliver_kernel(const FamilyBankView b, const int* __restrict__ recv, const int* __restrict__ slot, int n) {
    const int item = blockIdx.x;
    if (item >= n) return;
    const int r = recv[item], s = slot[item];
    if (s < 0) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* w = b.W + (size_t)r * b.Dp;
    float* sv = b.S + (size_t)s * b.Dp;         // consumed by this delivery only: UPDATE_MERGE's scratch copy
    const long long nr = b.cnt[r];
    long long aw = b.age[r];
    const long long as = b.slot_age[s];
    switch (b.mode) {
        case 1:                                 // UPDATE
            fb_copy_row(w, sv, b.Dp);
            __syncthreads();
            if (warp == 0) fb_mf_update(w, b, r, lane);
            aw = as + nr;
            break;
        case 2:                                 // MERGE_UPDATE
            fb_mf_merge(w, sv, aw, as, b);
            if (warp == 0) fb_mf_update(w, b, r, lane);
            aw += nr;
            break;
        case 3:                                 // UPDATE_MERGE: the two rows train concurrently, then merge
            if (warp == 0) fb_mf_update(w, b, r, lane);
            else if (warp == 1) fb_mf_update(sv, b, r, lane);
            __syncthreads();
            fb_mf_merge(w, sv, aw + nr, as + nr, b);
            aw += nr;
            break;
        default:                                // PASS
            fb_copy_row(w, sv, b.Dp);
            break;
    }
    if (threadIdx.x == 0) b.age[r] = aw;
}

// evaluation: sse[e] = sum of squared errors of node nodes[e] on its own test ratings (one warp per node;
// prediction Y[item] . X + b + c[item] as MFModelHandler.evaluate_async)
__global__ void __launch_bounds__(FB_THREADS)
mf_bank_eval_kernel(const FamilyBankView b, const int* __restrict__ nodes, int n_nodes, const float* __restrict__ te,
                    const int64_t* __restrict__ te_off, const int* __restrict__ te_cnt, float* __restrict__ sse) {
    const int e = blockIdx.x * FB_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (e >= n_nodes) return;
    const int node = nodes[e];
    const int k = b.k, m = b.dim;
    const float* Y = b.W + (size_t)node * b.Dp;
    const float* c = Y + (size_t)m * k;
    const float* Xu = c + m;
    const float bu = Xu[k];
    const int kpl = (k + 31) / 32;
    float x[4];
    for (int i = 0; i < 4; ++i) { const int f = i * 32 + lane; x[i] = (i < kpl && f < k) ? Xu[f] : 0.f; }
    const float* rt = te + 2 * te_off[node];
    float acc_sq = 0.f;
    for (int r = 0; r < te_cnt[node]; ++r) {
        const int item = (int)rt[2 * r];
        float acc = 0.f;
        for (int i = 0; i < 4; ++i) {
            const int f = i * 32 + lane;
            acc = fmaf(x[i], (i < kpl && f < k) ? Y[(size_t)item * k + f] : 0.f, acc);
        }
        const float err = rt[2 * r + 1] - (gb_warp_sum(acc) + bu + c[item]);
        acc_sq = fmaf(err, err, acc_sq);
    }
    if (lane == 0) sse[e] = acc_sq;
}

// ---- launchers ----------------------------------------------------------------------------------------------
void launch_family_snapshot(const FamilyBankView& b, const int* sender, const int* slot, int n, cudaStream_t st) {
    if (n <= 0) return;
    if (b.Dp <= 1024) {                         // narrow rows: the warp-per-item kernel of the linear bank
        BankView v{};
        v.W = b.W; v.age = b.age; v.S = b.S; v.slot_age = b.slot_age; v.D = b.Dp; v.Dp = b.Dp;
        launch_bank_snapshot(v, sender, slot, n, st);
        return;
    }
    bank_snapshot_wide_kernel<<<n, FB_THREADS, 0, st>>>(b, sender, slot, n);
}
bool launch_kmeans_bank_deliver(const FamilyBankView& b, const int* recv, const int* slot, int n, cudaStream_t st) {
    if (b.k < 1 || b.k > kFamilyMaxK || (b.hungarian && b.k > 8)) return false;
    if (n > 0) kmeans_bank_deliver_kernel<<<n, FB_THREADS, 0, st>>>(b, recv, slot, n);
    return true;
}
void launch_kmeans_bank_eval(const FamilyBankView& b, const int* nodes, int n_nodes, const float* Xte, const int64_t* yte,
                             int n_te, int n_true, int* ct, cudaStream_t st) {
    if (n_nodes <= 0 || n_te <= 0) return;
    const int chunks = std::max(1, std::min((n_te + FB_WARPS - 1) / FB_WARPS, 64));
    kmeans_bank_eval_kernel<<<dim3(chunks, n_nodes), FB_THREADS, 0, st>>>(b, nodes, Xte, yte, n_te, n_true, ct);
}
bool launch_mf_bank_deliver(const FamilyBankView& b, const int* recv, const int* slot, int n, cudaStream_t st) {
    if (b.k < 1 || b.k > 128) return false;
    if (n > 0) mf_bank_deliver_kernel<<<n, FB_THREADS, 0, st>>>(b, recv, slot, n);
    return true;
}
void launch_mf_bank_eval(const FamilyBankView& b, const int* nodes, int n_nodes, const float* te, const int64_t* te_off,
                         const int* te_cnt, float* sse, cudaStream_t st) {
    if (n_nodes <= 0) return;
    mf_bank_eval_kernel<<<(n_nodes + FB_WARPS - 1) / FB_WARPS, FB_THREADS, 0, st>>>(b, nodes, n_nodes, te, te_off, te_cnt, sse);
}

void preload_bank_families() {
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, bank_snapshot_wide_kernel);
    cudaFuncGetAttributes(&a, kmeans_bank_deliver_kernel);
    cudaFuncGetAttributes(&a, kmeans_bank_eval_kernel);
    cudaFuncGetAttributes(&a, mf_bank_deliver_kernel);
    cudaFuncGetAttributes(&a, mf_bank_eval_kernel);
}

}  // namespace gb
