// Launchers of the gossipy_b200 sm_100a kernels.  Plain CUDA/C++ (no torch headers): every function
// enqueues on `stream` and returns; errors are reported through cudaGetLastError() by the caller
// (csrc/bindings.cpp).  Pointers are device pointers of the CURRENT device unless stated otherwise;
// "peer" pointers may point into another GPU's HBM (mapped with CUDA IPC / peer access).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace gb {

// ---- cross-GPU row handshake (see kernels/common.cuh, parallel/runtime.py) ---------------------
// A kernel that READS a row owned by another GPU first spins until *ready >= gen (the owner
// publishes the generation after the producing kernel) and, when it is done with the row, adds 1
// to *done (the owner waits for it before the row is recycled).  Null pointers disable each side.
struct PeerSync {
    const uint32_t* ready;   // flag in the OWNER's memory (may be peer-mapped)
    uint32_t gen;
    uint32_t* done;          // read counter in the OWNER's memory (may be peer-mapped)
    uint32_t* fault;         // this device's fault word (bounded waits report here; see device_fault_word())
};
// one word per device, zero-initialised; bit 1: a wait for a `ready` generation timed out, bit 2: an all-reduce
// epoch wait timed out, bit 4: the ticket ring of the stand-alone flag operations overflowed
uint32_t* device_fault_word();

// ---- merge.cu ------------------------------------------------------------------------------------
void launch_merge_pair(float* dst, const float* src, float w_dst, float w_src, int64_t lo, int64_t hi,
                       PeerSync sync, cudaStream_t stream);
void launch_merge_segments(float* dst, const float* src, const int64_t* seg, int n_seg, float w_dst,
                           float w_src, PeerSync sync, cudaStream_t stream);
void launch_merge_indexed(float* dst, const float* src, const int64_t* idx, int64_t n, float w_dst,
                          float w_src, float* scratch, PeerSync sync, cudaStream_t stream);
constexpr int kMaxWay = 32;
void launch_merge_kway(float* dst, const float* const* srcs, const float* weights /* k+1 */, int k,
                       int64_t n, const PeerSync* syncs /* k or null */, cudaStream_t stream);
// publish / wait / acknowledge as stand-alone stream operations
void launch_flag_signal(uint32_t* flag, uint32_t value, cudaStream_t stream);
void launch_flag_wait(const uint32_t* flag, uint32_t value, cudaStream_t stream);
void launch_flag_add(uint32_t* flag, uint32_t value, cudaStream_t stream);

// ---- nvls.cu: one-shot all-reduce (mean) over symmetric buffers, NVLS multicast or P2P pull -----------
constexpr int kMaxRanks = 16;
struct AllReduceArgs {
    const float* mc;                    // multicast VA of the symmetric contribution buffer (null: P2P pull)
    const float* bufs[kMaxRanks];       // unicast VA of every rank's contribution buffer (peer-mapped)
    uint32_t* flags[kMaxRanks];         // every rank's flag block: ready[world] then done[world]
    int rank, world; uint32_t epoch; float scale;
};
bool launch_allreduce_mean(float* out, const AllReduceArgs& a, int64_t n, cudaStream_t stream);
void preload_nvls();

// ---- optim.cu ------------------------------------------------------------------------------------
// out[i] = keyed permutation of range(n) at i (the order in which the fused kernels and the oracle visit the samples)
void launch_keyed_perm(int64_t* out, int n, uint64_t key, cudaStream_t stream);
// out[i] = mix64(key ^ i) % n, i < k: k keyed draws from range(n) WITH replacement (SamplingTMH's coordinate sample)
void launch_keyed_randint(int64_t* out, int64_t k, int64_t n, uint64_t key, cudaStream_t stream);
void launch_sgd(float* p, const float* g, int64_t n, float lr, float wd, float momentum, float* buf,
                float dampening, bool nesterov, bool first, const float* scale, cudaStream_t stream);
void launch_adam(float* p, const float* g, int64_t n, float* m, float* v, int64_t step, float lr,
                 float beta1, float beta2, float eps, float wd, bool decoupled, cudaStream_t stream);

// ---- mlp1_train*.cu / mlp1_eval.cu ---------------------------------------------------------------
constexpr int kMaxPartsByValue = 16;
struct TrainParams {
    float* row; const float* X; const int64_t* y;
    int n, IN, H, OUT, B, epochs;
    float lr, wd; uint64_t key;
    // K3 (PartitionedTMH): part_id = partition of every parameter (device), ages = age of every partition -- either a
    // device array (`ages`) or, when that is null and use_ages_val is set, by value (<= 16 partitions; no H2D copy)
    const int64_t* part_id; const int64_t* ages; int n_parts;
    int64_t ages_val[kMaxPartsByValue]; bool use_ages_val;
    __host__ __device__ bool scaled() const { return part_id != nullptr && (ages != nullptr || use_ages_val); }
    __host__ __device__ int64_t age_of(int part) const { return ages != nullptr ? ages[part] : ages_val[part]; }
    int Hs, C, nbuf;
    float* dbg;                 // optional debug dump (tests)
    // torch.optim.SGD momentum (fused tcgen05 kernel only): `mom` = momentum-buffer row (same layout as `row`),
    // mom_first = the buffer holds no state yet (torch initialises it with the first gradient)
    float momentum, dampening; bool nesterov; float* mom; bool mom_first;
    // fused MERGE_UPDATE: when `peer` is set the kernel starts from w_self*row + w_peer*peer
    // (the peer row is pulled over NVLink while the weights are loaded on chip)
    const float* peer; float w_self, w_peer; PeerSync sync;
    // the tcgen05 kernel's operands are staged by a loader kernel that depends on (X, y, key) only, not on the model:
    // 0 = loader + training kernel, 1 = loader only (issued BEFORE the stream waits for the incoming snapshot, so it
    // is off the critical path of a gossip chain), 2 = training kernel only (operands already staged on this stream)
    int stage_mode;
};
// auto = fp32-equivalent: tc8 (3xTF32 on an 8-CTA cluster) -> cluster (fp32 CUDA cores).  Plain-tf32 kernels only by name:
// tc3 (CTA pair, whole step on the tensor core), tc8-tf32 (8-CTA cluster).
enum TrainImpl { kTrainAuto = 0, kTrainCluster = 1, kTrainTc3 = 4, kTrainTc8 = 7, kTrainTc8Tf32 = 8 };
// returns false when the shape is outside the envelope of the requested implementation
bool launch_mlp1_train(TrainParams p, TrainImpl impl, cudaStream_t stream, const char** why);
void set_default_train_impl(TrainImpl impl);   // meaning of kTrainAuto for this process
bool mlp1_train_tc3(const TrainParams& p, cudaStream_t stream);    // CTA pair, plain tf32, second layer on the tensor core too
// fourth generation: nc-CTA cluster (4 or 8), x3 = error-compensated 3xTF32 products (fp32-equivalent)
bool mlp1_train_tc4(const TrainParams& p, int nc, bool x3, cudaStream_t stream);
bool reserve_train_staging(int n, int IN, int B, int epochs, int nc, bool x3, cudaStream_t stream);
size_t mlp1_stage4_bytes(int n, int IN, int B, int epochs, int NC, bool x3, int* FPC_out, int* FP_out, int* steps_out);
// device-side data loader of the tc3 training kernel: shuffled mini-batches in both UMMA operand layouts
size_t mlp1_stage_bytes(int n, int IN, int B, int epochs, int* FPC_out, int* FP_out, int* steps_out);
bool launch_mlp1_stage(const float* X, const int64_t* y, int n, int IN, int B, int epochs, uint64_t key,
                       void* staging, cudaStream_t stream);
// score1 (optional, [n]): the class-1 logit of every sample, for the AUC of 2-output networks
bool launch_mlp1_eval(const float* row, const float* X, const int64_t* y, int n, int IN, int H, int OUT,
                      int n_classes, int* cm, float* score1, cudaStream_t stream);
// tcgen05 evaluation on a PRE-TILED copy of the test set (mlp1_eval_tc.cu)
int64_t mlp1_eval_pretile_floats(int n, int IN);
void launch_mlp1_eval_pretile(const float* X, int n, int IN, float* out, cudaStream_t stream);
bool launch_mlp1_eval_tc(const float* row, const float* xt, const int64_t* y, int n, int IN, int H, int OUT,
                         int n_classes, int* cm, float* score1, cudaStream_t stream);
void preload_eval_tc();
void set_eval_tf32(bool on);            // plain tf32 products instead of the fp32-equivalent 3xTF32 default

// ---- small.cu --------------------------------------------------------------------------------------
struct LogregParams {
    float* row; const float* X; const int64_t* y; int n, IN, OUT, B, epochs; float lr, wd; uint64_t key;
    const int64_t* part_id; const int64_t* ages; int n_parts;
    int64_t ages_val[kMaxPartsByValue]; bool use_ages_val;
    __host__ __device__ bool scaled() const { return part_id != nullptr && (ages != nullptr || use_ages_val); }
    __host__ __device__ int64_t age_of(int part) const { return ages != nullptr ? ages[part] : ages_val[part]; }
    const float* peer; float w_self, w_peer; PeerSync sync;
};
bool launch_logreg_train(LogregParams p, cudaStream_t stream);
void launch_logreg_scores(const float* row, const float* X, int n, int IN, int OUT, float* out,
                          cudaStream_t stream);
void launch_linear_seq(float* w, const float* X, const float* y, int n, int dim, int kind, float lr,
                       long long t0, cudaStream_t stream);
void launch_kmeans_assign(const float* C, const float* X, int n, int k, int dim, int64_t* out,
                          cudaStream_t stream);
void launch_kmeans_apply(float* C, const float* X, const int64_t* asg, int n, int k, int dim, float alpha,
                         cudaStream_t stream);
// optimal centroid matching (k <= 8, exhaustive) fused with the weighted merge; perm_out (optional, [k]) = assignment
bool launch_kmeans_match_merge(float* C, const float* P, int k, int dim, float w_own, float w_peer, PeerSync sync,
                               int64_t* perm_out, cudaStream_t stream);
void launch_mf_update(float* Xu, float* bu, float* Y, float* c, const float* ratings, int m, int k,
                      float reg, float lr, cudaStream_t stream);

// ---- bank.cu: many linear learners (AdaLine / Pegasos) per launch ---------------------------------------
struct BankView {
    float* W; long long* age;            // live models [N][Dp] and their ages
    float* S; long long* slot_age;       // in-flight snapshots [slots][Dp]
    int D, Dp;
    const float* X; const float* y;      // all nodes' samples, concatenated; labels as float (+-1)
    const int64_t* off; const int* cnt;  // node -> first sample, number of samples
    int kind;                            // 0 AdaLine, 1 Pegasos
    int mode;                            // CreateModelMode value (1 UPDATE, 2 MERGE_UPDATE, 3 UPDATE_MERGE, 4 PASS)
    float lr;
};
// several ranks: a snapshot is PUSHED into the slot bank of the receiver's GPU (remote stores over NVLink), so the
// delivery kernels only read local memory; phases are separated by a flag barrier across the ranks
struct BankPeers { float* S[kMaxRanks]; long long* slot_age[kMaxRanks]; };
struct RankBarrier { uint32_t* flags[kMaxRanks]; int rank, world; uint32_t gen; };   // flags[r][q] = generation rank q reached
void launch_bank_snapshot_push(const BankView& b, const BankPeers& peers, const int* sender, const int* slot,
                               const int* dst_rank, int n, cudaStream_t st);
void launch_rank_barrier(const RankBarrier& rb, cudaStream_t st);
void launch_bank_snapshot(const BankView& b, const int* sender, const int* slot, int n, cudaStream_t st);
bool launch_bank_deliver(const BankView& b, const int* recv, const int* slot, const int* item_mode, int n, cudaStream_t st);
bool launch_bank_update(const BankView& b, const int* nodes, int n, cudaStream_t st);
void launch_bank_scores(const BankView& b, const int* nodes, int n_nodes, const float* Xte, int n_te, float* scores,
                        cudaStream_t st);
void preload_bank();

// ---- bank_families.cu: many k-means / matrix-factorisation nodes per launch (one CTA per work item) ----------------
constexpr int kFamilyMaxK = 64;          // k-means: most centroids per model
struct FamilyBankView {
    float* W; long long* age;            // live models [N][Dp] and their ages
    float* S; long long* slot_age;       // in-flight snapshots [slots][Dp]
    int Dp;
    const float* data;                   // local data, concatenated: k-means samples [*][dim], MF ratings [*][2] (item, r)
    const int64_t* off; const int* cnt;  // node -> first sample / rating, number of them
    int k, dim;                          // k-means: k centroids of dim floats; MF: rank k, dim = number of items
    int mode;                            // CreateModelMode value (1 UPDATE, 2 MERGE_UPDATE, 3 UPDATE_MERGE, 4 PASS)
    int hungarian;                       // k-means: optimal centroid matching before the merge (k <= 8)
    float alpha;                         // k-means: EMA step
    float reg, lr;                       // MF: L2 regularisation, learning rate
};
// S[slot] = W[sender]: rows of up to 1024 floats go through bank.cu's warp-per-item kernel, wider ones one CTA per item
void launch_family_snapshot(const FamilyBankView& b, const int* sender, const int* slot, int n, cudaStream_t st);
bool launch_kmeans_bank_deliver(const FamilyBankView& b, const int* recv, const int* slot, int n, cudaStream_t st);
// ct [n_nodes][n_true][k] int32, zero on entry
void launch_kmeans_bank_eval(const FamilyBankView& b, const int* nodes, int n_nodes, const float* Xte, const int64_t* yte,
                             int n_te, int n_true, int* ct, cudaStream_t st);
bool launch_mf_bank_deliver(const FamilyBankView& b, const int* recv, const int* slot, int n, cudaStream_t st);
// sse [n_nodes]: squared error summed over each node's own test ratings te[te_off[node] ..][2]
void launch_mf_bank_eval(const FamilyBankView& b, const int* nodes, int n_nodes, const float* te, const int64_t* te_off,
                         const int* te_cnt, float* sse, cudaStream_t st);
void preload_bank_families();

int sm_count();
// load every kernel of the extension on the current device (see merge.cu: preload_merge)
void preload_merge(); void preload_optim(); void preload_small(); void preload_eval();
void preload_train_cluster(); void preload_train_tc3(); void preload_train_tc4(); void preload_stage();

}  // namespace gb
