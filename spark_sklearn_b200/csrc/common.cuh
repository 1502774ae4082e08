// common.cuh -- shared declarations of the libb200gs.so translation units (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>
#include "../../include/b200gs.h"

#define GS_CUDA(call)                                                                         \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess) {                                                              \
            gs_set_error(h, std::string(#call) + ": " + cudaGetErrorString(e_) + " @" +       \
                                __FILE__ + ":" + std::to_string(__LINE__));                   \
            return GS_ERR_CUDA;                                                               \
        }                                                                                     \
    } while (0)

// grow-only device buffer
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return (T *)p; }
};

// CUDA events owned by the handle: created on first use, reused by every later call, destroyed with the handle
// (no per-call cudaEventCreate / cudaEventDestroy, nothing to leak on an error return)
struct EventPool {
    std::vector<cudaEvent_t> ev;
    size_t used = 0;
    cudaEvent_t get()
    {
        if (used == ev.size()) { cudaEvent_t e = nullptr; cudaEventCreate(&e); ev.push_back(e); }
        return ev[used++];
    }
    void reset() { used = 0; }
    void release() { for (auto e : ev) cudaEventDestroy(e); ev.clear(); used = 0; }
};

// CUDA-event time and executed MMA flops of the tensor-core contraction launches of one call
struct TensorTimer {
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> spans;
    double flops = 0;
    cudaEvent_t open = nullptr;
    void reset() { spans.clear(); flops = 0; open = nullptr; }
    void begin(EventPool &p, cudaStream_t st) { open = p.get(); cudaEventRecord(open, st); }
    void end(EventPool &p, cudaStream_t st, double f)
    {
        cudaEvent_t e = p.get();
        cudaEventRecord(e, st);
        spans.emplace_back(open, e); flops += f;
    }
    float collect()                      // the stream must have been synchronised
    {
        float tot = 0;
        for (auto &s : spans) { float ms = 0; if (cudaEventElapsedTime(&ms, s.first, s.second) == cudaSuccess) tot += ms; }
        return tot;
    }
};

// Membership of every row in the training / test set of every CV split: two 64-bit words per row and kind (splits 0..127).
// Replaces the per-task index arrays of the reference (base_search.py:81-82 islice(cv.split(...))): any splitter fits --
// overlapping test sets (RepeatedKFold), rows in neither set (ShuffleSplit), rows that only ever train (PredefinedSplit -1).
struct SplitMasks {
    const unsigned long long *te, *tr;
};
#ifdef __CUDACC__
__device__ __forceinline__ bool split_test(const SplitMasks &m, int r, int k)      // k < 0 (refit): nobody is tested
{
    return k >= 0 && ((m.te[(size_t)r * 2 + (k >> 6)] >> (k & 63)) & 1ull);
}
__device__ __forceinline__ bool split_train(const SplitMasks &m, int r, int k)     // k < 0 (refit): every row trains
{
    return k < 0 || ((m.tr[(size_t)r * 2 + (k >> 6)] >> (k & 63)) & 1ull);
}
#endif

struct gs_handle {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t stream_hi = nullptr;   // second stream: the single-CTA SMO launch when a cluster launch runs beside it
    cudaStream_t stream_lo = nullptr;   // third stream: the shared-SM launch when cluster and exclusive-SM launches run beside it
    std::string err;
    // dataset (rows stored in INTERNAL order: sorted by class, then by original index)
    int64_t n = 0, d = 0;
    int n_splits = 0, n_classes = 0;
    bool classification = false;
    std::vector<int32_t> perm;        // internal row -> original row
    std::vector<int32_t> yc;          // [n] class ids, internal order
    std::vector<float> yt;            // [n] regression targets, internal order (empty for a classification dataset)
    std::vector<int8_t> fold;         // [n] fold ids, internal order (partition splitters; Ridge's fold blocks)
    std::vector<uint64_t> te_mask, tr_mask;   // [n][2] split membership, internal order
    bool partition = true;            // the splits are a partition into test folds whose complements train (gs_set_data's fold ids)
    bool is_test(int r, int k) const { return k >= 0 && ((te_mask[(size_t)r * 2 + (k >> 6)] >> (k & 63)) & 1ull); }
    bool is_train(int r, int k) const { return k < 0 || ((tr_mask[(size_t)r * 2 + (k >> 6)] >> (k & 63)) & 1ull); }
    SplitMasks masks() const { return SplitMasks{dTe.as<unsigned long long>(), dTr.as<unsigned long long>()}; }
    std::vector<int32_t> class_start; // [n_classes+1] internal row ranges per class
    DevBuf dX, dY, dFold, dYt;        // float X[n][d], int32 y[n], int8 fold[n], float yt[n]
    DevBuf dTe, dTr;                  // uint64 [n][2] test / training membership of every split
    DevBuf dX64;                      // double X[n][d] when the caller's matrix is float64
    int x_dtype = GS_F32;
    DevBuf dS, dXsq;                  // float64 Gram [n][n], squared norms [n]
    DevBuf dK;                        // float32 kernel matrices (batch)
    DevBuf dWork[9];                  // per-search scratch
    DevBuf dScore;                    // class counts / AUC pair counts of the non-default scorers
    int score_kind = 0, score_pos = 1;   // gs_set_scoring
    std::vector<double> class_w;         // gs_set_class_weight: [sets][n_classes]; empty = all ones
    int class_w_sets = 0;
    std::vector<float> sample_w;         // gs_set_sample_weight: [n] internal order; empty = all ones
    DevBuf dSw;                          // its device copy
    gs_profile prof;
    EventPool evp;                    // timing events of the current call
    TensorTimer tt;
};

void gs_set_error(gs_handle *h, const std::string &msg);

// ---- gram.cu ----
// S = X X^T in float64 from float32 X (exact products, float64 accumulation); xsq = diag(S).
cudaError_t launch_gram_f64(const void *X, int x_dtype, int n, int d, double *S, double *xsq, cudaStream_t st);
cudaError_t launch_widen_gram(const float *S32, int n, int64_t ld32, double *S, double *xsq, cudaStream_t st);
// K[r][c] = (float) k(x_r, x_c) from S: rbf exp(-gamma*(xsq_r + xsq_c - 2 S_rc)) or linear S_rc.
// *special (device int, pre-zeroed, may be null) is set when an entry is not a positive normal float.
cudaError_t launch_kernel_matrix(const double *S, const double *xsq, int n, int kernel, double gamma,
                                 float *K, int64_t ldk, int *special, cudaStream_t st);

// ---- smo.cu ----
struct SmoProblem {
    const float *K;       // float32 kernel matrix of this (kernel, gamma): [n][ldk]
    const double *qd;     // float64 diagonal by dataset row (linear kernel) or nullptr (rbf: QD == 1)
    const int *rows;      // [l] dataset rows in sub-problem order: n_pos rows of the +1 class first
    double *alpha;        // [l] workspace: alpha by position
    double *Gbar;         // [l] workspace
    int *scratch;         // [2*l + 64] workspace
    double *coef;         // [n] out: alpha*y scattered by dataset row (pre-zeroed)
    double *out_rho;      // out
    int *out_info;        // out: [0] n_iter [1] timed_out [2] n_sv [3] n_bounded_sv
    unsigned long long *out_ns;   // out: [0] start [1] end (globaltimer)
    // Device flag written by kernel_matrix_kernel: != 0 when K holds a zero, denormal or negative entry.  Both solver
    // instances are enqueued behind it; the branch-free (FAST) one returns at once when it is set, the general one when it
    // is clear -- the choice needs no host round trip in the middle of a search.  nullptr: run unconditionally.
    const int *guard;
    int64_t ldk;
    double C, Cn, eps;    // C of the +1 class (the pair's first class) and of the -1 class: C x class_weight
    int l, n_pos, max_iter, shrinking;
    // up to 4 column ranges (floats, multiples of 4) that cover this sub-problem's dataset rows: the single-CTA kernel
    // copies only these parts of a K row into shared memory (a fold's training rows are 2-3 contiguous runs of the
    // class-sorted dataset: 32 KB of a 40 KB row in config 2).  nseg == 0: copy the whole row.
    int nseg, seg_start[4], seg_len[4];
    int nslots;           // sum of seg_len: size of the slot space of smo_lean.cu (0 when nseg == 0)
};
// Solve problems order[0..n_prob) (one CTA each); lmax = max l (selects the template instance).
cudaError_t launch_smo(const SmoProblem *d_probs, const int *d_order, int n_prob, int lmax, bool fast, int rowcap,
                       cudaStream_t st, std::string *why);
int smo_max_rows();   // largest sub-problem the resident-state kernel supports
// smo_lean.cu: the throughput instance (static slots = the problem's column runs, two or more sub-problems per SM).  Every
// problem of the launch needs a slot layout: nseg > 0, nslots <= smo_lean_max_slots(), l < 16383; alpha and Gbar hold nslots doubles.
int smo_lean_max_slots();
// exclusive: one sub-problem per SM (the launch asks for more than half of an SM's shared memory)
cudaError_t launch_smo_lean(const SmoProblem *d_probs, const int *d_order, int n_prob, int max_slots, bool fast, bool exclusive, cudaStream_t st);
// smo_colown.cu: the same solver with one sub-problem spread over a thread-block cluster of cl CTAs (DSMEM exchange)
int smo_colown_max_rows(int cl);
void launch_delay(unsigned ns, cudaStream_t st);      // one thread sleeping ns nanoseconds (stream-ordering aid)
cudaError_t launch_smo_colown(const SmoProblem *d_probs, const int *d_order, int n_prob, int lmax, int cl, bool fast, cudaStream_t st);

// ---- score.cu ----
// dec[c][r] = sum_j k64(r, j) * coef[c][j]  (float64 kernel values recomputed from S, not the
// float32-rounded K: svm.cpp:2821 svm_predict_values uses k_function in double).
// decision_chunks: into how many slabs the support-row range of one launch is split so that its CTAs fill the GPU in whole
// rounds (157 row blocks on 592 resident CTAs: 4 slabs = 628 CTAs = two rounds for 1.06 rounds of work; 15 slabs = 3.98).
int decision_chunks(int n, int ncols, int sms);
cudaError_t launch_decision(const double *S, const double *xsq, int n, int kernel, double gamma,
                            const double *coef, int ncols, double *dec, double *part, int jchunks, cudaStream_t st);
struct VoteTask {          // one (candidate, fold) task
    int first_col;         // first decision column of this task inside its group (n_pairs consecutive)
    int fold;              // test fold id
};
// counts[task][0..3] = {test correct, test total, train correct, train total}
cudaError_t launch_vote(const double *dec, const double *rho, int n, int n_classes, const int *y,
                        SplitMasks sm, const VoteTask *tasks, int n_tasks, int *counts,
                        cudaStream_t st);

// per-class counts for the count-based scorers: counts[task][split (0 test, 1 train)][class][3 = support, tp, predicted]
cudaError_t launch_vote_classes(const double *dec, const double *rho, int n, int n_classes, const int *y,
                                SplitMasks sm, const VoteTask *tasks, int n_tasks, int *counts, cudaStream_t st);
// ROC-AUC pair counts of binary tasks: out[task][4] = {test wins, test ties, train wins, train ties}; rows are class-sorted
// (negative class = rows [0, n_a)); score row of task t = score + col_of_task[t] * ld; sign -1 for libsvm decision values
cudaError_t launch_auc_pairs_f64(const double *score, int64_t ld, int n, int n_a, SplitMasks sm, const int *col_of_task,
                                 const int *fold_of_task, int n_tasks, int sign, unsigned long long *out, cudaStream_t st);
cudaError_t launch_auc_pairs_f32(const float *score, int64_t ld, int n, int n_a, SplitMasks sm, const int *col_of_task,
                                 const int *fold_of_task, int n_tasks, int sign, unsigned long long *out, cudaStream_t st);
// score of one (task, split) from the class counts cnt[class][3] (float64, scikit-learn's formulas); NaN when undefined
double gs_score_from_counts(int kind, int pos_class, int n_classes, const int *cnt);

// ---- gemm_tc.cu: tcgen05 + TMA contraction  C[M][N] = sum_k A[M][k] B[N][k]  (3xTF32 split, fp32 accumulate) ----
struct alignas(64) TcMap { unsigned char bytes[128]; };            // CUtensorMap
struct TcBatch {                                                    // one GEMM of a batched launch (blockIdx.z)
    int a_row0, b_row0;   // first row of the A / B operand inside their tensor maps
    int k0, k1;           // contraction range [k0, k1) in elements; must be a multiple of 32 long (zero padded)
    float *c;             // output, row-major
    int64_t ldc;
};
cudaError_t tc_make_map(TcMap *out, const float *base, int64_t rows, int64_t cols, int64_t ld);
cudaError_t launch_split_tf32(const float *x, float *hi, float *lo, size_t n, cudaStream_t st);
constexpr int TC_KCHUNK = 512;   // longest accumulation chain kept inside the (truncating) TMEM accumulator
cudaError_t launch_sum_partials(const float *partial, int n_chunks, int64_t per, float *out, cudaStream_t st);
// symmetric: the A and B operands are the same matrix (M == N): tiles below the diagonal are not computed, their values are
// stored as transposes of the tiles above it (bitwise symmetric result)
cudaError_t launch_gemm_nt_tf32x3(const TcMap &a_hi, const TcMap &a_lo, const TcMap &b_hi, const TcMap &b_lo,
                                  const TcBatch *d_batches, int n_batches, int M, int N, float alpha, bool accumulate,
                                  cudaStream_t st, bool symmetric = false);
