// api.cu -- the C ABI of libb200gs.so (include/b200gs.h): lifecycle, dataset upload, SVC search/refit.
// Host-side planning only; every floating-point operation of the hot path runs in the CUDA kernels
// of gram.cu / smo.cu / score.cu.  There is no CPU fallback.
#include "common.cuh"
#include <algorithm>
#include <cmath>
#include <cstring>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <mutex>
#include <queue>
#include <numeric>

static std::string g_create_error;

// scikit-learn's count-based scores (metrics/_classification.py) from cnt[class][3] = {support, tp, predicted}, float64.
// Undefined ratios follow zero_division="warn": 0.0.  accuracy_score :187; balanced_accuracy_score :2362 (mean recall over
// the classes present in y_true); precision_recall_fscore_support :1573 with beta = 1: f = 2 tp / (2 tp + fp + fn).
// The averages run over the labels present in y_true or y_pred: a class with support + predicted == 0 adds nothing to the
// weighted f1 (weight 0) or to balanced accuracy (only y_true's classes), and is left out of the macro mean.
double gs_score_from_counts(int kind, int pos_class, int n_classes, const int *cnt)
{
    auto sup = [&](int c) { return (double)cnt[c * 3 + 0]; };
    auto tp = [&](int c) { return (double)cnt[c * 3 + 1]; };
    auto prd = [&](int c) { return (double)cnt[c * 3 + 2]; };
    auto f1c = [&](int c) { const double den = sup(c) + prd(c); return den > 0 ? 2.0 * tp(c) / den : 0.0; };   // 2tp + fp + fn = support + predicted
    double n = 0, correct = 0;
    for (int c = 0; c < n_classes; c++) { n += sup(c); correct += tp(c); }
    if (!(n > 0)) return NAN;
    switch (kind) {
    case GS_SCORE_DEFAULT: return correct / n;
    case GS_SCORE_BALANCED_ACCURACY: {
        double s = 0; int k = 0;
        for (int c = 0; c < n_classes; c++) if (sup(c) > 0) { s += tp(c) / sup(c); k++; }
        return k ? s / k : NAN;
    }
    case GS_SCORE_F1: return f1c(pos_class);
    case GS_SCORE_PRECISION: return prd(pos_class) > 0 ? tp(pos_class) / prd(pos_class) : 0.0;
    case GS_SCORE_RECALL: return sup(pos_class) > 0 ? tp(pos_class) / sup(pos_class) : 0.0;
    case GS_SCORE_F1_MACRO: {
        // mean over the labels of y_true and y_pred (unique_labels, :1573): a class of the dataset that is neither in this
        // set nor predicted for it does not count
        double s = 0; int k = 0;
        for (int c = 0; c < n_classes; c++) if (sup(c) + prd(c) > 0) { s += f1c(c); k++; }
        return s / k;                                                    // k >= 1: n > 0 rows were predicted
    }
    case GS_SCORE_F1_MICRO: return correct / n;                         // single-label: micro f1 == accuracy
    case GS_SCORE_F1_WEIGHTED: {
        double s = 0;
        for (int c = 0; c < n_classes; c++) s += f1c(c) * sup(c);
        return s / n;
    }
    default: return NAN;
    }
}

void gs_set_error(gs_handle *h, const std::string &msg)
{
    if (h) h->err = msg; else g_create_error = msg;
}

namespace {

// dst[r][:] = src[perm[r]][:]; optionally also a float32 copy of a float64 source
template <typename T>
__global__ void gather_rows_kernel(const T *__restrict__ src, const int *__restrict__ perm, int64_t n, int64_t d,
                                   T *__restrict__ dst, float *__restrict__ dst32)
{
    const int64_t total = n * d;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = idx / d, c = idx - r * d;
        const T v = src[(int64_t)perm[r] * d + c];
        dst[idx] = v;
        if (dst32) dst32[idx] = (float)v;
    }
}

struct EvTimer {       // accumulates elapsed ms between consecutive marks on one stream (events from the handle's pool)
    cudaStream_t st;
    EventPool &pool;
    std::vector<cudaEvent_t> evs;
    std::vector<int> tag;
    EvTimer(cudaStream_t s, EventPool &p) : st(s), pool(p) {}
    void mark(int t)
    {
        cudaEvent_t e = pool.get();
        cudaEventRecord(e, st);
        evs.push_back(e); tag.push_back(t);
    }
    // after a stream sync: add the time between mark k-1 and mark k to acc[tag[k]]
    void collect(float *acc, int ntags)
    {
        for (size_t k = 1; k < evs.size(); k++) {
            float ms = 0;
            cudaEventElapsedTime(&ms, evs[k - 1], evs[k]);
            if (tag[k] >= 0 && tag[k] < ntags) acc[tag[k]] += ms;
        }
        evs.clear(); tag.clear();
    }
};

inline uint64_t dbits(double x) { uint64_t u; memcpy(&u, &x, 8); return u; }

}  // namespace

extern "C" {

int gs_version(void) { return 101; }

int gs_set_class_weight(gs_handle *h, const double *w, int32_t n_sets)
{
    if (!h) return GS_ERR_ARG;
    if (!w || n_sets <= 0) { h->class_w.clear(); h->class_w_sets = 0; return GS_OK; }
    if (h->n_classes <= 0) { gs_set_error(h, "gs_set_class_weight: no classification dataset"); return GS_ERR_NO_DATA; }
    for (int64_t i = 0; i < (int64_t)n_sets * h->n_classes; i++)
        if (!(w[i] > 0) || !std::isfinite(w[i])) { gs_set_error(h, "gs_set_class_weight: weights must be positive and finite"); return GS_ERR_ARG; }
    h->class_w.assign(w, w + (size_t)n_sets * h->n_classes);
    h->class_w_sets = n_sets;
    return GS_OK;
}

int gs_set_sample_weight(gs_handle *h, const double *w)
{
    if (!h) return GS_ERR_ARG;
    if (!w) { h->sample_w.clear(); return GS_OK; }
    if (h->n == 0) { gs_set_error(h, "gs_set_sample_weight: no dataset (call gs_set_data first)"); return GS_ERR_NO_DATA; }
    std::vector<float> sw((size_t)h->n);
    for (int64_t i = 0; i < h->n; i++) {
        const double v = w[h->perm[i]];
        if (!(v >= 0) || !std::isfinite(v)) { gs_set_error(h, "gs_set_sample_weight: weights must be finite and >= 0"); return GS_ERR_ARG; }
        sw[i] = (float)v;                                     // scikit-learn: _check_sample_weight(..., dtype=X.dtype)
    }
    GS_CUDA(cudaSetDevice(h->device));
    GS_CUDA(h->dSw.reserve((size_t)h->n * 4));
    GS_CUDA(cudaMemcpyAsync(h->dSw.p, sw.data(), (size_t)h->n * 4, cudaMemcpyHostToDevice, h->stream));
    GS_CUDA(cudaStreamSynchronize(h->stream));
    h->sample_w.swap(sw);
    return GS_OK;
}

int gs_set_scoring(gs_handle *h, int32_t kind, int32_t pos_class)
{
    if (!h) return GS_ERR_ARG;
    const bool known = (kind >= GS_SCORE_DEFAULT && kind <= GS_SCORE_F1_WEIGHTED) || kind == GS_SCORE_NEG_MSE || kind == GS_SCORE_NEG_RMSE;
    if (!known || pos_class < 0 || pos_class > 31) { gs_set_error(h, "gs_set_scoring: unknown scorer or positive class"); return GS_ERR_ARG; }
    h->score_kind = kind; h->score_pos = pos_class;
    return GS_OK;
}

int gs_device_count(void)
{
    int count = 0, usable = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) return 0;
    for (int d = 0; d < count; d++) {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, d) == cudaSuccess && prop.major == 10) usable = d + 1;   // handles index devices 0..n-1
    }
    return usable;
}

const char *gs_last_error(const gs_handle *h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int gs_create(int device, gs_handle **out)
{
    if (!out) return GS_ERR_ARG;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e) + " (libb200gs has no CPU fallback)";
        return GS_ERR_CUDA;
    }
    if (device < 0 || device >= count) { g_create_error = "device index out of range"; return GS_ERR_ARG; }
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) { g_create_error = cudaGetErrorString(e); return GS_ERR_CUDA; }
    if (prop.major != 10) {
        g_create_error = "libb200gs is built for sm_100a only; device is sm_" + std::to_string(prop.major * 10 + prop.minor);
        return GS_ERR_UNSUPPORTED;
    }
    if ((e = cudaSetDevice(device)) != cudaSuccess) { g_create_error = cudaGetErrorString(e); return GS_ERR_CUDA; }
    gs_handle *h = new gs_handle();
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    if ((e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess) {
        g_create_error = cudaGetErrorString(e); delete h; return GS_ERR_CUDA;
    }
    {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if ((e = cudaStreamCreateWithPriority(&h->stream_hi, cudaStreamNonBlocking, hi)) != cudaSuccess) {
            g_create_error = cudaGetErrorString(e); cudaStreamDestroy(h->stream); delete h; return GS_ERR_CUDA;
        }
    }
    if ((e = cudaStreamCreateWithFlags(&h->stream_lo, cudaStreamNonBlocking)) != cudaSuccess) {
        g_create_error = cudaGetErrorString(e); cudaStreamDestroy(h->stream); cudaStreamDestroy(h->stream_hi); delete h; return GS_ERR_CUDA;
    }
    memset(&h->prof, 0, sizeof h->prof);
    *out = h;
    return GS_OK;
}

void gs_destroy(gs_handle *h)
{
    if (!h) return;
    cudaSetDevice(h->device);
    h->dX.release(); h->dY.release(); h->dFold.release(); h->dYt.release(); h->dTe.release(); h->dTr.release();
    h->dS.release(); h->dXsq.release(); h->dK.release(); h->dX64.release();
    h->evp.release(); h->dScore.release(); h->dSw.release();
    for (auto &w : h->dWork) w.release();
    if (h->stream) cudaStreamDestroy(h->stream);
    if (h->stream_hi) cudaStreamDestroy(h->stream_hi);
    if (h->stream_lo) cudaStreamDestroy(h->stream_lo);
    delete h;
}

int gs_set_data(gs_handle *h, const void *X, int32_t x_dtype, int64_t n, int64_t d, const int32_t *y_class,
                const float *y_target, const int8_t *fold_id, int32_t n_splits)
{
    if (!h) return GS_ERR_ARG;
    if (n_splits > 127) { if (h) gs_set_error(h, "gs_set_data: more than 127 CV splits"); return GS_ERR_UNSUPPORTED; }
    if (!X || n <= 0 || d <= 0 || !fold_id || n_splits < 1 || (!y_class && !y_target) ||
        (x_dtype != GS_F32 && x_dtype != GS_F64)) {
        gs_set_error(h, "gs_set_data: bad arguments"); return GS_ERR_ARG;
    }
    if (n > 65535) { gs_set_error(h, "gs_set_data: n > 65535 rows is outside the small-dense-data scope of this engine"); return GS_ERR_UNSUPPORTED; }
    GS_CUDA(cudaSetDevice(h->device));
    h->n = n; h->d = d; h->n_splits = n_splits; h->x_dtype = x_dtype;
    h->classification = y_class != nullptr;
    h->score_kind = GS_SCORE_DEFAULT; h->score_pos = 1;      // a new dataset starts from the estimator's own score and unit class weights
    h->class_w.clear(); h->class_w_sets = 0;
    h->sample_w.clear();
    h->perm.resize(n);
    std::iota(h->perm.begin(), h->perm.end(), 0);
    h->n_classes = 0;
    if (y_class) {
        for (int64_t i = 0; i < n; i++) {
            if (y_class[i] < 0) { gs_set_error(h, "gs_set_data: negative class id"); return GS_ERR_ARG; }
            h->n_classes = std::max(h->n_classes, y_class[i] + 1);
        }
        // internal order: by class, then original index -- makes every one-vs-one sub-problem a
        // (nearly) contiguous column range of the kernel matrix, so SMO row gathers coalesce
        std::stable_sort(h->perm.begin(), h->perm.end(), [&](int a, int b) { return y_class[a] < y_class[b]; });
    } else {
        // regression: internal order by fold (rows outside every test set last), so every fold is a contiguous
        // row range = a contiguous K-range of the fold-Gram contractions
        std::stable_sort(h->perm.begin(), h->perm.end(), [&](int a, int b) {
            const int fa = fold_id[a] < 0 ? 127 : fold_id[a], fb = fold_id[b] < 0 ? 127 : fold_id[b];
            return fa < fb;
        });
    }
    h->yc.assign(n, 0); h->fold.resize(n);
    h->class_start.assign(h->n_classes + 1, 0);
    for (int64_t i = 0; i < n; i++) {
        const int o = h->perm[i];
        if (y_class) { h->yc[i] = y_class[o]; h->class_start[y_class[o] + 1]++; }
        h->fold[i] = fold_id[o];
        if (fold_id[o] >= n_splits) { gs_set_error(h, "gs_set_data: fold id >= n_splits"); return GS_ERR_ARG; }
    }
    for (int c = 0; c < h->n_classes; c++) h->class_start[c + 1] += h->class_start[c];
    // split membership from the fold ids: row r is tested by split fold[r] and trains every other split
    h->partition = true;
    h->te_mask.assign((size_t)n * 2, 0); h->tr_mask.assign((size_t)n * 2, 0);
    for (int64_t i = 0; i < n; i++)
        for (int k = 0; k < n_splits; k++)
            (h->fold[i] == k ? h->te_mask : h->tr_mask)[(size_t)i * 2 + (k >> 6)] |= 1ull << (k & 63);

    h->evp.reset();
    cudaEvent_t e0 = h->evp.get(), e1 = h->evp.get();
    cudaEventRecord(e0, h->stream);
    const size_t esz = x_dtype == GS_F64 ? 8 : 4;
    GS_CUDA(h->dX.reserve((size_t)n * d * 4));
    if (x_dtype == GS_F64) GS_CUDA(h->dX64.reserve((size_t)n * d * 8));
    GS_CUDA(h->dWork[0].reserve((size_t)n * d * esz));
    GS_CUDA(h->dWork[1].reserve((size_t)n * 4));
    GS_CUDA(h->dY.reserve((size_t)n * 4));
    GS_CUDA(h->dFold.reserve((size_t)n));
    GS_CUDA(h->dTe.reserve((size_t)n * 16)); GS_CUDA(h->dTr.reserve((size_t)n * 16));
    GS_CUDA(h->dYt.reserve((size_t)n * 4));
    GS_CUDA(cudaMemcpyAsync(h->dWork[0].p, X, (size_t)n * d * esz, cudaMemcpyHostToDevice, h->stream));
    GS_CUDA(cudaMemcpyAsync(h->dWork[1].p, h->perm.data(), (size_t)n * 4, cudaMemcpyHostToDevice, h->stream));
    if (x_dtype == GS_F64)
        gather_rows_kernel<double><<<h->sm_count * 8, 256, 0, h->stream>>>(h->dWork[0].as<double>(), h->dWork[1].as<int>(), n, d,
                                                                           h->dX64.as<double>(), h->dX.as<float>());
    else
        gather_rows_kernel<float><<<h->sm_count * 8, 256, 0, h->stream>>>(h->dWork[0].as<float>(), h->dWork[1].as<int>(), n, d,
                                                                          h->dX.as<float>(), nullptr);
    GS_CUDA(cudaGetLastError());
    GS_CUDA(cudaMemcpyAsync(h->dY.p, h->yc.data(), (size_t)n * 4, cudaMemcpyHostToDevice, h->stream));
    GS_CUDA(cudaMemcpyAsync(h->dFold.p, h->fold.data(), (size_t)n, cudaMemcpyHostToDevice, h->stream));
    GS_CUDA(cudaMemcpyAsync(h->dTe.p, h->te_mask.data(), (size_t)n * 16, cudaMemcpyHostToDevice, h->stream));
    GS_CUDA(cudaMemcpyAsync(h->dTr.p, h->tr_mask.data(), (size_t)n * 16, cudaMemcpyHostToDevice, h->stream));
    h->yt.clear();
    if (y_target) {
        h->yt.resize(n);
        for (int64_t i = 0; i < n; i++) h->yt[i] = y_target[h->perm[i]];
        GS_CUDA(cudaMemcpyAsync(h->dYt.p, h->yt.data(), (size_t)n * 4, cudaMemcpyHostToDevice, h->stream));
        GS_CUDA(cudaStreamSynchronize(h->stream));
    }
    cudaEventRecord(e1, h->stream);
    GS_CUDA(cudaStreamSynchronize(h->stream));
    cudaEventElapsedTime(&h->prof.ms_h2d, e0, e1);
    h->prof.h2d_bytes = (int64_t)n * d * (int64_t)esz + n * 9;
    return GS_OK;
}

int gs_set_splits(gs_handle *h, const uint64_t *test_mask, const uint64_t *train_mask, int32_t n_splits)
{
    if (!h) return GS_ERR_ARG;
    if (h->n == 0) { gs_set_error(h, "gs_set_splits: no dataset (call gs_set_data first)"); return GS_ERR_NO_DATA; }
    if (!test_mask || !train_mask || n_splits < 1 || n_splits > 128) { gs_set_error(h, "gs_set_splits: bad arguments (1..128 splits)"); return GS_ERR_ARG; }
    GS_CUDA(cudaSetDevice(h->device));
    const int64_t n = h->n;
    for (int64_t i = 0; i < n; i++) {
        const int o = h->perm[i];
        for (int wd = 0; wd < 2; wd++) {
            const uint64_t te = test_mask[(size_t)o * 2 + wd], tr = train_mask[(size_t)o * 2 + wd];
            if (te & tr) { gs_set_error(h, "gs_set_splits: a row is in both the training and the test set of a split"); return GS_ERR_ARG; }
            h->te_mask[(size_t)i * 2 + wd] = te; h->tr_mask[(size_t)i * 2 + wd] = tr;
        }
    }
    h->n_splits = n_splits;
    h->partition = false;                                    // fold-block algorithms (Ridge) need gs_set_data's fold ids
    GS_CUDA(cudaMemcpyAsync(h->dTe.p, h->te_mask.data(), (size_t)n * 16, cudaMemcpyHostToDevice, h->stream));
    GS_CUDA(cudaMemcpyAsync(h->dTr.p, h->tr_mask.data(), (size_t)n * 16, cudaMemcpyHostToDevice, h->stream));
    GS_CUDA(cudaStreamSynchronize(h->stream));
    h->prof.h2d_bytes += n * 32;
    return GS_OK;
}

// ------------------------------------------------------------------------------------------------
// SVC: shared implementation of gs_svc (folds) and gs_svc_refit (all rows train).
// ------------------------------------------------------------------------------------------------
// ---- planning helpers (also exported: include/b200gs.h) ----
// Predicted SMO iterations / 1000 of a sub-problem with ~8000 rows.  For rbf the iteration count of config 2 / config 4
// (1600 measured fits, tests/golden) rises like (C * gamma*d)^0.95 and saturates at a level ~ 1/(gamma*d):
//     min(4 + 10.3 (C gamma d)^0.95, 9 + 7.3 / (gamma d))      (Spearman 0.985 against the measured counts, median error 12 %)
// Linear kernel: iterations grow with C; no plateau is modelled.  Only the ranking and the ratios are used.
extern "C" double gs_svc_predicted_iterations(int32_t kernel, double C, double gamma, int32_t d)
{
    if (kernel != GS_KERNEL_RBF) return C;
    const double gd = gamma * (double)d;
    if (!(gd > 0)) return C;
    return std::min(4.0 + 10.3 * std::pow(C * gd, 0.95), 9.0 + 7.3 / gd);
}

// Number n of (predicted-longest) problems on 4-CTA clusters that minimises the predicted makespan
//   f(n) = max( throughput bound [sum_rest + 2.0 * sum_clustered] / SMs,   (a cluster iteration costs 2x the SM-time)
//               0.9 * cost of the longest problem left on one SM,         (tail of the run: 6.4 vs 7.1 us per iteration)
//               0.5 * cost of the longest clustered problem )             (3.5 vs 7.1 us per iteration)
// in units of (predicted iterations x single-CTA iteration time); only cost RATIOS matter.  Near-ties go to the smaller n
// (measured on config 2: 10 clusters 297 ms, 14 clusters 313 ms, 19 clusters 323 ms -- the model is optimistic about clusters).
extern "C" int32_t gs_svc_cluster_count(const double *cost_desc, int32_t n, int32_t sm_count)
{
    if (!cost_desc || n < 2 || sm_count < 4) return 0;
    double total = 0;
    for (int q = 0; q < n; q++) total += cost_desc[q];
    const int nmax = std::min(n - 1, sm_count / 4);
    double best = 0, clustered = 0;
    int pick = 0;
    for (int k = 0; k <= nmax; k++) {
        const double f = std::max({(total + clustered) / sm_count, 0.9 * cost_desc[k], k > 0 ? 0.5 * cost_desc[0] : 0.0});
        if (k == 0 || f < 0.97 * best) { best = f; pick = k; }           // more clusters only for a clear (3 %) predicted gain
        clustered += cost_desc[k];
    }
    return pick;
}

// Three-tier schedule of the slot-layout solver (smo_lean.cu): how many of the predicted-longest problems go on 4-CTA
// clusters (n_cluster) and how many of the next-longest get an SM to themselves (n_exclusive); the rest run two per SM.
// Measured per-iteration times of an 8000-row sub-problem (profiles/r02_smo_*): 3.55 us on a 4-CTA cluster, 5.4-5.5 us alone on
// an SM (1024 threads x 8 slots), 10.5 us when two share an SM (= 5.25 us of SM time per iteration; a cluster costs 14.2).  Only the RATIOS enter:
//   T(n_cl, n_ex) = max( 0.34 c[0]                                       longest clustered problem
//                        0.52 c[n_cl]                                    longest exclusive problem
//                        0.50 sum(rest) / SMs left, 0.78 c[n_cl + n_ex]  shared SMs: throughput, and the longest shared
//                                                                        problem (paired for most of its life, alone at the end) )
// in units of (cost x shared-SM iteration time).  More specialised SMs only for a clear (3 %) predicted gain.
static void schedule_closed_form(const double *cost_desc, int32_t n, int32_t sm_count, int32_t *n_cluster, int32_t *n_exclusive)
{
    if (n_cluster) *n_cluster = 0;
    if (n_exclusive) *n_exclusive = 0;
    if (!cost_desc || n < 2 || sm_count < 8) return;
    std::vector<double> suffix(n + 1, 0.0);
    for (int q = n - 1; q >= 0; q--) suffix[q] = suffix[q + 1] + cost_desc[q];
    double best = -1;
    int bc = 0, be = 0;
    const int max_cl = std::min(n - 1, sm_count / 4);
    for (int nc = 0; nc <= max_cl; nc++) {
        for (int ne = 0; nc + ne < n && 4 * nc + ne <= sm_count - 8; ne++) {
            const int left = sm_count - 4 * nc - ne;
            double t = std::max(0.50 * suffix[nc + ne] / left, 0.78 * cost_desc[nc + ne]);
            if (nc > 0) t = std::max(t, 0.34 * cost_desc[0]);
            if (ne > 0) t = std::max(t, 0.52 * cost_desc[nc]);
            if (best < 0 || t < 0.97 * best || (t < best && nc + ne <= bc + be)) { best = t; bc = nc; be = ne; }
        }
    }
    if (n_cluster) *n_cluster = bc;
    if (n_exclusive) *n_exclusive = be;
}

// Alternative (B200GS_SCHEDULE=simulate; also the test hook gs_svc_simulate): the makespan of a candidate split is SIMULATED,
// not bounded by a formula: the block scheduler hands every SM that a finished cluster or exclusive problem gives back to
// the pending CTAs of the shared launch, so "SMs left for the shared tier" is not a constant.  Measured (1 x B200 and
// 8 x B200, tools/exp_sched2.sh, tools/exp_scale8.sh): config 2 255.0 vs 254.7 ms of solve, config 4 identical, the 8-GPU
// weak-scaling step 321.9 vs 315.7 ms (its choice of 15 clusters for the ranks that hold a second class of long problems
// did not shorten their solve phase) -- no gain, so the closed form above stays the default.  Inputs are the measured
// per-iteration times of an 8000-row sub-problem (profiles/r02_smo_*; only their RATIOS matter): 3.55 us on a 4-CTA
// cluster, 5.45 us alone on an SM, 9.4 us each when two share an SM.  Checked against tier timelines measured on config 2
// (B200GS_SMO_TIMELINE) and against forced splits of config 4 (0 / 20 / 40 / 70 exclusive problems: the order is right,
// the values 3 % high).
namespace {
constexpr double RATE_CLUSTER = 3.55, RATE_SOLO = 5.45, RATE_PAIR = 9.4;

// Event simulation of one launch: cost_desc[0..nc) on clusters (4 SMs each), [nc, nc+ne) alone on an SM, the others in
// launch order on the two slots of every SM as it becomes free.  Returns the makespan in cost x rate units.
double simulate_tiers(const double *c, int n, int sms, int nc, int ne)
{
    if (nc < 0 || ne < 0 || nc + ne > n || 4 * nc + ne > sms) return 1e300;
    struct Ev { double t; int sm, slot, ver; bool operator<(const Ev &o) const { return t > o.t; } };
    struct Sm { double rem[2] = {0, 0}; bool busy[2] = {false, false}; int ver[2] = {0, 0}; double last = 0; };
    std::vector<Sm> sm(sms);
    std::priority_queue<Ev> ev;
    double end = 0;
    int s = 0;
    for (int i = 0; i < nc; i++) { const double t = c[i] * RATE_CLUSTER; end = std::max(end, t); for (int k = 0; k < 4; k++) ev.push(Ev{t, s++, -1, 0}); }
    for (int i = 0; i < ne; i++) { const double t = c[nc + i] * RATE_SOLO; end = std::max(end, t); ev.push(Ev{t, s++, -1, 0}); }
    for (; s < sms; s++) ev.push(Ev{0.0, s, -1, 0});
    int next = nc + ne;
    auto resched = [&](int q, double t) {
        Sm &m = sm[q];
        const double per = (m.busy[0] && m.busy[1]) ? RATE_PAIR : RATE_SOLO;
        for (int k = 0; k < 2; k++)
            if (m.busy[k]) ev.push(Ev{t + m.rem[k] * per, q, k, ++m.ver[k]});
    };
    while (!ev.empty()) {
        const Ev e = ev.top(); ev.pop();
        Sm &m = sm[e.sm];
        if (e.slot < 0) {                                           // the SM joins the shared tier
            m.last = e.t;
            for (int k = 0; k < 2 && next < n; k++) { m.rem[k] = c[next++]; m.busy[k] = true; }
            resched(e.sm, e.t);
            continue;
        }
        if (!m.busy[e.slot] || e.ver != m.ver[e.slot]) continue;     // superseded by a rate change
        const double rate = 1.0 / ((m.busy[0] && m.busy[1]) ? RATE_PAIR : RATE_SOLO), dt = e.t - m.last;
        for (int k = 0; k < 2; k++)
            if (m.busy[k]) m.rem[k] = std::max(0.0, m.rem[k] - dt * rate);
        m.last = e.t;
        m.busy[e.slot] = false;
        end = std::max(end, e.t);
        if (next < n) { m.rem[e.slot] = c[next++]; m.busy[e.slot] = true; }
        resched(e.sm, e.t);
    }
    return end;
}
}  // namespace

extern "C" double gs_svc_simulate(const double *cost_desc, int32_t n, int32_t sm_count, int32_t n_cluster, int32_t n_exclusive)
{
    if (!cost_desc || n < 1 || sm_count < 1) return 0.0;
    return simulate_tiers(cost_desc, n, sm_count, n_cluster, n_exclusive);
}

static void schedule_simulated(const double *cost_desc, int32_t n, int32_t sm_count, int32_t *n_cluster, int32_t *n_exclusive)
{
    if (n_cluster) *n_cluster = 0;
    if (n_exclusive) *n_exclusive = 0;
    if (!cost_desc || n < 2 || sm_count < 8) return;
    // a repeated search of the same shape re-uses the last answer
    static std::mutex mu;
    static std::vector<double> last_cost;
    static int last_sms = 0, last_c = 0, last_e = 0;
    {
        std::lock_guard<std::mutex> lk(mu);
        if (last_sms == sm_count && (int)last_cost.size() == n && std::equal(last_cost.begin(), last_cost.end(), cost_desc)) {
            if (n_cluster) *n_cluster = last_c;
            if (n_exclusive) *n_exclusive = last_e;
            return;
        }
    }
    const double *c = cost_desc;
    std::vector<double> suffix(n + 1, 0.0);
    for (int q = n - 1; q >= 0; q--) suffix[q] = suffix[q + 1] + c[q];
    // candidates: tier boundaries at changes of the predicted cost (the folds of one candidate stay in one tier)
    std::vector<int> cut;
    for (int q = 0; q <= n - 1; q++)
        if (q == 0 || c[q - 1] > c[q] * (1.0 + 1e-9)) cut.push_back(q);
    double best = simulate_tiers(c, n, sm_count, 0, 0);
    int bc = 0, be = 0;
    const int max_cl = std::min(n - 1, sm_count / 4);
    // at most ~12 x 24 candidate splits (costs that are all distinct, e.g. one-vs-one pairs of different sizes, would
    // otherwise give one boundary per problem): every k-th boundary among those a tier can reach
    std::vector<int> cut_c, cut_e;
    for (int q : cut) { if (q <= max_cl) cut_c.push_back(q); if (q <= sm_count - 8) cut_e.push_back(q); }
    auto thin = [](std::vector<int> &v, size_t keep) {
        if (v.size() <= keep) return;
        std::vector<int> w;
        for (size_t i = 0; i < keep; i++) w.push_back(v[i * (v.size() - 1) / (keep - 1)]);
        w.erase(std::unique(w.begin(), w.end()), w.end());
        v.swap(w);
    };
    thin(cut_c, 12); thin(cut_e, 24);
    for (int nc : cut_c) {
        for (int pos : cut_e) {
            const int ne = pos - nc;
            if (ne < 0 || (nc == 0 && ne == 0)) continue;
            if (4 * nc + ne > sm_count - 8 || nc + ne >= n) break;
            // lower bounds: the longest problem of every tier, and the SM time of the whole split
            double lb = std::max(nc ? c[0] * RATE_CLUSTER : 0.0, std::max(ne ? c[nc] * RATE_SOLO : 0.0, c[nc + ne] * RATE_SOLO));
            lb = std::max(lb, (4.0 * RATE_CLUSTER * (suffix[0] - suffix[nc]) + RATE_SOLO * (suffix[nc] - suffix[nc + ne]) +
                               0.5 * RATE_PAIR * suffix[nc + ne]) / sm_count);
            if (lb >= 0.985 * best) continue;
            const double t = simulate_tiers(c, n, sm_count, nc, ne);
            // specialised SMs only for a clear (1.5 %) predicted gain; near-ties go to the split that uses fewer of them
            if (t < 0.985 * best || (t < best && 4 * nc + ne <= 4 * bc + be)) { best = t; bc = nc; be = ne; }
        }
    }
    {
        std::lock_guard<std::mutex> lk(mu);
        last_cost.assign(cost_desc, cost_desc + n); last_sms = sm_count; last_c = bc; last_e = be;
    }
    if (n_cluster) *n_cluster = bc;
    if (n_exclusive) *n_exclusive = be;
}

extern "C" void gs_svc_schedule(const double *cost_desc, int32_t n, int32_t sm_count, int32_t *n_cluster, int32_t *n_exclusive)
{
    const char *mode = getenv("B200GS_SCHEDULE");
    if (mode && !strcmp(mode, "simulate")) schedule_simulated(cost_desc, n, sm_count, n_cluster, n_exclusive);
    else schedule_closed_form(cost_desc, n, sm_count, n_cluster, n_exclusive);
}

static int svc_run(gs_handle *h, int n_cand, const int32_t *kernel, const double *Cv, const double *gamma,
                   double tol, int max_iter, uint32_t flags, bool refit,
                   double *test_scores, double *train_scores, int32_t *n_iter, int32_t *n_sv,
                   float *fit_ms, float *score_ms, double *pair_coef, double *rho_out, int32_t *pair_iter)
{
    if (!h) return GS_ERR_ARG;
    if (h->n == 0) { gs_set_error(h, "gs_svc: no dataset (call gs_set_data first)"); return GS_ERR_NO_DATA; }
    if (!h->classification) { gs_set_error(h, "gs_svc: dataset has no class labels"); return GS_ERR_ARG; }
    if (h->n_classes < 2 || h->n_classes > 32) { gs_set_error(h, "gs_svc: need 2..32 classes"); return GS_ERR_UNSUPPORTED; }
    if (n_cand <= 0 || !kernel || !Cv || !gamma) { gs_set_error(h, "gs_svc: bad arguments"); return GS_ERR_ARG; }
    if (!h->sample_w.empty()) {
        gs_set_error(h, "gs_svc: sample weights (a C per row) are not supported by the SMO kernels; class weights are (gs_set_class_weight)");
        return GS_ERR_UNSUPPORTED;
    }
    if (h->class_w_sets > 1 && h->class_w_sets != (refit ? 1 : h->n_splits)) {
        gs_set_error(h, "gs_svc: gs_set_class_weight was given a weight set per split, but not for this number of splits"); return GS_ERR_ARG;
    }
    GS_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const int n = (int)h->n, d = (int)h->d, nc = h->n_classes;
    const int n_splits = refit ? 1 : h->n_splits;
    const int n_pairs = nc * (nc - 1) / 2;
    const int n_tasks = n_cand * n_splits;
    const int64_t ldk = ((int64_t)n + 31) & ~31LL;
    for (int c = 0; c < n_cand; c++) {
        if (kernel[c] != GS_KERNEL_LINEAR && kernel[c] != GS_KERNEL_RBF) { gs_set_error(h, "gs_svc: unsupported kernel id"); return GS_ERR_UNSUPPORTED; }
        if (!(Cv[c] > 0)) { gs_set_error(h, "gs_svc: C must be > 0"); return GS_ERR_ARG; }
    }

    gs_profile &pf = h->prof;
    const float keep_h2d = pf.ms_h2d; const int64_t keep_h2d_bytes = pf.h2d_bytes;
    memset(&pf, 0, sizeof pf);
    pf.ms_h2d = keep_h2d; pf.h2d_bytes = keep_h2d_bytes;
    float acc[5] = {0, 0, 0, 0, 0};   // 0 gram, 1 kernel matrix, 2 solve, 3 score, 4 other
    h->evp.reset(); h->tt.reset();
    EvTimer tm(st, h->evp);
    cudaEvent_t ev_begin = h->evp.get(), ev_end = h->evp.get();
    cudaEventRecord(ev_begin, st);
    tm.mark(-1);

    // ---- 1. Gram X X^T (shared by every candidate, fold and pair) ----
    // default: float64 on the FP64 pipe (libsvm-faithful, gram.cu).  GS_GRAM_TENSOR: tcgen05 tensor cores, 3xTF32 split,
    // TMA-fed (gemm_tc.cu) -- fp32-faithful, so scores agree with scikit-learn to solver tolerance, not bit for bit.
    GS_CUDA(h->dS.reserve((size_t)n * n * 8));
    GS_CUDA(h->dXsq.reserve((size_t)n * 8));
    if (flags & GS_GRAM_TENSOR) {
        const int dpad = (d + 31) & ~31;
        const int64_t ld32 = ((int64_t)n + 3) & ~3LL;
        DevBuf &bx = h->dWork[1], &bs = h->dWork[2], &bb = h->dWork[6];
        GS_CUDA(bx.reserve((size_t)n * dpad * 4 * 3));
        GS_CUDA(bs.reserve((size_t)n * ld32 * 4));
        GS_CUDA(bb.reserve(sizeof(TcBatch) + 64));
        float *xp = bx.as<float>(), *xh = xp + (size_t)n * dpad, *xl = xh + (size_t)n * dpad;
        GS_CUDA(cudaMemsetAsync(xp, 0, (size_t)n * dpad * 4, st));
        GS_CUDA(cudaMemcpy2DAsync(xp, (size_t)dpad * 4, h->dX.p, (size_t)d * 4, (size_t)d * 4, n, cudaMemcpyDeviceToDevice, st));
        GS_CUDA(launch_split_tf32(xp, xh, xl, (size_t)n * dpad, st));
        TcMap mh, ml;
        GS_CUDA(tc_make_map(&mh, xh, n, dpad, dpad));
        GS_CUDA(tc_make_map(&ml, xl, n, dpad, dpad));
        TcBatch hb{0, 0, 0, dpad, bs.as<float>(), ld32};
        GS_CUDA(cudaMemcpyAsync(bb.p, &hb, sizeof hb, cudaMemcpyHostToDevice, st));
        h->tt.begin(h->evp, st);
        GS_CUDA(launch_gemm_nt_tf32x3(mh, ml, mh, ml, bb.as<TcBatch>(), 1, n, n, 1.0f, false, st, true));
        h->tt.end(h->evp, st, 3.0 * 2.0 * n * (double)n * dpad);
        GS_CUDA(launch_widen_gram(bs.as<float>(), n, ld32, h->dS.as<double>(), h->dXsq.as<double>(), st));
        pf.launches += 3;
    } else {
        GS_CUDA(launch_gram_f64(h->x_dtype == GS_F64 ? h->dX64.p : h->dX.p, h->x_dtype, n, d, h->dS.as<double>(), h->dXsq.as<double>(), st));
        pf.launches++;
    }
    pf.gram_flops = 2.0 * n * (double)n * d;
    pf.gram_bytes = (double)n * d * 4 + (double)n * n * ((flags & GS_GRAM_TENSOR) ? 4 : 8);
    tm.mark(0);

    // ---- 2. sub-problem row lists per (fold, pair): class a rows then class b rows, train rows only ----
    std::vector<int> rows_all;
    std::vector<int> sp_off((size_t)n_splits * n_pairs + 1, 0), sp_npos((size_t)n_splits * n_pairs, 0);
    int lmax = 0;
    for (int k = 0; k < n_splits; k++) {
        int p = 0;
        for (int a = 0; a < nc; a++)
            for (int b = a + 1; b < nc; b++, p++) {
                const size_t s = (size_t)k * n_pairs + p;
                sp_off[s] = (int)rows_all.size();
                for (int r = h->class_start[a]; r < h->class_start[a + 1]; r++)
                    if (refit || h->is_train(r, k)) rows_all.push_back(r);
                sp_npos[s] = (int)rows_all.size() - sp_off[s];
                for (int r = h->class_start[b]; r < h->class_start[b + 1]; r++)
                    if (refit || h->is_train(r, k)) rows_all.push_back(r);
                const int l = (int)rows_all.size() - sp_off[s];
                if (sp_npos[s] == 0 || sp_npos[s] == l) {
                    gs_set_error(h, "gs_svc: a training fold lacks one of the classes"); return GS_ERR_ARG;
                }
                lmax = std::max(lmax, l);
            }
    }
    sp_off.back() = (int)rows_all.size();
    // column ranges of every sub-problem (see SmoProblem::nseg): maximal runs of its rows, gaps below 64 columns merged,
    // starts rounded down and ends rounded up to 4 floats (16-byte bulk copies); more than 4 runs -> whole-row copies
    std::vector<int> sp_nseg((size_t)n_splits * n_pairs, 0), sp_seg((size_t)n_splits * n_pairs * 8, 0);
    for (size_t s = 0; s + 1 < sp_off.size(); s++) {
        std::vector<int> rs(rows_all.begin() + sp_off[s], rows_all.begin() + sp_off[s + 1]);
        std::sort(rs.begin(), rs.end());
        std::vector<std::pair<int, int>> runs;                               // [start, end)
        for (int r : rs) {
            const int a0 = r & ~3, a1 = (r + 4) & ~3;
            if (!runs.empty() && a0 <= runs.back().second + 64) runs.back().second = std::max(runs.back().second, a1);
            else runs.emplace_back(a0, a1);
        }
        if (runs.empty() || runs.size() > 4) continue;
        sp_nseg[s] = (int)runs.size();
        for (size_t e = 0; e < runs.size(); e++) {
            sp_seg[s * 8 + e] = runs[e].first;
            sp_seg[s * 8 + 4 + e] = std::min(runs[e].second, (int)ldk) - runs[e].first;
        }
    }
    if (lmax > smo_max_rows() && lmax > smo_colown_max_rows(4) && lmax >= 16383) {
        gs_set_error(h, "gs_svc: sub-problem with " + std::to_string(lmax) + " rows exceeds the resident-state SMO kernel limit of " +
                            std::to_string(smo_max_rows()));
        return GS_ERR_UNSUPPORTED;
    }

    // ---- 3. group tasks by kernel matrix (kernel, gamma) ----
    std::map<std::pair<int, uint64_t>, int> gmap;
    std::vector<std::pair<int, double>> groups;         // (kernel, gamma)
    std::vector<int> task_group(n_tasks);
    for (int c = 0; c < n_cand; c++)
        for (int k = 0; k < n_splits; k++) {
            const double g = kernel[c] == GS_KERNEL_RBF ? gamma[(size_t)c * n_splits + k] : 0.0;
            if (kernel[c] == GS_KERNEL_RBF && !(g > 0) ) { gs_set_error(h, "gs_svc: gamma must be > 0"); return GS_ERR_ARG; }
            auto key = std::make_pair((int)kernel[c], dbits(g));
            auto it = gmap.find(key);
            if (it == gmap.end()) { it = gmap.emplace(key, (int)groups.size()).first; groups.emplace_back(kernel[c], g); }
            task_group[(size_t)c * n_splits + k] = it->second;
        }
    const int n_groups = (int)groups.size();
    std::vector<std::vector<int>> group_tasks(n_groups);
    for (int t = 0; t < n_tasks; t++) group_tasks[task_group[t]].push_back(t);

    // ---- 4. memory plan: kernel matrices are processed in batches that fit in free HBM ----
    const size_t kbytes = (size_t)n * ldk * 4;
    int gpb = n_groups;
    if (h->dK.cap < kbytes * (size_t)n_groups) {
        // Ask the driver only when the buffer has to grow: cudaMemGetInfo takes anything from 0.1 to 100+ ms on a busy box
        // (measured as 16-119 ms outliers of this phase with the Gram already in flight), and a repeated search of the same
        // shape needs no new plan.
        size_t free_b = 0, total_b = 0;
        GS_CUDA(cudaMemGetInfo(&free_b, &total_b));
        free_b += h->dK.cap;
        const size_t budget = (size_t)(free_b * 0.6);
        gpb = (int)std::max<size_t>(1, std::min<size_t>(n_groups, budget / std::max<size_t>(kbytes, 1)));
        GS_CUDA(h->dK.reserve(kbytes * gpb));
    }

    GS_CUDA(h->dWork[0].reserve(rows_all.size() * 4));
    GS_CUDA(cudaMemcpyAsync(h->dWork[0].p, rows_all.data(), rows_all.size() * 4, cudaMemcpyHostToDevice, st));
    pf.h2d_bytes += rows_all.size() * 4;
    const int *d_rows = h->dWork[0].as<int>();

    std::vector<int> cnt_host;            // per task: 4 counters
    std::vector<int> task_iter(n_tasks, 0), task_sv(n_tasks, 0);
    std::vector<double> task_fit_ms(n_tasks, 0.0);
    std::vector<int> all_counts((size_t)n_tasks * 4, 0);
    std::vector<double> task_score((size_t)n_tasks * 2, 0.0);         // non-default scorers: test, train
    std::vector<char> task_bad(n_tasks, 0);
    std::vector<int> class_counts;
    std::vector<unsigned long long> score_raw;
    if (!refit && h->score_kind != GS_SCORE_DEFAULT) {
        const int kd = h->score_kind;
        if (kd == GS_SCORE_NEG_MSE || kd == GS_SCORE_NEG_RMSE) { gs_set_error(h, "gs_svc: regression scorer on a classifier"); return GS_ERR_ARG; }
        if ((kd == GS_SCORE_ROC_AUC || kd == GS_SCORE_F1 || kd == GS_SCORE_PRECISION || kd == GS_SCORE_RECALL) && nc != 2) {
            gs_set_error(h, "gs_svc: this scorer is defined for binary problems only"); return GS_ERR_UNSUPPORTED;
        }
        if (h->score_pos >= nc) { gs_set_error(h, "gs_svc: positive class out of range"); return GS_ERR_ARG; }
    }
    int64_t total_iter = 0;
    double solve_bytes = 0;

    for (int g0 = 0; g0 < n_groups; g0 += gpb) {
        const int g1 = std::min(n_groups, g0 + gpb);
        // -- kernel matrices of this batch --
        GS_CUDA(h->dWork[7].reserve(64));
        GS_CUDA(cudaMemsetAsync(h->dWork[7].p, 0, 4, st));
        bool fast = true;
        for (int g = g0; g < g1; g++) {
            GS_CUDA(launch_kernel_matrix(h->dS.as<double>(), h->dXsq.as<double>(), n, groups[g].first, groups[g].second,
                                         h->dK.as<float>() + (size_t)(g - g0) * n * ldk, ldk, h->dWork[7].as<int>(), st));
            pf.launches++;
            fast = fast && groups[g].first == GS_KERNEL_RBF;
        }
        // The branch-free SMO instance needs rbf (QD == 1) and only positive normal floats in K.  The second condition is a
        // device flag the kernel-matrix kernels raise: both instances are enqueued and the wrong one returns at once
        // (SmoProblem::guard), so the host never waits in the middle of a search and everything it prepares below overlaps
        // the Gram and kernel-matrix kernels already in flight.
        if (getenv("B200GS_SMO_NOFAST") && atoi(getenv("B200GS_SMO_NOFAST"))) fast = false;   // development switch: general instance only, unguarded
        const int *d_guard = fast ? h->dWork[7].as<int>() : nullptr;
        tm.mark(1);
        // -- problems: ordered by (group, task, pair); column index == problem index --
        std::vector<SmoProblem> probs;
        std::vector<int> prob_task, group_first(g1 - g0 + 1, 0);
        std::vector<VoteTask> vtasks;
        std::vector<int> vtask_id;
        size_t wl = 0, ws = 0;            // workspace doubles / ints
        for (int g = g0; g < g1; g++) {
            group_first[g - g0] = (int)probs.size();
            for (int t : group_tasks[g]) {
                const int c = t / n_splits, k = t % n_splits;
                vtasks.push_back(VoteTask{(int)probs.size(), refit ? -100 : k});
                vtask_id.push_back(t);
                for (int p = 0; p < n_pairs; p++) {
                    const size_t s = (size_t)k * n_pairs + p;
                    SmoProblem P;
                    memset(&P, 0, sizeof P);
                    P.K = h->dK.as<float>() + (size_t)(g - g0) * n * ldk;
                    P.qd = groups[g].first == GS_KERNEL_LINEAR ? h->dXsq.as<double>() : nullptr;
                    P.rows = d_rows + sp_off[s];
                    P.l = sp_off[s + 1] - sp_off[s];
                    P.nseg = sp_nseg[s];
                    for (int e = 0; e < 4; e++) { P.seg_start[e] = sp_seg[s * 8 + e]; P.seg_len[e] = sp_seg[s * 8 + 4 + e]; }
                    P.n_pos = sp_npos[s];
                    P.ldk = ldk; P.C = Cv[c]; P.Cn = Cv[c]; P.eps = tol; P.max_iter = max_iter;
                    if (h->class_w_sets > 0) {               // C_i = C x class_weight[class of i] (svm.cpp:2441-2470 weighted_C)
                        const double *cw = &h->class_w[(size_t)(h->class_w_sets == 1 ? 0 : k) * nc];
                        int a_ = 0, b_ = 0, q_ = 0;
                        for (int a = 0; a < nc; a++) for (int b = a + 1; b < nc; b++, q_++) if (q_ == p) { a_ = a; b_ = b; }
                        P.C = Cv[c] * cw[a_]; P.Cn = Cv[c] * cw[b_];
                    }
                    P.shrinking = (flags & GS_NO_SHRINKING) ? 0 : 1;
                    P.guard = d_guard;
                    P.nslots = 0;
                    for (int e = 0; e < P.nseg; e++) P.nslots += P.seg_len[e];
                    const size_t wlen = ((size_t)std::max(P.l, P.nslots) + 3) & ~(size_t)3;   // by position or by slot, 32-byte multiples
                    P.alpha = (double *)wl; wl += wlen;         // offsets now, pointers below
                    P.Gbar = (double *)wl; wl += wlen;
                    P.scratch = (int *)ws; ws += 2 * (size_t)P.l + 64;
                    probs.push_back(P);
                    prob_task.push_back(t);
                }
            }
        }
        group_first[g1 - g0] = (int)probs.size();
        const int np = (int)probs.size();
        // workspaces
        GS_CUDA(h->dWork[1].reserve(wl * 8));
        GS_CUDA(h->dWork[2].reserve(ws * 4));
        GS_CUDA(h->dWork[3].reserve((size_t)np * n * 8));                 // coef columns
        GS_CUDA(h->dWork[4].reserve((size_t)np * n * 8));                 // decision columns
        GS_CUDA(h->dWork[5].reserve((size_t)np * (8 + 16 + 96) + 64));    // rho, info[4], ns[12]
        GS_CUDA(h->dWork[6].reserve((size_t)np * sizeof(SmoProblem) + (size_t)np * 4 + vtasks.size() * (sizeof(VoteTask) + 16) + 256));
        double *d_rho = h->dWork[5].as<double>();
        int *d_info = (int *)(d_rho + np);
        unsigned long long *d_ns = (unsigned long long *)(d_info + 4 * (size_t)np);
        GS_CUDA(cudaMemsetAsync(d_ns, 0, (size_t)np * 12 * 8, st));
        for (int q = 0; q < np; q++) {
            SmoProblem &P = probs[q];
            P.alpha = h->dWork[1].as<double>() + (size_t)P.alpha;
            P.Gbar = h->dWork[1].as<double>() + (size_t)P.Gbar;
            P.scratch = h->dWork[2].as<int>() + (size_t)P.scratch;
            P.coef = h->dWork[3].as<double>() + (size_t)q * n;
            P.out_rho = d_rho + q; P.out_info = d_info + 4 * (size_t)q; P.out_ns = d_ns + 12 * (size_t)q;
        }
        // Predicted cost = rows x predicted SMO iterations (gs_svc_predicted_iterations): the predicted-longest problems lead
        // the launch order and the cluster policy below works on cost ratios.
        std::vector<double> cost(np);
        for (int q = 0; q < np; q++) {
            const int t = prob_task[q];
            const auto &grp = groups[task_group[t]];
            cost[q] = gs_svc_predicted_iterations(grp.first, Cv[t / n_splits], grp.second, (int32_t)d) * (double)probs[q].l;
        }
        std::vector<int> order(np);
        std::iota(order.begin(), order.end(), 0);
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return cost[a] > cost[b]; });
        unsigned char *dmeta = h->dWork[6].as<unsigned char>();
        SmoProblem *d_probs = (SmoProblem *)dmeta;
        int *d_order = (int *)(dmeta + (size_t)np * sizeof(SmoProblem));
        size_t off = (size_t)np * sizeof(SmoProblem) + (size_t)np * 4;
        off = (off + 15) & ~(size_t)15;
        VoteTask *d_vt = (VoteTask *)(dmeta + off);
        off += vtasks.size() * sizeof(VoteTask);
        off = (off + 15) & ~(size_t)15;
        int *d_counts = (int *)(dmeta + off);
        GS_CUDA(cudaMemcpyAsync(d_probs, probs.data(), (size_t)np * sizeof(SmoProblem), cudaMemcpyHostToDevice, st));
        GS_CUDA(cudaMemcpyAsync(d_order, order.data(), (size_t)np * 4, cudaMemcpyHostToDevice, st));
        GS_CUDA(cudaMemcpyAsync(d_vt, vtasks.data(), vtasks.size() * sizeof(VoteTask), cudaMemcpyHostToDevice, st));
        GS_CUDA(cudaMemsetAsync(d_counts, 0, vtasks.size() * 16, st));
        GS_CUDA(cudaMemsetAsync(h->dWork[3].p, 0, (size_t)np * n * 8, st));
        pf.h2d_bytes += (size_t)np * sizeof(SmoProblem) + (size_t)np * 4 + vtasks.size() * sizeof(VoteTask);
        tm.mark(4);
        // -- solve --
        // Policy (measured on config 2 / config 4, profiles/): a 4-CTA cluster solves one problem at 3.5 us per iteration
        // against 6.4-7.1 us for the single-CTA kernel, but costs twice the SM-time per iteration.  So clusters are for the
        // critical path only:
        //   * fewer problems than SMs: everything on the widest cluster that fits;
        //   * otherwise the number of clustered problems minimises a three-term makespan model (below): none for a
        //     throughput-bound search (config 4), exactly the ten 66-68k-iteration problems for config 2 (leaving ONE of
        //     them on a single SM costs +33 %), nineteen for the denser 8-GPU weak-scaling grid.
        // Development switches: B200GS_SMO_CLUSTER (0/2/4/8),
        // B200GS_SMO_CLUSTER_N.
        std::string why;
        // single-CTA launches go to the slot-layout kernel (smo_lean.cu) when every problem of the batch has one
        int max_slots = 0;
        bool lean_ok = lmax < 16383 && !(getenv("B200GS_SMO_LEAN") && atoi(getenv("B200GS_SMO_LEAN")) == 0);
        for (int q = 0; q < np && lean_ok; q++) {
            lean_ok = probs[q].nseg > 0 && probs[q].nslots <= smo_lean_max_slots();
            max_slots = std::max(max_slots, probs[q].nslots);
        }
        auto launch_single = [&](const int *ord, int cnt, cudaStream_t s_, bool exclusive) -> cudaError_t {
            for (int inst = fast ? 1 : 0; inst >= 0; inst--) {              // branch-free instance, then the general one (guarded)
                const cudaError_t e = lean_ok ? launch_smo_lean(d_probs, ord, cnt, max_slots, inst == 1, exclusive, s_)
                                              : launch_smo(d_probs, ord, cnt, lmax, inst == 1, (int)ldk, s_, &why);
                if (e != cudaSuccess) return e;
                pf.launches++;
            }
            return cudaSuccess;
        };
        // Policy (measured on config 2 / config 4, profiles/): clusters and exclusive SMs buy LATENCY for the critical path at
        // the price of SM time (gs_svc_schedule above); a throughput-bound search (config 4) uses neither.
        //   * fewer problems than SMs: everything on the widest cluster that fits;
        //   * otherwise the three-tier schedule of the slot-layout kernel, or -- when a problem has no slot layout -- the
        //     two-tier schedule of the position-owned kernel (gs_svc_cluster_count).
        // Development switches: B200GS_SMO_CLUSTER (0/2/4/8), B200GS_SMO_CLUSTER_N, B200GS_SMO_EXCLUSIVE_N.
        int cl = 0, n_cl = 0, n_ex = 0;
        if (lmax > 2048) {
            if (np * 8 <= h->sm_count) { cl = 8; n_cl = np; }
            else if (np * 4 <= h->sm_count) { cl = 4; n_cl = np; }
            else if (np * 2 <= h->sm_count) { cl = 2; n_cl = np; }
            else {
                std::vector<double> sorted_cost(np);
                for (int q = 0; q < np; q++) sorted_cost[q] = cost[order[q]];
                if (lean_ok) gs_svc_schedule(sorted_cost.data(), np, h->sm_count, &n_cl, &n_ex);
                else n_cl = gs_svc_cluster_count(sorted_cost.data(), np, h->sm_count);
                if (n_cl > 0) cl = 4;
            }
        }
        if (const char *e = getenv("B200GS_SMO_CLUSTER")) { cl = atoi(e); if (n_cl == 0) n_cl = std::max(1, np * 6 / 100); }
        if (const char *e = getenv("B200GS_SMO_CLUSTER_N")) n_cl = std::min(np, atoi(e));
        if (!(cl == 2 || cl == 4 || cl == 8) || lmax > smo_colown_max_rows(cl) || lmax <= 2048) n_cl = 0;
        if (const char *e = getenv("B200GS_SMO_EXCLUSIVE_N")) n_ex = atoi(e);
        if (!lean_ok) n_ex = 0;
        n_ex = std::max(0, std::min(n_ex, np - n_cl));
        if (n_cl > 0 || n_ex > 0) {
            // The latency tiers must get their SMs before the shared-SM launch floods the GPU (a late start of the critical
            // path costs the makespan that much: measured 292 vs 333 ms when the order of arrival flipped).  So the cluster
            // kernel goes on the engine stream itself, in order behind the uploads; the exclusive and the shared launches go
            // on two more streams behind the same point plus a 30 / 60 us delay kernel; the engine stream joins them afterwards.
            cudaEvent_t ready = h->evp.get();
            cudaEventRecord(ready, st);
            cudaError_t ce = cudaSuccess;
            if (n_cl > 0) {
                for (int inst = fast ? 1 : 0; inst >= 0 && ce == cudaSuccess; inst--) {
                    ce = launch_smo_colown(d_probs, d_order, n_cl, lmax, cl, inst == 1, st);
                    pf.launches++;
                }
                if (ce != cudaSuccess) { gs_set_error(h, std::string("launch_smo_colown: ") + cudaGetErrorString(ce)); return GS_ERR_CUDA; }
            }
            if (n_ex > 0) {
                cudaEvent_t done = h->evp.get();
                cudaStreamWaitEvent(h->stream_hi, ready, 0);
                launch_delay(30000, h->stream_hi);
                ce = launch_single(d_order + n_cl, n_ex, h->stream_hi, true);
                if (ce != cudaSuccess) { gs_set_error(h, why.empty() ? std::string("launch_smo: ") + cudaGetErrorString(ce) : why); return why.empty() ? GS_ERR_CUDA : GS_ERR_UNSUPPORTED; }
                pf.launches++;
                cudaEventRecord(done, h->stream_hi);
                cudaStreamWaitEvent(st, done, 0);
            }
            if (np - n_cl - n_ex > 0) {
                cudaStream_t s2 = n_ex > 0 ? h->stream_lo : h->stream_hi;
                cudaEvent_t done = h->evp.get();
                cudaStreamWaitEvent(s2, ready, 0);
                launch_delay(n_ex > 0 ? 60000 : 30000, s2);
                ce = launch_single(d_order + n_cl + n_ex, np - n_cl - n_ex, s2, false);
                if (ce != cudaSuccess) { gs_set_error(h, why.empty() ? std::string("launch_smo: ") + cudaGetErrorString(ce) : why); return why.empty() ? GS_ERR_CUDA : GS_ERR_UNSUPPORTED; }
                pf.launches++;
                cudaEventRecord(done, s2);
                cudaStreamWaitEvent(st, done, 0);
            }
        } else {
            cudaError_t ce = launch_single(d_order, np, st, false);
            if (ce != cudaSuccess) { gs_set_error(h, why.empty() ? std::string("launch_smo: ") + cudaGetErrorString(ce) : why); return why.empty() ? GS_ERR_CUDA : GS_ERR_UNSUPPORTED; }
        }
        tm.mark(2);
        // -- score (skipped for refit) --
        if (!refit) {
            size_t part_doubles = 0;                                              // partial sums of the j-slabs
            std::vector<int> jch(g1 - g0, 1);
            for (int g = g0; g < g1; g++) {
                const int cols = group_first[g - g0 + 1] - group_first[g - g0];
                jch[g - g0] = decision_chunks(n, cols, h->sm_count);
                if (jch[g - g0] > 1) part_doubles = std::max(part_doubles, (size_t)jch[g - g0] * cols * n);
            }
            if (part_doubles) GS_CUDA(h->dWork[8].reserve(part_doubles * 8));
            for (int g = g0; g < g1; g++) {
                const int c0 = group_first[g - g0], c1 = group_first[g - g0 + 1], jc = jch[g - g0];
                GS_CUDA(launch_decision(h->dS.as<double>(), h->dXsq.as<double>(), n, groups[g].first, groups[g].second,
                                        h->dWork[3].as<double>() + (size_t)c0 * n, c1 - c0,
                                        h->dWork[4].as<double>() + (size_t)c0 * n, jc > 1 ? h->dWork[8].as<double>() : nullptr, jc, st));
                pf.launches += jc > 1 ? 2 : 1;
            }
            const int kind = h->score_kind, nvt = (int)vtasks.size();
            if (kind == GS_SCORE_DEFAULT) {
                GS_CUDA(launch_vote(h->dWork[4].as<double>(), d_rho, n, nc, h->dY.as<int>(), h->masks(),
                                    d_vt, nvt, d_counts, st));
            } else if (kind == GS_SCORE_ROC_AUC) {
                // rank statistic of the decision values already in HBM (scikit-learn: roc_auc_score(y, decision_function(X)))
                std::vector<int> meta((size_t)nvt * 2);
                for (int v = 0; v < nvt; v++) { meta[v] = vtasks[v].first_col; meta[nvt + v] = vtasks[v].fold; }
                GS_CUDA(h->dScore.reserve((size_t)nvt * (8 + 32)));
                unsigned long long *d_auc = h->dScore.as<unsigned long long>();
                int *d_meta = (int *)(d_auc + (size_t)nvt * 4);
                GS_CUDA(cudaMemcpyAsync(d_meta, meta.data(), meta.size() * 4, cudaMemcpyHostToDevice, st));
                GS_CUDA(cudaMemsetAsync(d_auc, 0, (size_t)nvt * 32, st));
                GS_CUDA(launch_auc_pairs_f64(h->dWork[4].as<double>(), n, n, h->class_start[1], h->masks(), d_meta, d_meta + nvt,
                                             nvt, -1, d_auc, st));
                score_raw.resize((size_t)nvt * 4);
                GS_CUDA(cudaMemcpyAsync(score_raw.data(), d_auc, (size_t)nvt * 32, cudaMemcpyDeviceToHost, st));
            } else {
                GS_CUDA(h->dScore.reserve((size_t)nvt * 2 * nc * 3 * 4));
                GS_CUDA(cudaMemsetAsync(h->dScore.p, 0, (size_t)nvt * 2 * nc * 3 * 4, st));
                GS_CUDA(launch_vote_classes(h->dWork[4].as<double>(), d_rho, n, nc, h->dY.as<int>(), h->masks(),
                                            d_vt, nvt, h->dScore.as<int>(), st));
                class_counts.resize((size_t)nvt * 2 * nc * 3);
                GS_CUDA(cudaMemcpyAsync(class_counts.data(), h->dScore.p, class_counts.size() * 4, cudaMemcpyDeviceToHost, st));
            }
            pf.launches++;
        }
        tm.mark(3);
        // -- results of this batch --
        std::vector<int> info((size_t)np * 4), counts(vtasks.size() * 4);
        std::vector<unsigned long long> ns((size_t)np * 12);
        std::vector<double> rho(np);
        GS_CUDA(cudaMemcpyAsync(info.data(), d_info, info.size() * 4, cudaMemcpyDeviceToHost, st));
        GS_CUDA(cudaMemcpyAsync(ns.data(), d_ns, ns.size() * 8, cudaMemcpyDeviceToHost, st));
        GS_CUDA(cudaMemcpyAsync(rho.data(), d_rho, rho.size() * 8, cudaMemcpyDeviceToHost, st));
        GS_CUDA(cudaMemcpyAsync(counts.data(), d_counts, counts.size() * 4, cudaMemcpyDeviceToHost, st));
        std::vector<double> coef_host;
        if (refit && pair_coef) {
            coef_host.resize((size_t)np * n);
            GS_CUDA(cudaMemcpyAsync(coef_host.data(), h->dWork[3].p, coef_host.size() * 8, cudaMemcpyDeviceToHost, st));
        }
        GS_CUDA(cudaStreamSynchronize(st));
        pf.d2h_bytes += info.size() * 4 + ns.size() * 8 + rho.size() * 8 + counts.size() * 4 + coef_host.size() * 8;
        tm.collect(acc, 5);
        tm.mark(-1);
        for (int q = 0; q < np; q++) {
            const int t = prob_task[q];
            task_iter[t] += info[(size_t)q * 4]; task_sv[t] += info[(size_t)q * 4 + 2];
            task_fit_ms[t] += (double)(ns[(size_t)q * 12 + 1] - ns[(size_t)q * 12]) * 1e-6;
            total_iter += info[(size_t)q * 4];
            // two gathered K rows of the problem's (initially full) active set per iteration
            solve_bytes += (double)info[(size_t)q * 4] * 2.0 * probs[q].l * 4.0;
            // a task whose solve went non-finite scores NaN; the caller applies error_score to THAT task only
            // (reference base_search.py:69,87: _fit_and_score(..., error_score) fills per task)
            if (!std::isfinite(rho[q])) { if (refit) { gs_set_error(h, "gs_svc_refit: non-finite intercept"); return GS_ERR_NUMERIC; } task_bad[t] = 1; }
        }
        if (getenv("B200GS_SMO_TIMELINE") && atoi(getenv("B200GS_SMO_TIMELINE"))) {
            // development aid: when each tier starts and ends (globaltimer of the sub-problems, ms after the first start)
            unsigned long long t0 = ~0ull;
            for (int q = 0; q < np; q++) if (ns[(size_t)q * 12]) t0 = std::min(t0, ns[(size_t)q * 12]);
            auto span = [&](int a, int b, const char *name) {
                if (b <= a) return;
                double s0 = 1e30, s1 = 0, e0 = 1e30, e1 = 0; long long it_max = 0;
                for (int i = a; i < b; i++) {
                    const int q = order[i];
                    const double st_ = (double)(ns[(size_t)q * 12] - t0) * 1e-6, en = (double)(ns[(size_t)q * 12 + 1] - t0) * 1e-6;
                    s0 = std::min(s0, st_); s1 = std::max(s1, st_); e0 = std::min(e0, en); e1 = std::max(e1, en);
                    it_max = std::max<long long>(it_max, info[(size_t)q * 4]);
                }
                fprintf(stderr, "[timeline] %-9s %4d problems: starts %.2f..%.2f ms, ends %.2f..%.2f ms, longest %lld iterations\n",
                        name, b - a, s0, s1, e0, e1, it_max);
            };
            span(0, n_cl, "cluster"); span(n_cl, n_cl + n_ex, "exclusive"); span(n_cl + n_ex, np, "shared");
            for (int i = 0; i < std::min(np, 16); i++) {
                const int q = order[i];
                fprintf(stderr, "[timeline]   #%d: %d iterations, %.2f -> %.2f ms (%.3f us/iteration)\n", i, info[(size_t)q * 4],
                        (double)(ns[(size_t)q * 12] - t0) * 1e-6, (double)(ns[(size_t)q * 12 + 1] - t0) * 1e-6,
                        (double)(ns[(size_t)q * 12 + 1] - ns[(size_t)q * 12]) * 1e-3 / std::max(1, info[(size_t)q * 4]));
            }
        }
        if (getenv("B200GS_SMO_PROF") && atoi(getenv("B200GS_SMO_PROF"))) {
            int qmax = 0;
            for (int q = 1; q < np; q++) if (info[(size_t)q * 4] > info[(size_t)qmax * 4]) qmax = q;
            const unsigned long long *pn = &ns[(size_t)qmax * 12];
            const double it = (double)info[(size_t)qmax * 4];
            // single-CTA kernel slots: scanA | bar1+redA | rowI+phaseB | bar2 | fetchJ+scalar | update
            // cluster kernel slots:    redA | xchg1 | rowI | phaseB | xchg2 | scalar | bar3 | rowJ | update
            fprintf(stderr, "[smo prof] longest problem: %d iters, %.1f ms (%.2f us/iter); cycles/iter by slot:", info[(size_t)qmax * 4],
                    (double)(pn[1] - pn[0]) * 1e-6, (double)(pn[1] - pn[0]) * 1e-3 / it);
            for (int e = 0; e < 10; e++) fprintf(stderr, " %.0f", pn[2 + e] / it);
            fprintf(stderr, "\n");
        }
        for (size_t v = 0; v < vtasks.size(); v++)
            for (int e = 0; e < 4; e++) all_counts[(size_t)vtask_id[v] * 4 + e] = counts[v * 4 + e];
        if (!refit && h->score_kind == GS_SCORE_ROC_AUC) {
            for (size_t v = 0; v < vtasks.size(); v++) {
                const int k = vtasks[v].fold;
                double na_te = 0, nb_te = 0, na_tr = 0, nb_tr = 0;            // rows of the first / second class inside / outside fold k
                for (int r = 0; r < n; r++) {
                    const bool b = r >= h->class_start[1];
                    if (h->is_test(r, k)) (b ? nb_te : na_te) += 1;
                    else if (h->is_train(r, k)) (b ? nb_tr : na_tr) += 1;
                }
                const unsigned long long *a = &score_raw[v * 4];
                task_score[(size_t)vtask_id[v] * 2 + 0] = na_te * nb_te > 0 ? ((double)a[0] + 0.5 * (double)a[1]) / (na_te * nb_te) : NAN;
                task_score[(size_t)vtask_id[v] * 2 + 1] = na_tr * nb_tr > 0 ? ((double)a[2] + 0.5 * (double)a[3]) / (na_tr * nb_tr) : NAN;
            }
        } else if (!refit && h->score_kind != GS_SCORE_DEFAULT) {
            for (size_t v = 0; v < vtasks.size(); v++)
                for (int sp = 0; sp < 2; sp++)
                    task_score[(size_t)vtask_id[v] * 2 + sp] =
                        gs_score_from_counts(h->score_kind, h->score_pos, nc, &class_counts[(v * 2 + sp) * nc * 3]);
        }
        if (refit) {
            for (int q = 0; q < np; q++) {
                if (rho_out) rho_out[q] = rho[q];
                if (pair_iter) pair_iter[q] = info[(size_t)q * 4];
                if (pair_coef)
                    for (int r = 0; r < n; r++) pair_coef[(size_t)q * n + h->perm[r]] = coef_host[(size_t)q * n + r];
            }
        }
    }
    cudaEventRecord(ev_end, st);
    GS_CUDA(cudaStreamSynchronize(st));
    tm.collect(acc, 5);
    cudaEventElapsedTime(&pf.ms_total, ev_begin, ev_end);
    pf.ms_tensor = h->tt.collect(); pf.tensor_flops = h->tt.flops;
    pf.ms_gram = acc[0]; pf.ms_kernel_matrix = acc[1]; pf.ms_solve = acc[2]; pf.ms_score = acc[3];
    pf.smo_iterations = total_iter;
    pf.solve_bytes = solve_bytes;

    if (!refit) {
        for (int t = 0; t < n_tasks; t++) {
            const int *cn = &all_counts[(size_t)t * 4];
            if (h->score_kind == GS_SCORE_DEFAULT) {
                test_scores[t] = cn[1] > 0 ? (double)cn[0] / (double)cn[1] : NAN;
                if (train_scores) train_scores[t] = cn[3] > 0 ? (double)cn[2] / (double)cn[3] : NAN;
            } else {
                test_scores[t] = task_score[(size_t)t * 2];
                if (train_scores) train_scores[t] = task_score[(size_t)t * 2 + 1];
            }
            if (task_bad[t]) { test_scores[t] = NAN; if (train_scores) train_scores[t] = NAN; }
            if (n_iter) n_iter[t] = task_iter[t];
            if (n_sv) n_sv[t] = task_sv[t];
            if (fit_ms) fit_ms[t] = (float)task_fit_ms[t];
            if (score_ms) score_ms[t] = pf.ms_score / (float)n_tasks;
        }
    }
    return GS_OK;
}

int gs_svc(gs_handle *h, int32_t n_cand, const int32_t *kernel, const double *C, const double *gamma, double tol,
           int32_t max_iter, uint32_t flags, double *test_scores, double *train_scores, int32_t *n_iter,
           int32_t *n_sv, float *fit_ms, float *score_ms)
{
    if (h && !test_scores) { gs_set_error(h, "gs_svc: test_scores is NULL"); return GS_ERR_ARG; }
    return svc_run(h, n_cand, kernel, C, gamma, tol, max_iter, flags, false, test_scores,
                   (flags & GS_RETURN_TRAIN) ? train_scores : nullptr, n_iter, n_sv, fit_ms, score_ms, nullptr, nullptr, nullptr);
}

int gs_svc_refit(gs_handle *h, int32_t kernel, double C, double gamma, double tol, int32_t max_iter, uint32_t flags,
                 double *pair_coef, double *rho, int32_t *n_iter)
{
    const int32_t k = kernel;
    return svc_run(h, 1, &k, &C, &gamma, tol, max_iter, flags, true, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                   pair_coef, rho, n_iter);
}

int gs_debug_gram(gs_handle *h, double *S_out, double *xsq_out)
{
    if (!h) return GS_ERR_ARG;
    if (h->n == 0) { gs_set_error(h, "gs_debug_gram: no dataset"); return GS_ERR_NO_DATA; }
    GS_CUDA(cudaSetDevice(h->device));
    const int n = (int)h->n, d = (int)h->d;
    GS_CUDA(h->dS.reserve((size_t)n * n * 8));
    GS_CUDA(h->dXsq.reserve((size_t)n * 8));
    GS_CUDA(launch_gram_f64(h->x_dtype == GS_F64 ? h->dX64.p : h->dX.p, h->x_dtype, n, d, h->dS.as<double>(), h->dXsq.as<double>(), h->stream));
    std::vector<double> S((size_t)n * n), xs(n);
    GS_CUDA(cudaMemcpyAsync(S.data(), h->dS.p, S.size() * 8, cudaMemcpyDeviceToHost, h->stream));
    GS_CUDA(cudaMemcpyAsync(xs.data(), h->dXsq.p, xs.size() * 8, cudaMemcpyDeviceToHost, h->stream));
    GS_CUDA(cudaStreamSynchronize(h->stream));
    for (int r = 0; r < n; r++) {
        if (xsq_out) xsq_out[h->perm[r]] = xs[r];
        if (S_out)
            for (int c = 0; c < n; c++) S_out[(size_t)h->perm[r] * n + h->perm[c]] = S[(size_t)r * n + c];
    }
    return GS_OK;
}

int gs_debug_kernel_matrix(gs_handle *h, int32_t kernel, double gamma, float *K_out)
{
    if (!h || !K_out) return GS_ERR_ARG;
    int st = gs_debug_gram(h, nullptr, nullptr);
    if (st) return st;
    const int n = (int)h->n;
    const int64_t ldk = ((int64_t)n + 31) & ~31LL;
    GS_CUDA(h->dK.reserve((size_t)n * ldk * 4));
    GS_CUDA(launch_kernel_matrix(h->dS.as<double>(), h->dXsq.as<double>(), n, kernel, gamma, h->dK.as<float>(), ldk, nullptr, h->stream));
    std::vector<float> K((size_t)n * ldk);
    GS_CUDA(cudaMemcpyAsync(K.data(), h->dK.p, K.size() * 4, cudaMemcpyDeviceToHost, h->stream));
    GS_CUDA(cudaStreamSynchronize(h->stream));
    for (int r = 0; r < n; r++)
        for (int c = 0; c < n; c++) K_out[(size_t)h->perm[r] * n + h->perm[c]] = K[(size_t)r * ldk + c];
    return GS_OK;
}

int gs_get_profile(const gs_handle *h, gs_profile *out)
{
    if (!h || !out) return GS_ERR_ARG;
    *out = h->prof;
    return GS_OK;
}

}  // extern "C"
