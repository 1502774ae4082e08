// linear.cu -- linear regressors on fold Grams: Ridge (gs_ridge / gs_ridge_refit) and Lasso / ElasticNet (gs_enet / gs_enet_refit).
//
// Ridge path (replaces sklearn Ridge.fit/score reached from reference base_search.py:83-87:
// linear_model/_ridge.py:919 fit, :964 _preprocess_data centring, :215-227 _solve_cholesky, base.py:716 r2):
//   1. Z = [X | y | 1]  (n x (d+2)); per CV fold k the Gram  G_k = Z_k^T Z_k  holds X^T X, X^T y, column sums,
//      y^T y, sum y and the row count of the fold at once.  One tcgen05 contraction per fold (gemm_tc.cu, 3xTF32
//      split, K-range = the fold's contiguous rows).  scikit-learn recomputes X^T X for each of the
//      n_alpha x n_folds fits (SURVEY.md 8a-a9); here it is built ONCE and the training statistics of fold k are
//      T - G_k with T = sum_k G_k (float64).
//   2. Per fold: centred normal matrix A_k = X^T X - n xbar xbar^T and rhs (float64 -> float32).
//   3. (A_k + alpha I) w = rhs for ALL alphas of a fold at once by conjugate gradients whose matrix product is the
//      same tensor-core contraction (P[alphas x d] times the symmetric A_k); the per-system vector updates and dot
//      products are one small kernel per iteration.  Converged systems freeze; non-convergence fails loudly.
//   4. R^2 (or -MSE / -RMSE) on the held-out fold and on the training rows from the Gram statistics in float64, no pass over
//      X: the quadratic forms w^T G w of all systems are one float64 tile product with a fused row-dot (ridge_quad_kernel).
// Splits whose test sets are no partition (gs_set_splits): one Gram per training / test ROW LIST of a split instead of
// T - G_k.  Sample weights (gs_set_sample_weight): a second, sqrt(w)-scaled copy of the row blocks gives the weighted training
// statistics; the scores stay unweighted.  Lasso / ElasticNet: steps 1, 2 and 4 as above, step 3 is scikit-learn's cyclic
// coordinate descent restated on (A_k, rhs) -- enet_cd_kernel below.
// With fit_intercept the Grams are formed from SHIFTED data, Z = [X - c | y - c_y | 1] with c the column means over all
// rows (float64 sums, rounded to float32): the raw-moment subtractions X^T X - n xbar xbar^T and yy - ys^2/n then cancel
// nothing even when a feature's mean dwarfs its spread (scikit-learn centres before forming products, _ridge.py:964).
// w and R^2 are invariant under the shift; the intercept gets c_y - c.w added back.
#include "common.cuh"
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

namespace {

constexpr int CG_MAX_ITER = 4000;
constexpr double CG_TOL = 1e-6;          // relative residual; fp32 Cholesky (sklearn) is accurate to ~cond*6e-8

// shift[j] = (float) mean over all rows of column j of [X | y]  (float64 accumulation); block = 32 columns x 32 row stripes
__global__ void column_means_kernel(const float *__restrict__ X, const float *__restrict__ y, int n, int d, float *__restrict__ shift)
{
    __shared__ double acc[32][33];
    const int j = blockIdx.x * 32 + threadIdx.x;
    double s = 0;
    if (j <= d)
        for (int r = threadIdx.y; r < n; r += 32) s += (double)(j < d ? X[(size_t)r * d + j] : y[r]);
    acc[threadIdx.y][threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.y == 0 && j <= d) {
        double t = 0;
        for (int q = 0; q < 32; q++) t += acc[q][threadIdx.x];
        shift[j] = (float)(t / (double)n);
    }
}

// (sample weights: the chunk list is doubled; chunks >= first_weighted build sqrt(w)-scaled rows, whose Grams are the weighted
// training statistics sum w z z^T, while the unweighted copy keeps serving the scores -- _fit_and_score weights the fit only)
// Zt[j][poff[b] + r] = X[row][j] - shift[j] (j<d) | y[row] - shift[d] (j==d) | 1 (j==d+1); rows of block b are row0[b] .. row0[b]+cnt[b],
// or rowidx[row0[b] .. row0[b]+cnt[b]) when the blocks are row lists (general splits: the training / test rows of a split)
__global__ void build_zt_kernel(const float *__restrict__ X, const float *__restrict__ y, const float *__restrict__ shift, int d, int n_blocks,
                                const int *__restrict__ row0, const int *__restrict__ cnt, const int *__restrict__ poff,
                                const int *__restrict__ rowidx, const float *__restrict__ sw, int first_weighted,
                                float *__restrict__ Zt, int64_t ldz)
{
    __shared__ float tile[32][33];
    const int b = blockIdx.z;
    if (b >= n_blocks) return;
    const int r0 = blockIdx.x * 32, j0 = blockIdx.y * 32;
    if (r0 >= cnt[b]) return;
    {   // coalesced read along j
        const int r = r0 + threadIdx.y, j = j0 + threadIdx.x;
        float v = 0.f;
        if (r < cnt[b]) {
            const int row = rowidx ? rowidx[row0[b] + r] : row0[b] + r;
            if (j < d) v = X[(size_t)row * d + j] - shift[j];
            else if (j == d) v = y[row] - shift[d];
            else if (j == d + 1) v = 1.f;
            if (sw && b >= first_weighted) v *= sqrtf(sw[row]);      // chunks of the weighted copy: rows scaled by sqrt(sample_weight)
        }
        tile[threadIdx.y][threadIdx.x] = v;
    }
    __syncthreads();
    {   // coalesced write along r
        const int j = j0 + threadIdx.y, r = r0 + threadIdx.x;
        if (j < d + 2 && r < cnt[b]) Zt[(size_t)j * ldz + poff[b] + r] = tile[threadIdx.x][threadIdx.y];
    }
}

// The Gram of a row block is contracted in chunks of <= TC_KCHUNK rows (the TMEM accumulator truncates); the chunk
// partials Gq are added here in float64: G_b = sum of the chunks of block b (chunks qs[b] .. qs[b+1]), T = sum_b G_b.
__global__ void sum_grams_kernel(const float *__restrict__ Gq, const int *__restrict__ qs, int n_blocks, int n_plain, int64_t per,
                                 float *__restrict__ G, double *__restrict__ T, double *__restrict__ Tw)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < per; i += (int64_t)gridDim.x * blockDim.x) {
        double tot = 0, totw = 0;                                   // blocks [0, n_plain): unweighted; [n_plain, n_blocks): weighted copy
        for (int b = 0; b < n_blocks; b++) {
            double s = 0;
            for (int q = qs[b]; q < qs[b + 1]; q++) s += (double)Gq[(size_t)q * per + i];
            G[(size_t)b * per + i] = (float)s;
            if (b < n_plain) tot += s; else totw += s;
        }
        T[i] = tot;
        if (Tw) Tw[i] = totw;
    }
}

// Per system-group g (a split, or "all rows" for the refit): training statistics S = T - G_test (test folds that
// partition the rows) or S = G_train (general splits: the split's own training block), centred normal matrix
// A (float32, [dp][dp], zero padded) and rhs (float32 [dp]); means kept in float64 for the intercept.
__global__ void build_systems_kernel(const double *__restrict__ T, const float *__restrict__ G, const int *__restrict__ test_block,
                                     const int *__restrict__ train_block, int wofs /* block offset of the weighted copy */,
                                     int d, int Dp, int dp, int fit_intercept, float *__restrict__ A, float *__restrict__ rhs,
                                     double *__restrict__ means /* [groups][dp + 3]: xbar[0..d), ybar, n_train, centred y^T y */)
{
    const int g = blockIdx.z;
    const int tb = test_block[g], trb = train_block[g];
    const float *Gt = tb >= 0 ? G + (size_t)(tb + wofs) * Dp * Dp : nullptr;
    const float *Gtr = trb >= 0 ? G + (size_t)(trb + wofs) * Dp * Dp : nullptr;
    auto S = [&](int a, int b) -> double {
        if (Gtr) return (double)Gtr[(size_t)a * Dp + b];
        return T[(size_t)a * Dp + b] - (Gt ? (double)Gt[(size_t)a * Dp + b] : 0.0);
    };
    const double ntr = S(d + 1, d + 1);
    const double ybar = fit_intercept ? S(d, d + 1) / ntr : 0.0;
    const int j = blockIdx.y * blockDim.y + threadIdx.y;
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= dp || l >= dp) return;
    double v = 0.0;
    if (j < d && l < d) {
        v = S(j, l);
        if (fit_intercept) v -= S(j, d + 1) * S(l, d + 1) / ntr;            // n xbar_j xbar_l
    }
    A[((size_t)g * dp + j) * dp + l] = (float)v;
    if (l == 0) {
        double r = 0.0;
        if (j < d) {
            r = S(j, d);
            if (fit_intercept) r -= S(j, d + 1) * ybar;                     // n xbar_j ybar
            means[(size_t)g * (dp + 3) + j] = fit_intercept ? S(j, d + 1) / ntr : 0.0;
        }
        rhs[(size_t)g * dp + j] = (float)r;
        if (j == 0) {
            means[(size_t)g * (dp + 3) + dp] = ybar; means[(size_t)g * (dp + 3) + dp + 1] = ntr;
            means[(size_t)g * (dp + 3) + dp + 2] = S(d, d) - (fit_intercept ? ntr * ybar * ybar : 0.0);
        }
    }
}

__device__ __forceinline__ double block_sum(double v, double *sh)
{
#pragma unroll
    for (int m = 16; m; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double r = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) r += sh[w];
    return r;
}

__device__ __forceinline__ void split_store(float v, float *hi, float *lo, size_t i)
{
    const float h = __uint_as_float(__float_as_uint(v) & 0xffffe000u);
    hi[i] = h; lo[i] = v - h;
}

// one CTA per system s = g * n_cand + c:  x = 0, r = p = rhs_g
__global__ void cg_init_kernel(const float *__restrict__ rhs, int n_cand, int dp, float *__restrict__ Xs, float *__restrict__ R,
                               float *__restrict__ P, float *__restrict__ Ph, float *__restrict__ Pl, double *__restrict__ rr,
                               double *__restrict__ bb, int *__restrict__ done)
{
    __shared__ double sh[32];
    const int s = blockIdx.x, g = s / n_cand;
    double acc = 0;
    for (int j = threadIdx.x; j < dp; j += blockDim.x) {
        const float v = rhs[(size_t)g * dp + j];
        const size_t i = (size_t)s * dp + j;
        Xs[i] = 0.f; R[i] = v; P[i] = v;
        split_store(v, Ph, Pl, i);
        acc += (double)v * v;
    }
    acc = block_sum(acc, sh);
    if (threadIdx.x == 0) { rr[s] = acc; bb[s] = acc; done[s] = acc == 0.0; }
}

// q = Q + alpha_c p;  a = rr / p.q;  x += a p;  r -= a q;  beta = rr' / rr;  p = r + beta p   (Hestenes-Stiefel CG)
__global__ void cg_step_kernel(const float *__restrict__ Q, const double *__restrict__ alphas, int n_cand, int dp,
                               float *__restrict__ Xs, float *__restrict__ R, float *__restrict__ P, float *__restrict__ Ph,
                               float *__restrict__ Pl, double *__restrict__ rr, const double *__restrict__ bb,
                               int *__restrict__ done, int *__restrict__ n_open, double tol2)
{
    __shared__ double sh[32];
    const int s = blockIdx.x, c = s % n_cand;
    if (done[s]) return;
    const float al = (float)alphas[c];
    float q[8], p[8], r[8];                                      // dp <= 8 * blockDim.x (256 threads)
    double pq = 0;
#pragma unroll
    for (int u = 0; u < 8; u++) {
        const int j = threadIdx.x + u * 256;
        p[u] = q[u] = r[u] = 0.f;
        if (j < dp) {
            const size_t i = (size_t)s * dp + j;
            p[u] = P[i];
            q[u] = Q[i] + al * p[u];
            pq += (double)p[u] * q[u];
        }
    }
    pq = block_sum(pq, sh);
    const double rr0 = rr[s];
    if (!(pq > 0)) {                                             // breakdown: only possible when p == 0 (already solved)
        if (threadIdx.x == 0) done[s] = 1;
        return;
    }
    const float a = (float)(rr0 / pq);
    double rn = 0;
#pragma unroll
    for (int u = 0; u < 8; u++) {
        const int j = threadIdx.x + u * 256;
        if (j < dp) {
            const size_t i = (size_t)s * dp + j;
            Xs[i] += a * p[u];
            r[u] = R[i] - a * q[u];
            R[i] = r[u];
            rn += (double)r[u] * r[u];
        }
    }
    rn = block_sum(rn, sh);
    const float beta = (float)(rn / rr0);
#pragma unroll
    for (int u = 0; u < 8; u++) {
        const int j = threadIdx.x + u * 256;
        if (j < dp) {
            const size_t i = (size_t)s * dp + j;
            const float pn = r[u] + beta * p[u];
            P[i] = pn;
            split_store(pn, Ph, Pl, i);
        }
    }
    if (threadIdx.x == 0) {
        rr[s] = rn;
        if (rn <= tol2 * bb[s]) done[s] = 1; else atomicAdd(n_open, 1);
    }
}

// ---- ElasticNet / Lasso: cyclic coordinate descent in the Gram domain -------------------------------------------------
// scikit-learn minimises  1/2 ||y - Xw||^2 + a ||w||_1 + b/2 ||w||^2  (a = alpha*l1_ratio*n, b = alpha*(1-l1_ratio)*n,
// linear_model/_coordinate_descent.py:781-782) by cyclic coordinate descent on the residual R = y - Xw
// (_cd_fast.pyx:243-506 enet_coordinate_descent).  Every quantity of that loop is a function of the centred training Gram
// A = X^T X, rhs = X^T y and y^T y, which the fold-Gram pipeline above already holds:
//     X_j . R = q_j  with  q = rhs - A w,       ||X_j||^2 = A_jj,       R . R = yy - w.rhs - w.q,       R . y = yy - w.rhs
// so one warp runs one (candidate, split) system: q in registers (coordinate k = 128 i + 4 lane + c in register 4 i + c),
// w in shared memory, one row of A (= column, A is symmetric) streamed from L2 per coordinate.  Same coordinate order,
// same stopping rule (max |dw| / max |w| <= tol, then duality gap <= tol * yy: _cd_fast.pyx:458-471, gap_enet :162-240)
// and the same gap-safe screening of provably-zero features (:399-422, :473-492).  State is float64 (scikit-learn: the dtype
// of X); A and rhs are the float32 system matrices.
template <int NI>
__global__ void __launch_bounds__(256) enet_cd_kernel(const float *__restrict__ A, const float *__restrict__ rhs,
                                                      const double *__restrict__ means, const double *__restrict__ alphas,
                                                      const double *__restrict__ l1_ratio, int n_cand, int nsys, int d, int dp,
                                                      int max_iter, double tol_rel, float *__restrict__ Xs,
                                                      int *__restrict__ n_iter_out, double *__restrict__ gap_out)
{
    extern __shared__ double enet_w[];
    constexpr unsigned FULL = 0xffffffffu;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int s = blockIdx.x * (blockDim.x >> 5) + warp;
    if (s >= nsys) return;                                    // whole warps leave; there is no block-level barrier below
    const int g = s / n_cand, c = s % n_cand;
    double *w = enet_w + (size_t)warp * (NI * 128);
    const float *Ag = A + (size_t)g * dp * dp, *bg = rhs + (size_t)g * dp;
    const double ntr = means[(size_t)g * (dp + 3) + dp + 1], yy = means[(size_t)g * (dp + 3) + dp + 2];
    const double alpha = alphas[c] * l1_ratio[c] * ntr, beta = alphas[c] * (1.0 - l1_ratio[c]) * ntr;
    const double tol = tol_rel * yy;

    double q[NI * 4];
    unsigned excl = 0;                                        // bit r: the coordinate of register r is screened out (or >= d)
#pragma unroll
    for (int i = 0; i < NI; i++)
#pragma unroll
        for (int cc = 0; cc < 4; cc++) {
            const int k = 128 * i + 4 * lane + cc;
            q[i * 4 + cc] = k < d ? (double)bg[k] : 0.0;
            w[k] = 0.0;
            if (k >= d) excl |= 1u << (i * 4 + cc);
        }
    __syncwarp();

    auto load_row = [&](int j, float4 *col) {
#pragma unroll
        for (int i = 0; i < NI; i++) {
            const int k = 128 * i + 4 * lane;
            col[i] = k < dp ? __ldg(reinterpret_cast<const float4 *>(Ag + (size_t)j * dp + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    auto axpy_row = [&](double a, const float4 *col) {         // q += a * A[:, j]
#pragma unroll
        for (int i = 0; i < NI; i++) {
            q[i * 4 + 0] += a * (double)col[i].x; q[i * 4 + 1] += a * (double)col[i].y;
            q[i * 4 + 2] += a * (double)col[i].z; q[i * 4 + 3] += a * (double)col[i].w;
        }
    };
    auto wsum = [&](double v) {
#pragma unroll
        for (int m = 16; m; m >>= 1) v += __shfl_xor_sync(FULL, v, m);
        return v;
    };

    double gap = 0.0;
    // duality gap of the current w (gap_enet, _cd_fast.pyx:162-240); not converged -> gap-safe screening (:473-492)
    auto converged = [&]() -> bool {
        double mx = 0, wb = 0, wq = 0, l1 = 0, l2 = 0, qq = 0;
#pragma unroll
        for (int r = 0; r < NI * 4; r++) {
            const int k = 128 * (r >> 2) + 4 * lane + (r & 3);
            if (k < d) {
                const double wk = w[k];
                mx = fmax(mx, fabs(q[r] - beta * wk));
                wb += wk * (double)bg[k]; wq += wk * q[r]; l1 += fabs(wk); l2 += wk * wk; qq += q[r] * q[r];
            }
        }
#pragma unroll
        for (int m = 16; m; m >>= 1) mx = fmax(mx, __shfl_xor_sync(FULL, mx, m));
        wb = wsum(wb); wq = wsum(wq); l1 = wsum(l1); l2 = wsum(l2); qq = wsum(qq);
        const double Rn2 = yy - wb - wq, Ry = yy - wb;
        double dn;
        if (alpha == 0.0) {                                   // formulation B (ridge) / OLS first-order condition
            dn = qq;
            gap = beta == 0.0 ? qq : Rn2 + 0.5 * beta * l2 - Ry + qq / (2.0 * beta);
        } else {                                              // formulation A (dual_gap_formulation_A, :138-159)
            dn = mx;
            const double primal = 0.5 * (Rn2 + beta * l2) + alpha * l1;
            const double scale = dn > alpha ? alpha / dn : 1.0;
            gap = primal - (-0.5 * scale * scale * (Rn2 + beta * l2) + scale * Ry);
        }
        if (gap <= tol) return true;
        if (alpha > 0.0) {
            const double thr = sqrt(2.0 * gap) / alpha, den = fmax(alpha, dn);
            unsigned nw = 0;                                  // decided on the X^T R of the gap, before any exclusion changes q
#pragma unroll
            for (int r = 0; r < NI * 4; r++) {
                if ((excl >> r) & 1u) continue;
                const int k = 128 * (r >> 2) + 4 * lane + (r & 3);
                const double akk = (double)Ag[(size_t)k * dp + k];
                const double dk = (1.0 - fabs((q[r] - beta * w[k]) / den)) / sqrt(akk + beta);
                if (!(dk <= thr)) nw |= 1u << r;
            }
#pragma unroll
            for (int r = 0; r < NI * 4; r++) {
                const int k = 128 * (r >> 2) + 4 * lane + (r & 3);
                const bool mine = (nw >> r) & 1u;
                unsigned m = __ballot_sync(FULL, mine && w[k] != 0.0);
                while (m) {                                   // R += w_j X_j ; w_j = 0
                    const int lo = __ffs(m) - 1;
                    m &= m - 1;
                    const int j = 128 * (r >> 2) + 4 * lo + (r & 3);
                    float4 col[NI];
                    load_row(j, col);
                    const double wj = __shfl_sync(FULL, w[k], lo);
                    axpy_row(wj, col);
                    if (lane == lo) w[k] = 0.0;
                }
            }
            excl |= nw;
            __syncwarp();
        }
        return false;
    };

    int n_iter = 0;
    if (!converged()) {
        int it = 0;
        for (; it < max_iter; it++) {
            double w_max = 0.0, d_w_max = 0.0;
#pragma unroll
            for (int i = 0; i < NI; i++) {
                for (int lo = 0; lo < 32; lo++) {
                    const int jb = 128 * i + 4 * lo;
                    if (jb >= d) break;
                    const unsigned ex = __shfl_sync(FULL, excl, lo);
#pragma unroll
                    for (int cc = 0; cc < 4; cc++) {
                        const int r = i * 4 + cc, j = jb + cc;
                        if ((ex >> r) & 1u) continue;
                        float4 col[NI];
                        load_row(j, col);
                        const float cself = cc == 0 ? col[i].x : cc == 1 ? col[i].y : cc == 2 ? col[i].z : col[i].w;
                        const double ajj = __shfl_sync(FULL, (double)cself, lo);
                        if (ajj == 0.0) continue;
                        const double qj = __shfl_sync(FULL, q[r], lo);
                        const double wj = __shfl_sync(FULL, lane == 0 ? w[j] : 0.0, 0);     // lane 0 alone reads and writes w[j]
                        const double tmp = qj + wj * ajj;                                    // X_j . (R + w_j X_j)
                        const double mag = fmax(fabs(tmp) - alpha, 0.0) / (ajj + beta);
                        const double wn = tmp > 0.0 ? mag : tmp < 0.0 ? -mag : 0.0;
                        if (wn != wj) {
                            axpy_row(wj - wn, col);
                            if (lane == 0) w[j] = wn;
                        }
                        d_w_max = fmax(d_w_max, fabs(wn - wj));
                        w_max = fmax(w_max, fabs(wn));
                    }
                }
            }
            __syncwarp();
            if (w_max == 0.0 || d_w_max / w_max <= tol_rel || it == max_iter - 1)
                if (converged()) break;
        }
        n_iter = it < max_iter ? it + 1 : max_iter;
    }
    __syncwarp();
    for (int k = lane; k < dp; k += 32) Xs[(size_t)s * dp + k] = (float)w[k];
    if (lane == 0) { n_iter_out[s] = n_iter; gap_out[s] = gap; }
}

template <int NI>
cudaError_t launch_enet_cd(const float *A, const float *rhs, const double *means, const double *alphas, const double *l1r, int n_cand,
                           int nsys, int d, int dp, int max_iter, double tol, float *Xs, int *n_iter, double *gap, cudaStream_t st)
{
    const size_t smem = (size_t)8 * NI * 128 * 8;
    cudaError_t e = cudaFuncSetAttribute(enet_cd_kernel<NI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    enet_cd_kernel<NI><<<(nsys + 7) / 8, 256, smem, st>>>(A, rhs, means, alphas, l1r, n_cand, nsys, d, dp, max_iter, tol, Xs, n_iter, gap);
    return cudaGetLastError();
}

// Quadratic forms w_s^T M w_s of every system s against its test-block Gram (z = 0) and its training statistics (z = 1):
// a float64 tile product C[s][j] = sum_l w_s[l] M[l][j] (M symmetric, so row l is read along j: coalesced) with the
// row-dot against w_s[j] fused into the epilogue.  One CTA = 64 systems x 64 columns j; the partial of column tile jt
// goes to part[s][z][jt] and is summed in a fixed order by ridge_r2_kernel (deterministic, no atomics).
constexpr int QT = 64, QL = 16;
__global__ void __launch_bounds__(256) ridge_quad_kernel(const float *__restrict__ Xs, const double *__restrict__ T,
                                                         const float *__restrict__ G, const int *__restrict__ test_block,
                                                         const int *__restrict__ train_block, int n_cand, int d, int Dp, int dp,
                                                         int njt, double *__restrict__ part)
{
    __shared__ double Ws[QL][QT + 1], Ms[QL][QT + 1];
    const int g = blockIdx.y, z = blockIdx.z;
    const int s0 = (blockIdx.x / njt) * QT, jt = blockIdx.x % njt, j0 = jt * QT;
    const int tb = test_block[g], trb = train_block[g];
    const float *Mf = z == 0 ? G + (size_t)tb * Dp * Dp : (trb >= 0 ? G + (size_t)trb * Dp * Dp : nullptr);   // else T (float64)
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int mj = threadIdx.x & 63, ml = threadIdx.x >> 6;
    const float *Wg = Xs + (size_t)g * n_cand * dp;
    double acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int k = 0; k < 4; k++) acc[i][k] = 0.0;
    for (int l0 = 0; l0 < d; l0 += QL) {
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int sl = ty + 16 * q, c = s0 + sl, l = l0 + tx;
            Ws[tx][sl] = (c < n_cand && l < d) ? (double)Wg[(size_t)c * dp + l] : 0.0;
            const int lm = l0 + ml + 4 * q, j = j0 + mj;                     // lm < Dp: d + 2 <= Dp and QL | Dp
            double v = 0.0;
            if (j < d && lm < d) v = Mf ? (double)Mf[(size_t)lm * Dp + j] : T[(size_t)lm * Dp + j];
            Ms[ml + 4 * q][mj] = v;
        }
        __syncthreads();
#pragma unroll
        for (int l = 0; l < QL; l++) {
            double a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; i++) { a[i] = Ws[l][ty + 16 * i]; b[i] = Ms[l][tx + 16 * i]; }
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int k = 0; k < 4; k++) acc[i][k] += a[i] * b[k];
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int c = s0 + ty + 16 * i;
        double v = 0.0;
        if (c < n_cand) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int j = j0 + tx + 16 * k;
                if (j < d) v += acc[i][k] * (double)Wg[(size_t)c * dp + j];
            }
        }
#pragma unroll
        for (int m = 8; m; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
        if (tx == 0 && c < n_cand) part[(((size_t)g * n_cand + c) * 2 + z) * njt + jt] = v;
    }
}

// R^2 (or -MSE / -RMSE) of system s on its test block and on its training rows, from Gram statistics in float64: the
// quadratic forms come from ridge_quad_kernel, the linear terms (rows d and d+1 of the symmetric Grams) are read here.
__global__ void ridge_r2_kernel(const float *__restrict__ Xs, const double *__restrict__ T, const float *__restrict__ G,
                                const int *__restrict__ test_block, const int *__restrict__ train_block,
                                const double *__restrict__ means, const double *__restrict__ part, int njt, int n_cand, int d, int Dp,
                                int dp, int fit_intercept, int kind, double *__restrict__ out /* [systems][2] */)
{
    __shared__ double sh[32];
    const int s = blockIdx.x, g = s / n_cand;
    const int tb = test_block[g], trb = train_block[g];
    const float *Gk = G + (size_t)tb * Dp * Dp;
    const float *Gtr = trb >= 0 ? G + (size_t)trb * Dp * Dp : nullptr;      // general splits: own training block; else T - Gk
    auto Tr = [&](int a, int b) -> double { return Gtr ? (double)Gtr[(size_t)a * Dp + b] : T[(size_t)a * Dp + b]; };
    double wxy_k = 0, wxy_t = 0, ws_k = 0, ws_t = 0, xbw = 0;
    for (int j = threadIdx.x; j < d; j += blockDim.x) {
        const double w = (double)Xs[(size_t)s * dp + j];
        wxy_k += w * (double)Gk[(size_t)d * Dp + j]; wxy_t += w * Tr(d, j);
        ws_k += w * (double)Gk[(size_t)(d + 1) * Dp + j]; ws_t += w * Tr(d + 1, j);
        xbw += w * means[(size_t)g * (dp + 3) + j];
    }
    wxy_k = block_sum(wxy_k, sh); wxy_t = block_sum(wxy_t, sh);
    ws_k = block_sum(ws_k, sh); ws_t = block_sum(ws_t, sh);
    xbw = block_sum(xbw, sh);
    if (threadIdx.x == 0) {
        double qk = 0, qt = 0;
        for (int t = 0; t < njt; t++) { qk += part[((size_t)s * 2) * njt + t]; qt += part[((size_t)s * 2 + 1) * njt + t]; }
        const double b0 = fit_intercept ? means[(size_t)g * (dp + 3) + dp] - xbw : 0.0;
        auto r2 = [&](double yy, double ys, double nn, double q, double wxy, double ws) {
            const double res = yy - 2 * wxy - 2 * b0 * ys + q + 2 * b0 * ws + nn * b0 * b0;
            const double tot = yy - ys * ys / nn;
            if (kind == GS_SCORE_NEG_MSE) return -res / nn;              // sklearn.metrics.mean_squared_error, negated by the scorer
            if (kind == GS_SCORE_NEG_RMSE) return -sqrt(fmax(res, 0.0) / nn);
            return 1.0 - res / tot;
        };
        const double yy_k = Gk[(size_t)d * Dp + d], ys_k = Gk[(size_t)d * Dp + d + 1], n_k = Gk[(size_t)(d + 1) * Dp + d + 1];
        const double yy_t = Tr(d, d), ys_t = Tr(d, d + 1), n_t = Tr(d + 1, d + 1);
        out[(size_t)s * 2] = r2(yy_k, ys_k, n_k, qk, wxy_k, ws_k);
        out[(size_t)s * 2 + 1] = Gtr ? r2(yy_t, ys_t, n_t, qt, wxy_t, ws_t)
                                     : r2(yy_t - yy_k, ys_t - ys_k, n_t - n_k, qt - qk, wxy_t - wxy_k, ws_t - ws_k);
    }
}

struct RidgeTimers { float gram = 0, solve = 0, score = 0, total = 0; };
// ElasticNet / Lasso instead of the Ridge CG solve: per-candidate l1_ratio, scikit-learn's tol / max_iter; outputs [n_cand][n_splits]
struct EnetSpec { const double *l1_ratio; double tol; int max_iter; int32_t *n_iter; double *dual_gap; };

// groups: fold k (test block k) for the search; one group with test block -1 for the refit
int ridge_run(gs_handle *h, int n_cand, const double *alpha, int fit_intercept, bool refit,
              double *test_scores, double *train_scores, double *coef_out, RidgeTimers *tmr, const EnetSpec *en = nullptr)
{
    if (!h) return GS_ERR_ARG;
    if (h->n == 0) { gs_set_error(h, "gs_ridge: no dataset (call gs_set_data first)"); return GS_ERR_NO_DATA; }
    if (h->classification) { gs_set_error(h, "gs_ridge: dataset has no regression targets"); return GS_ERR_ARG; }
    if (n_cand <= 0 || !alpha) { gs_set_error(h, "gs_ridge: bad arguments"); return GS_ERR_ARG; }
    for (int c = 0; c < n_cand; c++)
        if (!(alpha[c] >= 0)) { gs_set_error(h, "gs_ridge: alpha must be >= 0"); return GS_ERR_ARG; }
    if (h->score_kind != GS_SCORE_DEFAULT && h->score_kind != GS_SCORE_NEG_MSE && h->score_kind != GS_SCORE_NEG_RMSE) {
        gs_set_error(h, "gs_ridge: classification scorer on a regressor"); return GS_ERR_ARG;
    }
    GS_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const int n = (int)h->n, d = (int)h->d, ns = h->n_splits;
    const int D = d + 2, Dp = (D + 31) & ~31, dp = (d + 31) & ~31;
    if (dp > 8 * 256) { gs_set_error(h, "gs_ridge: more than 2048 features is not supported by the CG kernels"); return GS_ERR_UNSUPPORTED; }
    if (en) {
        if (dp > 1024) { gs_set_error(h, "gs_enet: more than 1024 features is not supported by the coordinate-descent kernel"); return GS_ERR_UNSUPPORTED; }
        if (!en->l1_ratio || !(en->tol >= 0) || en->max_iter < 1) { gs_set_error(h, "gs_enet: bad arguments"); return GS_ERR_ARG; }
        for (int c = 0; c < n_cand; c++)
            if (!(en->l1_ratio[c] >= 0 && en->l1_ratio[c] <= 1)) { gs_set_error(h, "gs_enet: l1_ratio must be in [0, 1]"); return GS_ERR_ARG; }
    }

    // row blocks.  Test folds that partition the rows: one contiguous block per fold (rows are sorted by fold; fold -1
    // rows, never tested, form a trailing block), training statistics = T - G_fold.  General splits (gs_set_splits):
    // blocks 2k / 2k+1 are the row lists of split k's training / test set, each contracted on its own.
    const bool lists = !h->partition;
    std::vector<int> row0, cnt, rowidx;
    if (lists && refit) { row0.push_back(0); cnt.push_back(n); }
    else if (lists) {
        for (int k = 0; k < ns; k++)
            for (int side = 0; side < 2; side++) {
                row0.push_back((int)rowidx.size());
                for (int r = 0; r < n; r++)
                    if (side == 0 ? h->is_train(r, k) : h->is_test(r, k)) rowidx.push_back(r);
                cnt.push_back((int)rowidx.size() - row0.back());
                if (cnt.back() == 0) {
                    gs_set_error(h, std::string("gs_ridge: split ") + std::to_string(k) + " has an empty " + (side ? "test" : "training") + " set");
                    return GS_ERR_ARG;
                }
            }
    } else {
        int r = 0;
        for (int k = 0; k < ns; k++) {
            int c = 0;
            while (r + c < n && h->fold[r + c] == k) c++;
            row0.push_back(r); cnt.push_back(c); r += c;
        }
        if (r < n) { row0.push_back(r); cnt.push_back(n - r); }
    }
    // sample weights (gs_set_sample_weight): every block once more, its rows scaled by sqrt(w) -- the second copy gives the
    // weighted training statistics, the first one the (unweighted) scores
    const bool weighted = !h->sample_w.empty();
    const int nb_plain = (int)row0.size();
    if (weighted)
        for (int b = 0; b < nb_plain; b++) { row0.push_back(row0[b]); cnt.push_back(cnt[b]); }
    const int nb = (int)row0.size();
    // contraction chunks: <= TC_KCHUNK rows each, zero-padded to a multiple of 32 columns of Z^T
    std::vector<int> crow0, ccnt, qs(nb + 1, 0);
    for (int b = 0; b < nb; b++) {
        for (int r = 0; r < cnt[b]; r += TC_KCHUNK) { crow0.push_back(row0[b] + r); ccnt.push_back(std::min(TC_KCHUNK, cnt[b] - r)); }
        qs[b + 1] = (int)crow0.size();
    }
    const int nq = (int)crow0.size();
    const int first_weighted = weighted ? qs[nb_plain] : nq;
    std::vector<int> poff(nq + 1, 0);
    for (int q = 0; q < nq; q++) poff[q + 1] = poff[q] + ((ccnt[q] + 31) & ~31);
    const int64_t ldz = poff[nq];
    const int groups = refit ? 1 : ns;
    const int nsys = groups * n_cand;

    h->evp.reset(); h->tt.reset();
    cudaEvent_t ev[5];
    for (auto &e : ev) e = h->evp.get();
    cudaEventRecord(ev[0], st);

    // ---- buffers ----
    DevBuf &bZ = h->dWork[0], &bZh = h->dWork[1], &bZl = h->dWork[2], &bG = h->dWork[3], &bMisc = h->dWork[4],
           &bA = h->dWork[5], &bV = h->dWork[6], &bMeta = h->dWork[7];
    GS_CUDA(bZ.reserve((size_t)Dp * ldz * 4)); GS_CUDA(bZh.reserve((size_t)Dp * ldz * 4)); GS_CUDA(bZl.reserve((size_t)Dp * ldz * 4));
    GS_CUDA(bG.reserve((size_t)(nb + nq) * Dp * Dp * 4));                   // per-block Grams, then the chunk partials
    const size_t tBytes = (size_t)Dp * Dp * 8 * 2, meansBytes = (size_t)groups * (dp + 3) * 8;
    GS_CUDA(bMisc.reserve(tBytes + meansBytes + (size_t)nsys * (8 + 8 + 16) + (size_t)n_cand * 8 + (size_t)(d + 1) * 4 + 256));
    GS_CUDA(bA.reserve((size_t)groups * dp * dp * 4 * 3 + (size_t)groups * dp * 4));
    GS_CUDA(bV.reserve((size_t)nsys * dp * 4 * (6 + (size_t)((dp + TC_KCHUNK - 1) / TC_KCHUNK))));
    const int nkc = (dp + TC_KCHUNK - 1) / TC_KCHUNK;                          // K-chunks of the CG product
    GS_CUDA(bMeta.reserve((size_t)(nq * 3 + nb + 1 + 2 * groups) * 4 + (size_t)(nq + groups * nkc) * sizeof(TcBatch) + (size_t)nsys * 4 + rowidx.size() * 4 + 128));
    double *dT = bMisc.as<double>(), *dTw = dT + (size_t)Dp * Dp;          // totals of the unweighted / weighted block Grams
    double *dMeans = dTw + (size_t)Dp * Dp;
    double *dRR = dMeans + (size_t)groups * (dp + 3), *dBB = dRR + nsys, *dOut = dBB + nsys, *dAlpha = dOut + 2 * (size_t)nsys;
    float *dShift = reinterpret_cast<float *>(dAlpha + n_cand);               // [d + 1] column shifts of [X | y]
    float *dA = bA.as<float>(), *dAh = dA + (size_t)groups * dp * dp, *dAl = dAh + (size_t)groups * dp * dp,
          *dRhs = dAl + (size_t)groups * dp * dp;
    float *dX = bV.as<float>(), *dR = dX + (size_t)nsys * dp, *dP = dR + (size_t)nsys * dp, *dPh = dP + (size_t)nsys * dp,
          *dPl = dPh + (size_t)nsys * dp, *dQ = dPl + (size_t)nsys * dp, *dQp = dQ + (size_t)nsys * dp;
    float *dGq = bG.as<float>() + (size_t)nb * Dp * Dp;
    int *dRow0 = bMeta.as<int>(), *dCnt = dRow0 + nq, *dPoff = dCnt + nq, *dQs = dPoff + nq, *dTestBlock = dQs + nb + 1,
        *dTrainBlock = dTestBlock + groups;
    int *dDone = dTrainBlock + groups;
    int *dOpen = dDone + nsys;
    TcBatch *dBatchG = reinterpret_cast<TcBatch *>(((uintptr_t)(dOpen + 4) + 15) & ~(uintptr_t)15);
    TcBatch *dBatchCG = dBatchG + nq;
    int *dRowIdx = lists && !rowidx.empty() ? reinterpret_cast<int *>(dBatchCG + (size_t)groups * nkc) : nullptr;

    std::vector<int> testBlock(groups), trainBlock(groups);
    for (int g = 0; g < groups; g++) {
        testBlock[g] = refit ? -1 : (lists ? 2 * g + 1 : g);
        trainBlock[g] = (!refit && lists) ? 2 * g : -1;
    }
    GS_CUDA(cudaMemcpyAsync(dRow0, crow0.data(), nq * 4, cudaMemcpyHostToDevice, st));
    GS_CUDA(cudaMemcpyAsync(dCnt, ccnt.data(), nq * 4, cudaMemcpyHostToDevice, st));
    GS_CUDA(cudaMemcpyAsync(dPoff, poff.data(), nq * 4, cudaMemcpyHostToDevice, st));
    GS_CUDA(cudaMemcpyAsync(dQs, qs.data(), (nb + 1) * 4, cudaMemcpyHostToDevice, st));
    GS_CUDA(cudaMemcpyAsync(dTestBlock, testBlock.data(), groups * 4, cudaMemcpyHostToDevice, st));
    GS_CUDA(cudaMemcpyAsync(dTrainBlock, trainBlock.data(), groups * 4, cudaMemcpyHostToDevice, st));
    if (dRowIdx) GS_CUDA(cudaMemcpyAsync(dRowIdx, rowidx.data(), rowidx.size() * 4, cudaMemcpyHostToDevice, st));
    GS_CUDA(cudaMemcpyAsync(dAlpha, alpha, (size_t)n_cand * 8, cudaMemcpyHostToDevice, st));
    std::vector<TcBatch> bg(nq), bc;
    for (int q = 0; q < nq; q++) bg[q] = TcBatch{0, 0, poff[q], poff[q + 1], dGq + (size_t)q * Dp * Dp, (int64_t)Dp};
    for (int kc = 0; kc < nkc; kc++)                                               // partial kc of Q = P A_g
        for (int g = 0; g < groups; g++)
            bc.push_back(TcBatch{g * n_cand, g * dp, kc * TC_KCHUNK, std::min(dp, (kc + 1) * TC_KCHUNK),
                                 dQp + (size_t)kc * nsys * dp + (size_t)g * n_cand * dp, (int64_t)dp});
    GS_CUDA(cudaMemcpyAsync(dBatchG, bg.data(), nq * sizeof(TcBatch), cudaMemcpyHostToDevice, st));
    GS_CUDA(cudaMemcpyAsync(dBatchCG, bc.data(), bc.size() * sizeof(TcBatch), cudaMemcpyHostToDevice, st));
    int64_t launches = 0;

    // ---- 1. Z^T, split, fold Grams on tensor cores ----
    GS_CUDA(cudaMemsetAsync(bZ.p, 0, (size_t)Dp * ldz * 4, st));
    {
        dim3 grid((TC_KCHUNK + 31) / 32, (D + 31) / 32, nq), block(32, 32);
        if (fit_intercept) column_means_kernel<<<(d + 1 + 31) / 32, dim3(32, 32), 0, st>>>(h->dX.as<float>(), h->dYt.as<float>(), n, d, dShift);
        else GS_CUDA(cudaMemsetAsync(dShift, 0, (size_t)(d + 1) * 4, st));
        GS_CUDA(cudaGetLastError());
        build_zt_kernel<<<grid, block, 0, st>>>(h->dX.as<float>(), h->dYt.as<float>(), dShift, d, nq, dRow0, dCnt, dPoff, dRowIdx,
                                                weighted ? h->dSw.as<float>() : nullptr, first_weighted, bZ.as<float>(), ldz);
        GS_CUDA(cudaGetLastError());
    }
    GS_CUDA(launch_split_tf32(bZ.as<float>(), bZh.as<float>(), bZl.as<float>(), (size_t)Dp * ldz, st));
    TcMap mzh, mzl;
    GS_CUDA(tc_make_map(&mzh, bZh.as<float>(), Dp, ldz, ldz));
    GS_CUDA(tc_make_map(&mzl, bZl.as<float>(), Dp, ldz, ldz));
    h->tt.begin(h->evp, st);
    GS_CUDA(launch_gemm_nt_tf32x3(mzh, mzl, mzh, mzl, dBatchG, nq, D, D, 1.0f, false, st, true));   // Gram: upper tiles + mirror
    h->tt.end(h->evp, st, 3.0 * 2.0 * (double)D * D * (double)ldz * (((D + 127) / 128 + 1) / (2.0 * ((D + 127) / 128))));   // tiles on/above the diagonal
    sum_grams_kernel<<<592, 256, 0, st>>>(dGq, dQs, nb, nb_plain, (int64_t)Dp * Dp, bG.as<float>(), dT, weighted ? dTw : nullptr);
    GS_CUDA(cudaGetLastError());
    launches += 5;
    cudaEventRecord(ev[1], st);

    // ---- 2. per-group centred systems ----
    {
        dim3 block(32, 8), grid((dp + 31) / 32, (dp + 7) / 8, groups);
        build_systems_kernel<<<grid, block, 0, st>>>(weighted ? dTw : dT, bG.as<float>(), dTestBlock, dTrainBlock, weighted ? nb_plain : 0, d, Dp, dp,
                                                     fit_intercept, dA, dRhs, dMeans);
        GS_CUDA(cudaGetLastError());
    }
    int it = 0;
    if (en) {
        // ---- 3'. ElasticNet / Lasso: one warp per system, coordinate descent on (A_g, rhs_g) ----
        GS_CUDA(cudaMemcpyAsync(dBB, en->l1_ratio, (size_t)n_cand * 8, cudaMemcpyHostToDevice, st));
        cudaError_t e;
        if (dp <= 128) e = launch_enet_cd<1>(dA, dRhs, dMeans, dAlpha, dBB, n_cand, nsys, d, dp, en->max_iter, en->tol, dX, dDone, dRR, st);
        else if (dp <= 256) e = launch_enet_cd<2>(dA, dRhs, dMeans, dAlpha, dBB, n_cand, nsys, d, dp, en->max_iter, en->tol, dX, dDone, dRR, st);
        else if (dp <= 512) e = launch_enet_cd<4>(dA, dRhs, dMeans, dAlpha, dBB, n_cand, nsys, d, dp, en->max_iter, en->tol, dX, dDone, dRR, st);
        else e = launch_enet_cd<8>(dA, dRhs, dMeans, dAlpha, dBB, n_cand, nsys, d, dp, en->max_iter, en->tol, dX, dDone, dRR, st);
        GS_CUDA(e);
        launches++;
    } else {
        GS_CUDA(launch_split_tf32(dA, dAh, dAl, (size_t)groups * dp * dp, st));
        TcMap mah, mal, mph, mpl;
        GS_CUDA(tc_make_map(&mah, dAh, (int64_t)groups * dp, dp, dp));
        GS_CUDA(tc_make_map(&mal, dAl, (int64_t)groups * dp, dp, dp));
        GS_CUDA(tc_make_map(&mph, dPh, nsys, dp, dp));
        GS_CUDA(tc_make_map(&mpl, dPl, nsys, dp, dp));
        launches += 2;

        // ---- 3. batched CG: Q = P A_g on tensor cores, vector updates in cg_step_kernel ----
        cg_init_kernel<<<nsys, 256, 0, st>>>(dRhs, n_cand, dp, dX, dR, dP, dPh, dPl, dRR, dBB, dDone);
        GS_CUDA(cudaGetLastError());
        launches++;
        int open = 1;
        while (open > 0 && it < CG_MAX_ITER) {
            for (int rep = 0; rep < 4; rep++, it++) {
                h->tt.begin(h->evp, st);
                GS_CUDA(launch_gemm_nt_tf32x3(mph, mpl, mah, mal, dBatchCG, groups * nkc, n_cand, dp, 1.0f, false, st));
                h->tt.end(h->evp, st, 3.0 * 2.0 * (double)groups * n_cand * (double)dp * dp);
                if (nkc > 1) GS_CUDA(launch_sum_partials(dQp, nkc, (int64_t)nsys * dp, dQ, st));
                GS_CUDA(cudaMemsetAsync(dOpen, 0, 4, st));
                cg_step_kernel<<<nsys, 256, 0, st>>>(nkc > 1 ? dQ : dQp, dAlpha, n_cand, dp, dX, dR, dP, dPh, dPl, dRR, dBB, dDone, dOpen, CG_TOL * CG_TOL);
                GS_CUDA(cudaGetLastError());
                launches += 2;
            }
            GS_CUDA(cudaMemcpyAsync(&open, dOpen, 4, cudaMemcpyDeviceToHost, st));
            GS_CUDA(cudaStreamSynchronize(st));
        }
        if (open > 0) {
            gs_set_error(h, "gs_ridge: conjugate gradients did not converge in " + std::to_string(CG_MAX_ITER) + " iterations for " +
                                std::to_string(open) + " systems (ill-conditioned normal matrix)");
            return GS_ERR_NUMERIC;
        }
    }
    cudaEventRecord(ev[2], st);

    // ---- 4. scores / coefficients ----
    if (!refit) {
        const int njt = (d + QT - 1) / QT;
        GS_CUDA(h->dWork[8].reserve((size_t)nsys * 2 * njt * 8));
        double *dPart = h->dWork[8].as<double>();
        ridge_quad_kernel<<<dim3(((n_cand + QT - 1) / QT) * njt, groups, 2), 256, 0, st>>>(dX, dT, bG.as<float>(), dTestBlock, dTrainBlock,
                                                                                          n_cand, d, Dp, dp, njt, dPart);
        GS_CUDA(cudaGetLastError());
        ridge_r2_kernel<<<nsys, 128, 0, st>>>(dX, dT, bG.as<float>(), dTestBlock, dTrainBlock, dMeans, dPart, njt, n_cand, d, Dp, dp,
                                              fit_intercept, h->score_kind, dOut);
        GS_CUDA(cudaGetLastError());
        launches++;
        launches++;
        std::vector<double> out((size_t)nsys * 2);
        GS_CUDA(cudaMemcpyAsync(out.data(), dOut, out.size() * 8, cudaMemcpyDeviceToHost, st));
        cudaEventRecord(ev[3], st);
        GS_CUDA(cudaStreamSynchronize(st));
        // R^2 of a set whose targets are all equal: the total sum of squares is 0, and the one ridge_r2_kernel divides by is
        // float32 rounding noise of the Gram statistics (a large finite value of either sign, or inf / NaN).  scikit-learn's
        // r2_score (force_finite=True) gives 1.0 for an exact prediction and 0.0 otherwise; the residual from Gram statistics
        // cannot certify an exact zero, so such a set scores 0.0.
        auto constant_targets = [&](int k, bool test) {
            bool any = false;
            float v = 0.f;
            for (int r = 0; r < n; r++) {
                if (!(test ? h->is_test(r, k) : h->is_train(r, k))) continue;
                if (!any) { v = h->yt[r]; any = true; }
                else if (h->yt[r] != v) return false;
            }
            return any;
        };
        for (int g = 0; g < groups; g++) {
            const bool r2 = h->score_kind == GS_SCORE_DEFAULT;
            const bool const_te = r2 && constant_targets(g, true), const_tr = r2 && train_scores && constant_targets(g, false);
            for (int c = 0; c < n_cand; c++) {
                const size_t s = (size_t)g * n_cand + c;
                test_scores[(size_t)c * ns + g] = const_te ? 0.0 : out[s * 2];
                if (train_scores) train_scores[(size_t)c * ns + g] = const_tr ? 0.0 : out[s * 2 + 1];
            }
        }
        h->prof.d2h_bytes = (int64_t)out.size() * 8;
    } else {
        std::vector<float> w(dp), shift(d + 1);
        std::vector<double> means(dp + 3);
        GS_CUDA(cudaMemcpyAsync(w.data(), dX, (size_t)dp * 4, cudaMemcpyDeviceToHost, st));
        GS_CUDA(cudaMemcpyAsync(shift.data(), dShift, (size_t)(d + 1) * 4, cudaMemcpyDeviceToHost, st));
        GS_CUDA(cudaMemcpyAsync(means.data(), dMeans, (size_t)(dp + 3) * 8, cudaMemcpyDeviceToHost, st));
        cudaEventRecord(ev[3], st);
        GS_CUDA(cudaStreamSynchronize(st));
        double b0 = means[dp] + (double)shift[d];                  // intercept in the caller's (unshifted) coordinates
        for (int j = 0; j < d; j++) {
            const int o = j;                                       // feature order is unchanged
            coef_out[o] = (double)w[j];
            b0 -= (means[j] + (double)shift[j]) * (double)w[j];
        }
        coef_out[d] = fit_intercept ? b0 : 0.0;
    }
    if (en) {                                                      // sweeps and duality gap of every system
        std::vector<int> ni(nsys);
        std::vector<double> gp(nsys);
        GS_CUDA(cudaMemcpyAsync(ni.data(), dDone, (size_t)nsys * 4, cudaMemcpyDeviceToHost, st));
        GS_CUDA(cudaMemcpyAsync(gp.data(), dRR, (size_t)nsys * 8, cudaMemcpyDeviceToHost, st));
        GS_CUDA(cudaStreamSynchronize(st));
        for (int g = 0; g < groups; g++)
            for (int c = 0; c < n_cand; c++) {
                const size_t s = (size_t)g * n_cand + c, o = (size_t)c * groups + g;
                if (en->n_iter) en->n_iter[o] = ni[s];
                if (en->dual_gap) en->dual_gap[o] = gp[s];
                it = std::max(it, ni[s]);
            }
    }
    cudaEventRecord(ev[4], st);
    GS_CUDA(cudaStreamSynchronize(st));
    cudaEventElapsedTime(&tmr->gram, ev[0], ev[1]);
    cudaEventElapsedTime(&tmr->solve, ev[1], ev[2]);
    cudaEventElapsedTime(&tmr->score, ev[2], ev[3]);
    cudaEventElapsedTime(&tmr->total, ev[0], ev[4]);
    gs_profile &pf = h->prof;
    const float keep_h2d = pf.ms_h2d; const int64_t keep_b = pf.h2d_bytes, keep_d2h = pf.d2h_bytes;
    memset(&pf, 0, sizeof pf);
    pf.ms_h2d = keep_h2d; pf.h2d_bytes = keep_b; pf.d2h_bytes = keep_d2h;
    pf.ms_total = tmr->total; pf.ms_gram = tmr->gram; pf.ms_solve = tmr->solve; pf.ms_score = tmr->score;
    pf.launches = launches;
    pf.smo_iterations = it;                                        // CG iterations
    { double rows = 0; for (int c : cnt) rows += c; pf.gram_flops = 2.0 * rows * D * D; pf.gram_bytes = rows * D * 4 + (double)nq * D * D * 4; }
    pf.solve_bytes = 0;
    pf.ms_tensor = h->tt.collect(); pf.tensor_flops = h->tt.flops;
    return GS_OK;
}

}  // namespace

extern "C" {

int gs_ridge(gs_handle *h, int32_t n_cand, const double *alpha, int32_t fit_intercept, uint32_t flags, double *test_scores,
             double *train_scores, float *fit_ms, float *score_ms)
{
    if (h && !test_scores) { gs_set_error(h, "gs_ridge: test_scores is NULL"); return GS_ERR_ARG; }
    RidgeTimers t;
    const int st = ridge_run(h, n_cand, alpha, fit_intercept, false, test_scores, (flags & GS_RETURN_TRAIN) ? train_scores : nullptr,
                             nullptr, &t);
    if (st) return st;
    const int nt = n_cand * h->n_splits;
    for (int i = 0; i < nt; i++) {
        if (fit_ms) fit_ms[i] = (t.gram + t.solve) / (float)nt;
        if (score_ms) score_ms[i] = t.score / (float)nt;
    }
    return GS_OK;
}

int gs_ridge_refit(gs_handle *h, double alpha, int32_t fit_intercept, double *coef_out)
{
    if (h && !coef_out) { gs_set_error(h, "gs_ridge_refit: coef_out is NULL"); return GS_ERR_ARG; }
    RidgeTimers t;
    return ridge_run(h, 1, &alpha, fit_intercept, true, nullptr, nullptr, coef_out, &t);
}

int gs_enet(gs_handle *h, int32_t n_cand, const double *alpha, const double *l1_ratio, int32_t fit_intercept, double tol,
            int32_t max_iter, uint32_t flags, double *test_scores, double *train_scores, int32_t *n_iter, float *fit_ms, float *score_ms)
{
    if (h && !test_scores) { gs_set_error(h, "gs_enet: test_scores is NULL"); return GS_ERR_ARG; }
    RidgeTimers t;
    EnetSpec en{l1_ratio, tol, max_iter, n_iter, nullptr};
    const int st = ridge_run(h, n_cand, alpha, fit_intercept, false, test_scores, (flags & GS_RETURN_TRAIN) ? train_scores : nullptr,
                             nullptr, &t, &en);
    if (st) return st;
    const int nt = n_cand * h->n_splits;
    for (int i = 0; i < nt; i++) {
        if (fit_ms) fit_ms[i] = (t.gram + t.solve) / (float)nt;
        if (score_ms) score_ms[i] = t.score / (float)nt;
    }
    return GS_OK;
}

int gs_enet_refit(gs_handle *h, double alpha, double l1_ratio, int32_t fit_intercept, double tol, int32_t max_iter, double *coef_out,
                  int32_t *n_iter, double *dual_gap)
{
    if (h && !coef_out) { gs_set_error(h, "gs_enet_refit: coef_out is NULL"); return GS_ERR_ARG; }
    RidgeTimers t;
    EnetSpec en{&l1_ratio, tol, max_iter, n_iter, dual_gap};
    return ridge_run(h, 1, &alpha, fit_intercept, true, nullptr, nullptr, coef_out, &t, &en);
}

// ---- test hook: one tensor-core GEMM with host buffers ----
int gs_debug_gemm_nt(gs_handle *h, const float *A, int32_t M, const float *B, int32_t N, int32_t K, float *C)
{
    if (!h || !A || !B || !C || M <= 0 || N <= 0 || K <= 0) return GS_ERR_ARG;
    GS_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const int Kp = (K + 31) & ~31;                                   // zero-padded contraction length
    DevBuf a, ah, al, b, bh, bl, c, bt;
    GS_CUDA(a.reserve((size_t)M * Kp * 4)); GS_CUDA(ah.reserve((size_t)M * Kp * 4)); GS_CUDA(al.reserve((size_t)M * Kp * 4));
    GS_CUDA(b.reserve((size_t)N * Kp * 4)); GS_CUDA(bh.reserve((size_t)N * Kp * 4)); GS_CUDA(bl.reserve((size_t)N * Kp * 4));
    GS_CUDA(c.reserve((size_t)M * N * 4)); GS_CUDA(bt.reserve(sizeof(TcBatch)));
    GS_CUDA(cudaMemsetAsync(a.p, 0, (size_t)M * Kp * 4, st));
    GS_CUDA(cudaMemsetAsync(b.p, 0, (size_t)N * Kp * 4, st));
    GS_CUDA(cudaMemcpy2DAsync(a.p, (size_t)Kp * 4, A, (size_t)K * 4, (size_t)K * 4, M, cudaMemcpyHostToDevice, st));
    GS_CUDA(cudaMemcpy2DAsync(b.p, (size_t)Kp * 4, B, (size_t)K * 4, (size_t)K * 4, N, cudaMemcpyHostToDevice, st));
    GS_CUDA(launch_split_tf32(a.as<float>(), ah.as<float>(), al.as<float>(), (size_t)M * Kp, st));
    GS_CUDA(launch_split_tf32(b.as<float>(), bh.as<float>(), bl.as<float>(), (size_t)N * Kp, st));
    TcMap mah, mal, mbh, mbl;
    GS_CUDA(tc_make_map(&mah, ah.as<float>(), M, Kp, Kp)); GS_CUDA(tc_make_map(&mal, al.as<float>(), M, Kp, Kp));
    GS_CUDA(tc_make_map(&mbh, bh.as<float>(), N, Kp, Kp)); GS_CUDA(tc_make_map(&mbl, bl.as<float>(), N, Kp, Kp));
    TcBatch hb{0, 0, 0, Kp, c.as<float>(), (int64_t)N};
    GS_CUDA(cudaMemcpyAsync(bt.p, &hb, sizeof hb, cudaMemcpyHostToDevice, st));
    GS_CUDA(launch_gemm_nt_tf32x3(mah, mal, mbh, mbl, bt.as<TcBatch>(), 1, M, N, 1.0f, false, st, A == B && M == N));   // same matrix: Gram mode
    GS_CUDA(cudaMemcpyAsync(C, c.p, (size_t)M * N * 4, cudaMemcpyDeviceToHost, st));
    GS_CUDA(cudaStreamSynchronize(st));
    a.release(); ah.release(); al.release(); b.release(); bh.release(); bl.release(); c.release(); bt.release();
    return GS_OK;
}

}  // extern "C"
