// Gram-domain solvers ON THE DEVICE -- K6 of SURVEY 2.7 without the host round trip.
//
// Krum / Multi-Krum scoring (reference krum.py:73-125), Weiszfeld iterations of the geometric median (geomed.py:62-82)
// and the centered-clipping iterations (centeredclipping.py:30-44) are all functions of the N x N Gram matrix that the
// tcgen05 pass leaves in device memory.  The reference runs them on the driver CPU over the gathered [N, d] updates;
// round 1 of this repo copied G to the host (D2H sync + numpy/C++ per round, which also kept these rounds out of CUDA
// graphs).  Here each solver is one small fp64 kernel that turns G into the weight vector w (fp32, device memory) that
// row_combine reads directly: the aggregation path Gram -> (in-switch reduce) -> solve -> combine has no host sync.
//
// The Min-Max / Min-Sum scale search (attackers/_agr.py::gram_scale is its host twin) runs here as well: it leaves the
// scale and the parameter of the malicious virtual row in device memory, where the select and attack-row kernels read it.
//
// The arithmetic mirrors csrc/host/selectors.cpp statement for statement (same clamps, same stopping rule, stable
// tie-breaking by index), so both produce the same weights up to fp64 summation order.
#include "common.cuh"

namespace {

constexpr int kSolveThreads = 512;                 // >= BL_MAX_ROWS: one thread per row
static_assert(kSolveThreads >= BL_MAX_ROWS, "one thread per Gram row");

struct GramView {
    const float* G;       // padded Gram accumulators [*, ld]
    const int* idx;       // logical row -> padded row
    int ld;
    __device__ __forceinline__ float at(int i, int j) const {         // 0.5 * (G + G^T), in fp32 like the host path
        const int a = idx[i], b = idx[j];
        return 0.5f * (G[(long long)a * ld + b] + G[(long long)b * ld + a]);
    }
};

// deterministic block-wide sum (fixed tree), result broadcast to every thread
__device__ double block_sum(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[wid] = v;
    __syncthreads();
    if (wid == 0) {
        double t = lane < (int)(blockDim.x >> 5) ? red[lane] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_down_sync(0xffffffffu, t, o);
        if (lane == 0) red[0] = t;
    }
    __syncthreads();
    return red[0];
}

// block-wide maximum, result broadcast to every thread
__device__ double block_max(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_down_sync(0xffffffffu, v, o));
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[wid] = v;
    __syncthreads();
    if (wid == 0) {
        double t = lane < (int)(blockDim.x >> 5) ? red[lane] : -INFINITY;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t = fmax(t, __shfl_down_sync(0xffffffffu, t, o));
        if (lane == 0) red[0] = t;
    }
    __syncthreads();
    return red[0];
}

}  // namespace

// ------------------------------------------------------------------------------------------------- Krum / Multi-Krum
struct KrumParams {
    const float* G; const int* idx; int ld;
    int n;                 // rows that take part (the first n logical rows)
    int n_out;             // length of w (rows >= n get weight 0)
    int f, m;
    int squared_twice;     // reference quirk Q3: the squared distance is squared again
    float value;           // weight of a selected row (1 = sum of the selected rows, 1/m = mean)
    double* scores;        // [n] scratch
    unsigned* counter;     // zero-initialised; left at zero
    float* w;              // [n_out] out
};

__global__ void __launch_bounds__(kSolveThreads)
gram_krum_kernel(const __grid_constant__ KrumParams p) {
    __shared__ double d[BL_MAX_ROWS];
    __shared__ double red[32];
    __shared__ bool last;
    const GramView g{p.G, p.idx, p.ld};
    const int i = blockIdx.x, j = threadIdx.x, n = p.n;
    const int k = max(0, min(n - p.f - 2, n - 1));
    double mine = INFINITY;
    if (j < n && j != i) {
        double v = fmax((double)g.at(i, i) + (double)g.at(j, j) - 2.0 * (double)g.at(i, j), 0.0);
        mine = p.squared_twice ? v * v : v;
    }
    if (j < BL_MAX_ROWS) d[j] = mine;
    __syncthreads();
    double contrib = 0.0;
    if (j < n && j != i) {
        int rank = 0;
        for (int l = 0; l < n; ++l) {
            const double o = d[l];
            rank += (o < mine || (o == mine && l < j)) ? 1 : 0;        // stable: ties by index (self is +inf, last)
        }
        if (rank < k) contrib = mine;
    }
    const double s = block_sum(contrib, red);
    if (threadIdx.x == 0) {
        p.scores[i] = s;
        __threadfence();
        last = (atomicAdd(p.counter, 1u) == (unsigned)(n - 1));
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    // the last block ranks the scores (stable argsort) and writes the weights
    if (j < BL_MAX_ROWS) d[j] = j < n ? ((volatile double*)p.scores)[j] : INFINITY;
    __syncthreads();
    if (j < p.n_out) {
        float w = 0.f;
        if (j < n) {
            const double me = d[j];
            int rank = 0;
            for (int l = 0; l < n; ++l) {
                const double o = d[l];
                rank += (o < me || (o == me && l < j)) ? 1 : 0;
            }
            if (rank < p.m) w = p.value;
        }
        p.w[j] = w;
    }
    if (threadIdx.x == 0) *p.counter = 0u;
}

extern "C" int bl_gram_krum(const KrumParams* p, void* stream) {
    if (p->n < 1 || p->n > BL_MAX_ROWS || p->n_out < p->n || p->n_out > BL_MAX_ROWS) return -1;
    gram_krum_kernel<<<p->n, kSolveThreads, 0, (cudaStream_t)stream>>>(*p);
    return (int)cudaGetLastError();
}
extern "C" int bl_sizeof_krum_params() { return (int)sizeof(KrumParams); }

// ------------------------------------------------------------------------------- Weiszfeld / centered clipping
struct IterParams {
    const float* G; const int* idx; int ld;
    int n;                   // Gram rows (centered clipping: n clients + 1 momentum row)
    int kind;                // 0 Weiszfeld, 1 centered clipping, 2 AutoGM (Weiszfeld inside a water-filling loop)
    int maxiter;             // Weiszfeld: max iterations; centered clipping: n_iter
    int compounding;         // Weiszfeld quirk Q5: new weights derive from the previous weights
    double eps, ftol, tau;
    const float* alphas;     // Weiszfeld point weights (nullptr: uniform)
    float* gs;               // [n*n] scratch for the symmetrised Gram when it does not fit in shared memory
    int use_smem;            // launcher: n*n floats fit in dynamic shared memory
    float* w;                // [n] out (centered clipping: coefficients over [u_0..u_{n-2}, m_prev])
    int* iters;              // out: Weiszfeld iterations taken
    double lamb;             // AutoGM regulariser
    int sort_by_index;       // AutoGM quirk Q6: the water-filling visits the clients in index order
    int pad_;
};

// dist_j = || sum_i w_i u_i - u_j ||  from the Gram matrix:  sqrt(max(w^T G w - 2 (G w)_j + G_jj, 0))
__device__ double dist_to_combo(const float* gs, int n, const double* w, int j, double* red) {
    double gw = 0.0;
    if (j < n)
        for (int i = 0; i < n; ++i) gw = fma((double)gs[(long long)i * n + j], w[i], gw);
    const double wgw = block_sum(j < n ? w[j] * gw : 0.0, red);
    if (j >= n) return 0.0;
    return sqrt(fmax(wgw - 2.0 * gw + (double)gs[(long long)j * n + j], 0.0));
}

// Weiszfeld iterations for point weights `alpha` (one per thread); leaves the weights in w[], returns this thread's
// distance to the final iterate and the iteration count.  Mirrors selectors.cpp::weiszfeld statement for statement.
__device__ int weiszfeld_run(const float* gs, int n, int j, double alpha, const IterParams& p, double* w, double* red,
                             double& dist_out) {
    double run = alpha;
    __syncthreads();
    if (j <= BL_MAX_ROWS) w[j] = j < n ? 1.0 / n : 0.0;                 // start at the plain mean (geomed.py:66)
    __syncthreads();
    double dist = dist_to_combo(gs, n, w, j, red);
    double obj = block_sum(j < n ? run * dist : 0.0, red);
    int it = 0;
    for (it = 1; it <= p.maxiter; ++it) {
        const double prev = obj;
        const double base = p.compounding ? run : alpha;
        double nw = j < n ? fmax(p.eps, base / fmax(p.eps, dist)) : 0.0;
        const double sum = block_sum(nw, red);
        nw /= sum;
        run = nw;
        __syncthreads();
        if (j < n) w[j] = nw;
        __syncthreads();
        dist = dist_to_combo(gs, n, w, j, red);
        obj = block_sum(j < n ? run * dist : 0.0, red);
        if (fabs(prev - obj) < p.ftol * obj) break;                      // uniform: obj is a broadcast value
    }
    dist_out = dist;
    return min(it, p.maxiter);
}

__global__ void __launch_bounds__(kSolveThreads)
gram_iter_kernel(const __grid_constant__ IterParams p) {
    extern __shared__ float gsm[];
    __shared__ double w[BL_MAX_ROWS + 1];
    __shared__ double red[32];
    const GramView g{p.G, p.idx, p.ld};
    const int n = p.n, j = threadIdx.x;
    float* gs = p.use_smem ? gsm : p.gs;
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) gs[e] = g.at(e / n, e % n);
    __syncthreads();

    if (p.kind == 0) {
        const double alpha = j < n ? (p.alphas ? (double)p.alphas[j] : 1.0 / n) : 0.0;
        double dist;
        const int it = weiszfeld_run(gs, n, j, alpha, p, w, red, dist);
        if (j < n) p.w[j] = (float)w[j];
        if (j == 0 && p.iters) *p.iters = it;
    } else if (p.kind == 2) {
        // AutoGM (reference autogm.py:36-65, host twin selectors.cpp::bl_autogm): alternate a weighted geometric median
        // with the water-filling update alpha = max(eta - dist, 0) / lambda; the serial prefix scan of the water
        // filling (n <= 512 steps) runs on thread 0 over shared memory
        __shared__ double s_dist[BL_MAX_ROWS];
        __shared__ int s_order[BL_MAX_ROWS];
        __shared__ double s_eta;
        double alpha = j < n ? 1.0 / n : 0.0, dist;
        weiszfeld_run(gs, n, j, alpha, p, w, red, dist);
        double glob = block_sum(j < n ? alpha * dist : 0.0, red) + p.lamb * block_sum(alpha * alpha, red) / 2.0;
        for (int iter = 0; iter < p.maxiter; ++iter) {
            const double prev = glob;
            __syncthreads();
            if (j < n) s_dist[j] = dist;
            __syncthreads();
            if (j < n) {
                int rank = j;
                if (!p.sort_by_index) {                                    // stable argsort of the distances
                    rank = 0;
                    for (int l = 0; l < n; ++l) rank += (s_dist[l] < dist || (s_dist[l] == dist && l < j)) ? 1 : 0;
                }
                s_order[rank] = j;
            }
            __syncthreads();
            if (j == 0) {
                double eta_opt = 1e16, csum = 0.0;
                for (int q = 0; q < n; ++q) {
                    const double dq = s_dist[s_order[q]];
                    csum += dq;
                    const double eta = (csum + p.lamb) / (q + 1);
                    if (eta - dq < 0) break;
                    eta_opt = eta;
                }
                s_eta = eta_opt;
            }
            __syncthreads();
            alpha = j < n ? fmax(s_eta - dist, 0.0) / p.lamb : 0.0;
            weiszfeld_run(gs, n, j, alpha, p, w, red, dist);
            glob = block_sum(j < n ? alpha * dist : 0.0, red) + p.lamb * block_sum(alpha * alpha, red) / 2.0;
            if (fabs(prev - glob) < p.ftol * glob) break;
        }
        if (j < n) p.w[j] = (float)w[j];
    } else {
        const int nc = n - 1;                                            // clients; row nc is the previous momentum
        if (j <= BL_MAX_ROWS) w[j] = (j == nc) ? 1.0 : 0.0;
        __syncthreads();
        for (int it = 0; it < p.maxiter; ++it) {
            const double dist = dist_to_combo(gs, n, w, j, red);
            const double scale = j < nc ? (dist > 0.0 ? fmin(1.0, p.tau / dist) : 1.0) : 0.0;
            const double ssum = block_sum(scale, red);
            double c = j < n ? w[j] * (1.0 - ssum / nc) : 0.0;
            if (j < nc) c += scale / nc;
            __syncthreads();
            if (j < n) w[j] = c;
            __syncthreads();
        }
        if (j < n) p.w[j] = (float)w[j];
    }
}

// ------------------------------------------------------------------------------------------------- FLTrust
// w_i = relu(cos(u_t, u_i)) * ||u_t|| / ||u_i|| / sum_j relu(cos(u_t, u_j)),  w_t = 0   (reference fltrust.py:25-37,
// host twin aggregators/_gramops.py::fltrust_weights; torch CosineSimilarity eps semantics)
struct TrustParams {
    const float* G; const int* idx; int ld;
    int n, trusted;
    double eps;
    float* w;
};

__global__ void __launch_bounds__(kSolveThreads)
gram_fltrust_kernel(const __grid_constant__ TrustParams p) {
    __shared__ double red[32];
    const GramView g{p.G, p.idx, p.ld};
    const int j = threadIdx.x, n = p.n, t = p.trusted;
    double ts = 0.0, nrm = 1.0;
    const double nrm_t = sqrt(fmax((double)g.at(t, t), 0.0));
    if (j < n) {
        nrm = sqrt(fmax((double)g.at(j, j), 0.0));
        const double c = (double)g.at(t, j) / fmax(nrm_t * nrm, p.eps);
        ts = (j == t) ? 0.0 : fmax(c, 0.0);
    }
    const double sum = block_sum(ts, red);
    if (j < n) p.w[j] = (j == t) ? 0.f : (float)(ts * nrm_t / nrm / sum);
}

extern "C" int bl_gram_fltrust(const TrustParams* p, void* stream) {
    if (p->n < 1 || p->n > BL_MAX_ROWS || p->trusted < 0 || p->trusted >= p->n) return -1;
    gram_fltrust_kernel<<<1, kSolveThreads, 0, (cudaStream_t)stream>>>(*p);
    return (int)cudaGetLastError();
}
extern "C" int bl_sizeof_trust_params() { return (int)sizeof(TrustParams); }

extern "C" int bl_gram_iter(const IterParams* p, void* stream) {
    if (p->n < 1 || p->n > BL_MAX_ROWS) return -1;
    IterParams q = *p;
    const size_t need = (size_t)p->n * p->n * sizeof(float);
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(gram_iter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return (int)e;
        attr = true;
    }
    q.use_smem = need <= 200 * 1024 ? 1 : 0;
    if (!q.use_smem && !q.gs) return -2;
    gram_iter_kernel<<<1, kSolveThreads, q.use_smem ? need : 0, (cudaStream_t)stream>>>(q);
    return (int)cudaGetLastError();
}
extern "C" int bl_sizeof_iter_params() { return (int)sizeof(IterParams); }

// ------------------------------------------------------------------------------------- Min-Max / Min-Sum scale
// Shejwalkar & Houmansadr (NDSS 2021): the malicious row is m(g) = mu - g * p over the honest rows H, with g the largest
// scale that passes   minmax: max_i ||m - u_i||^2 <= max_{i,j} ||u_i - u_j||^2
//                     minsum: sum_i ||m - u_i||^2 <= max_i sum_j ||u_i - u_j||^2.
// Everything is a function of the Gram matrix of [U; q]:
//   ||m - u_i||^2 = ||mu - u_i||^2 - 2 g (mu.p - u_i.p) + g^2 ||p||^2,   mu.u_i = mean_j G_ij,  ||mu||^2 = mean_i mu.u_i
// with p = mu / ||mu|| (unit_vec: no q row, all from G), or p = q (std / sign: q is the extra Gram row).
// One thread per honest row; the search loop is the authors' bisection, in fp64, capped at 128 iterations.
struct AgrScaleParams {
    const float* G; const int* idx; int ld;
    const int* honest;     // [n_h] logical Gram rows of the honest clients
    int n_h;
    int q_row;             // logical Gram row of q (std / sign); -1 for unit_vec
    int minsum;            // 0 Min-Max, 1 Min-Sum
    int dev_type;          // 0 unit_vec, 1 std, 2 sign
    double gamma_init, tol;
    double* gamma;         // [1] out: the scale
    float* param;          // [1] out: parameter of the virtual row's kernel form (IPM for unit_vec, ALIE for std, 3 sign)
};

constexpr int kAgrMaxIter = 128;

__global__ void __launch_bounds__(kSolveThreads)
gram_agr_scale_kernel(const __grid_constant__ AgrScaleParams p) {
    __shared__ double red[32];
    const GramView g{p.G, p.idx, p.ld};
    const int t = threadIdx.x, nh = p.n_h;
    const bool live = t < nh;
    const int i = live ? p.honest[t] : 0;
    double mui = 0.0, gii = 0.0, rmax = 0.0, rsum = 0.0;
    if (live) {
        gii = (double)g.at(i, i);
        for (int k = 0; k < nh; ++k) {
            const int j = p.honest[k];
            const double gij = (double)g.at(i, j);
            mui += gij;
            const double d = fmax(gii + (double)g.at(j, j) - 2.0 * gij, 0.0);
            rmax = fmax(rmax, d);
            rsum += d;
        }
        mui /= nh;
    }
    const double mumu = block_sum(live ? mui : 0.0, red) / nh;
    const double thr = block_max(live ? (p.minsum ? rsum : rmax) : 0.0, red);
    double up = 0.0, mup = 0.0, pp = 0.0, nrm = 0.0;
    if (p.dev_type == 0) {
        nrm = sqrt(fmax(mumu, 0.0));
        if (nrm > 0.0) { up = mui / nrm; mup = nrm; pp = 1.0; }
    } else {
        up = live ? (double)g.at(i, p.q_row) : 0.0;
        mup = block_sum(up, red) / nh;
        pp = (double)g.at(p.q_row, p.q_row);
    }
    const double d0 = fmax(mumu - 2.0 * mui + gii, 0.0), a = mup - up;
    double gam = p.gamma_init, step = p.gamma_init, ok = 0.0;
    for (int it = 0; it < kAgrMaxIter && fabs(ok - gam) > p.tol; ++it) {     // uniform: every value is a broadcast
        const double di = live ? fmax(d0 - 2.0 * gam * a + gam * gam * pp, 0.0) : 0.0;
        const double v = p.minsum ? block_sum(di, red) : block_max(di, red);
        if (v <= thr) { ok = gam; gam += step / 2.0; }
        else gam -= step / 2.0;
        step /= 2.0;
    }
    if (t == 0) {
        *p.gamma = ok;
        *p.param = p.dev_type == 0 ? (nrm > 0.0 ? (float)(ok / nrm - 1.0) : -1.f) : (float)ok;
    }
}

extern "C" int bl_gram_agr_scale(const AgrScaleParams* p, void* stream) {
    if (p->n_h < 1 || p->n_h > kSolveThreads || p->dev_type < 0 || p->dev_type > 2) return -1;
    if ((p->dev_type != 0) != (p->q_row >= 0)) return -1;
    if (!(p->gamma_init > 0.0) || !(p->tol > 0.0)) return -1;
    gram_agr_scale_kernel<<<1, kSolveThreads, 0, (cudaStream_t)stream>>>(*p);
    return (int)cudaGetLastError();
}
extern "C" int bl_sizeof_agr_scale_params() { return (int)sizeof(AgrScaleParams); }
