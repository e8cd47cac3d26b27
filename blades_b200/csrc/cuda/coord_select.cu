// Dispatcher + large-N fallback of the coordinate-select kernels; the register-network kernels themselves live in
// coord_select_impl.cuh and are instantiated by coord_select_p*.cu (one group of padded sizes per translation unit).
#include "coord_select_impl.cuh"

// ---------------------------------------------------------------------------------------------
// Large-N fallback (128 < N <= 512): a block sorts a [NP x 32-coordinate] tile in shared memory
// with a bitonic network (one __syncthreads per stage).  Virtual rows are materialised into the
// tile (value computed per coordinate first).
struct SelectLargeParams {
    const float* rows[BL_MAX_ROWS];
    int n_real, n_stat, n_virtual, virt_kind;
    float virt_param;
    int mode, trim_b;
    long long c0, c1;
    BlEpilogue ep;
    const float* virt_param_ptr;   // non-null: the virtual row's parameter is read from device memory
};

template <int NP>
__global__ void __launch_bounds__(256)
coord_select_large_kernel(const __grid_constant__ SelectLargeParams p) {
    extern __shared__ float tile[];                 // [NP][33]
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const long long c = p.c0 + (long long)blockIdx.x * 32 + lane;
    const bool live = c < p.c1;
    const int n = p.n_real, f = p.n_virtual, N = n + f;
    for (int i = wid; i < NP; i += nw) {
        float x = INFINITY;
        if (i < n && live) x = bl_sanitize(bl_ldg_stream(p.rows[i] + c));
        tile[i * 33 + lane] = x;
    }
    __syncthreads();
    if (f > 0) {
        // per-coordinate statistics by warp 0 (n_stat <= 512 values, sequential per lane)
        if (wid == 0) {
            float s = 0.f;
            for (int i = 0; i < p.n_stat; ++i) s += tile[i * 33 + lane];
            const float mu = s / (float)p.n_stat;
            const float param = bl_virt_param(p);
            float m;
            if (p.virt_kind == 1) {
                float q = 0.f;
                for (int i = 0; i < p.n_stat; ++i) { float d = tile[i * 33 + lane] - mu; q += d * d; }
                m = mu - param * sqrtf(q / (float)(p.n_stat - 1));
            } else if (p.virt_kind == 3) {
                m = mu - param * bl_sign(mu);
            } else m = -param * mu;
            for (int i = n; i < N; ++i) tile[i * 33 + lane] = live ? m : INFINITY;
        }
        __syncthreads();
    }
    for (int k = 2; k <= NP; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = wid; t < NP / 2; t += nw) {
                const int i = 2 * t - (t & (j - 1));      // index with bit j clear
                const int ixj = i + j;
                const bool up = ((i & k) == 0);
                float a = tile[i * 33 + lane], b = tile[ixj * 33 + lane];
                const float lo = fminf(a, b), hi = fmaxf(a, b);
                tile[i * 33 + lane] = up ? lo : hi;
                tile[ixj * 33 + lane] = up ? hi : lo;
            }
            __syncthreads();
        }
    if (wid == 0 && live) {
        float agg;
        if (p.mode == 0) {
            float s = 0.f;
            for (int i = p.trim_b; i < N - p.trim_b; ++i) s += tile[i * 33 + lane];
            agg = s / (float)(N - 2 * p.trim_b);
        } else {
            agg = 0.5f * (tile[((N - 1) >> 1) * 33 + lane] + tile[(N >> 1) * 33 + lane]);
        }
        bl_epilogue_store(p.ep, c, agg);
    }
}

// Which kernel bl_coord_select would launch for these parameters (no CUDA call: usable without a GPU by the tests):
// 0 = none (n_real outside 1..128: the large-N kernel is a different entry point), 1 = full sorting network,
// 2 = partition-only trimmed mean.
extern "C" int bl_coord_select_choice(const SelectParams* p) {
    if (p->n_real < 1 || p->n_real > 128) return 0;
    return partition_applies(*p, (p->n_real + 7) / 8 * 8) ? 2 : 1;
}

#define DECL(K) extern "C" int bl_select_launch_k##K(const SelectParams* p, void* stream);
DECL(1) DECL(2) DECL(3) DECL(4) DECL(5) DECL(6) DECL(7) DECL(8)
DECL(9) DECL(10) DECL(11) DECL(12) DECL(13) DECL(14) DECL(15) DECL(16)
#undef DECL

extern "C" int bl_coord_select(const SelectParams* p, void* stream) {
    const int n = p->n_real;
    if (n < 1 || n > 128) return -1;
    switch ((n + 7) / 8) {
#define CASE(K) case K: return bl_select_launch_k##K(p, stream);
        CASE(1) CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8)
        CASE(9) CASE(10) CASE(11) CASE(12) CASE(13) CASE(14) CASE(15) CASE(16)
#undef CASE
    }
    return -1;
}

extern "C" int bl_coord_select_large(const SelectLargeParams* p, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const int N = p->n_real + p->n_virtual;
    if (N < 1 || N > BL_MAX_ROWS) return -1;
    const long long cols = p->c1 - p->c0;
    if (cols <= 0) return 0;
    const unsigned grid = (unsigned)((cols + 31) / 32);
    int np = 64;
    while (np < N) np <<= 1;
    const size_t smem = (size_t)np * 33 * sizeof(float);
    cudaError_t e;
#define LAUNCH(NPV)                                                                              \
    e = cudaFuncSetAttribute(coord_select_large_kernel<NPV>,                                       \
                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);              \
    if (e != cudaSuccess) return (int)e;                                                           \
    coord_select_large_kernel<NPV><<<grid, 256, smem, st>>>(*p);
    if (np == 64) { LAUNCH(64) } else if (np == 128) { LAUNCH(128) }
    else if (np == 256) { LAUNCH(256) } else { LAUNCH(512) }
#undef LAUNCH
    return (int)cudaGetLastError();
}

extern "C" int bl_sizeof_select_params() { return (int)sizeof(SelectParams); }
extern "C" int bl_sizeof_select_large_params() { return (int)sizeof(SelectLargeParams); }
