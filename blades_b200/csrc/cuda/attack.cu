// On-device attacker kernels (K7 of SURVEY 2.7).
//  * fill_normal: Noise attacker (reference noiseclient.py:22-25) -- Philox4x32-10 counter RNG +
//    Box-Muller written straight into the client's row of the update matrix.
//  * alie_ipm_row: standalone ALIE/IPM row (mean - z*std / -eps*mean over the honest rows) for
//    aggregators that need the malicious row materialised (Gram-based ones); coordinate-wise
//    aggregators use the fused prologue in coord_select.cu instead.  Kind 3 is the sign form mean - p*sign(mean)
//    of the Min-Max / Min-Sum attacks; p may be read from device memory (param_ptr), where the scale solver of
//    gram_solve.cu left it.
//  * agr_deviation: the deviation vector q of Min-Max / Min-Sum over the honest rows (mean, std or sign(mean)),
//    the extra row of the Gram pass whose result the scale solver searches.
#include "common.cuh"

__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t (&k)[2]) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
    const uint32_t hi0 = __umulhi(M0, c[0]), lo0 = M0 * c[0];
    const uint32_t hi1 = __umulhi(M1, c[2]), lo1 = M1 * c[2];
    c[0] = hi1 ^ c[1] ^ k[0]; c[1] = lo1; c[2] = hi0 ^ c[3] ^ k[1]; c[3] = lo0;
    k[0] += 0x9E3779B9u; k[1] += 0xBB67AE85u;
}

__global__ void fill_normal_kernel(float* __restrict__ out, long long n, float mean, float stdv,
                                   unsigned long long seed, unsigned long long offset) {
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // 4 outputs per thread
    if (q * 4 >= n) return;
    uint32_t c[4] = {(uint32_t)(q + offset), (uint32_t)((q + offset) >> 32), 0u, 0u};
    uint32_t k[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
#pragma unroll
    for (int r = 0; r < 10; ++r) philox_round(c, k);
    const float inv = 2.3283064365386963e-10f;     // 2^-32
    float u0 = ((float)c[0] + 0.5f) * inv, u1 = ((float)c[1] + 0.5f) * inv;
    float u2 = ((float)c[2] + 0.5f) * inv, u3 = ((float)c[3] + 0.5f) * inv;
    float r0 = sqrtf(-2.f * __logf(u0)), r1 = sqrtf(-2.f * __logf(u2));
    float s0, c0, s1, c1;
    __sincosf(6.283185307179586f * u1, &s0, &c0);
    __sincosf(6.283185307179586f * u3, &s1, &c1);
    float z[4] = {r0 * c0, r0 * s0, r1 * c1, r1 * s1};
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (q * 4 + j < n) out[q * 4 + j] = fmaf(stdv, z[j], mean);
}

extern "C" int bl_fill_normal(float* out, long long n, float mean, float stdv,
                              unsigned long long seed, unsigned long long offset, void* stream) {
    if (n <= 0) return 0;
    const long long quads = (n + 3) / 4;
    fill_normal_kernel<<<(unsigned)((quads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        out, n, mean, stdv, seed, offset);
    return (int)cudaGetLastError();
}

struct AttackRowParams {
    const float* rows[BL_MAX_ROWS];   // honest rows
    int n_stat;
    int kind;                         // 1 ALIE, 2 IPM, 3 sign (mean - param * sign(mean))
    float param;
    long long c0, c1;
    float* out[BL_MAX_ROWS];          // destination rows (the Byzantine clients' rows, local GPU)
    int n_out;
    const float* param_ptr;           // non-null: the parameter is read from device memory instead of `param`
};

__device__ __forceinline__ float bl_signf(float x) { return (float)((x > 0.f) - (x < 0.f)); }

__global__ void __launch_bounds__(256)
attack_row_kernel(const __grid_constant__ AttackRowParams p) {
    const long long c = p.c0 + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.c1) return;
    float s = 0.f;
    for (int i = 0; i < p.n_stat; ++i) s += bl_sanitize(bl_ldg_stream(p.rows[i] + c));
    const float mu = s / (float)p.n_stat;
    const float param = p.param_ptr ? __ldg(p.param_ptr) : p.param;
    float m;
    if (p.kind == 1) {
        float q = 0.f;     // second pass hits L2 (the tile was just read)
        for (int i = 0; i < p.n_stat; ++i) { float d = bl_sanitize(__ldg(p.rows[i] + c)) - mu; q = fmaf(d, d, q); }
        m = mu - param * sqrtf(q / (float)(p.n_stat - 1));
    } else if (p.kind == 3) {
        m = mu - param * bl_signf(mu);
    } else m = -param * mu;
    for (int j = 0; j < p.n_out; ++j) p.out[j][c] = m;
}

extern "C" int bl_attack_rows(const AttackRowParams* p, void* stream) {
    const long long cols = p->c1 - p->c0;
    if (cols <= 0) return 0;
    attack_row_kernel<<<(unsigned)((cols + 255) / 256), 256, 0, (cudaStream_t)stream>>>(*p);
    return (int)cudaGetLastError();
}
extern "C" int bl_sizeof_attack_params() { return (int)sizeof(AttackRowParams); }

// q[c] for c in [c0, c1): the deviation vector of Min-Max / Min-Sum over the honest rows, with the statistics of
// attack_row_kernel (sanitised values, fp32 mean, two-pass unbiased std).  Under coordinate sharding every rank fills
// only its own range (rows of peers are read over NVLink like the select kernels do); the Gram pass reads no more.
struct DeviationParams {
    const float* rows[BL_MAX_ROWS];   // honest rows
    int n_stat;
    int dev_type;                     // 0 mean, 1 std (unbiased), 2 sign(mean)
    long long c0, c1;
    float* q;                         // indexed by coordinate
};

__global__ void __launch_bounds__(256)
agr_deviation_kernel(const __grid_constant__ DeviationParams p) {
    const long long c = p.c0 + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.c1) return;
    float s = 0.f;
    for (int i = 0; i < p.n_stat; ++i) s += bl_sanitize(bl_ldg_stream(p.rows[i] + c));
    const float mu = s / (float)p.n_stat;
    float q;
    if (p.dev_type == 1) {
        float v = 0.f;
        for (int i = 0; i < p.n_stat; ++i) { float d = bl_sanitize(__ldg(p.rows[i] + c)) - mu; v = fmaf(d, d, v); }
        q = sqrtf(v / (float)(p.n_stat - 1));
    } else if (p.dev_type == 2) {
        q = bl_signf(mu);
    } else q = mu;
    p.q[c] = q;
}

extern "C" int bl_agr_deviation(const DeviationParams* p, void* stream) {
    if (p->n_stat < 1 || p->n_stat > BL_MAX_ROWS || p->dev_type < 0 || p->dev_type > 2) return -1;
    if (p->dev_type == 1 && p->n_stat < 2) return -1;
    const long long cols = p->c1 - p->c0;
    if (cols <= 0) return 0;
    agr_deviation_kernel<<<(unsigned)((cols + 255) / 256), 256, 0, (cudaStream_t)stream>>>(*p);
    return (int)cudaGetLastError();
}
extern "C" int bl_sizeof_deviation_params() { return (int)sizeof(DeviationParams); }
