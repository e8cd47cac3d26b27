// Coordinate-wise robust selection over the client dimension -- K3/K4 (+K7 prologue, K8 epilogue)
// of SURVEY 2.7: trimmed mean (reference trimmedmean.py:38-41: two strided topk + 3 temporaries)
// and median (reference median.py:23-24: two kthvalue passes) in ONE streaming pass.
//
// One thread owns one coordinate: it loads that coordinate from every client row (rows may live
// on peer GPUs -- plain global loads on NVLink-mapped pointers, coalesced 128 B per warp per row),
// sorts the <=128 values in registers with a static pruned Batcher network, and reduces the ranks
// it needs.  ALIE / IPM attackers are *virtual rows*: their common value (mean - z*std, or
// -eps*mean, over the honest rows) is computed from the same registers and merged analytically
// with multiplicity f -- f identical malicious rows are never stored or sorted.
// The result is written to every replica and theta += lr*agg is applied in the same kernel.
#pragma once
#include "common.cuh"
#include "tc_common.cuh"
#include <cstdlib>

// Compare-exchange formulations.  The networks are bound by the ALU pipe (FMNMX issues every 2nd cycle per SM
// sub-partition; ncu: ALU 84 %, FMA 15 %).  lo = min(a, b) stays an FMNMX; hi can be taken as the second FMNMX or --
// because lo is bit-identical to one of the inputs -- as  bits(a) + bits(b) - bits(lo)  in exact 32-bit integer
// arithmetic, issued as two IMADs on the otherwise idle FMA pipe (the +-1 multipliers come from constant memory, so
// ptxas cannot fold the pair back into one ALU-pipe IADD3).  MIX picks which comparators take the IMAD form:
//   0 none, 1 all, 2 two of three, 3 one of two, 4 one of three, 5 three of four, 6 four of five (comparator index
//   from __COUNTER__).
static __constant__ int bl_ce_k[2] = {1, -1};
template <int MIX, int K>
__device__ __forceinline__ void bl_ce(float& x, float& y) {
    const float lo = fminf(x, y);
    constexpr bool imad = MIX == 1 || (MIX == 2 && K % 3 != 0) || (MIX == 3 && K % 2 == 0) || (MIX == 4 && K % 3 == 0) ||
                          (MIX == 5 && K % 4 != 0) || (MIX == 6 && K % 5 != 0);
    if constexpr (imad) {
        int t, h;
        asm("mad.lo.s32 %0, %1, %2, %3;" : "=r"(t) : "r"(__float_as_int(lo)), "r"(bl_ce_k[1]), "r"(__float_as_int(y)));
        asm("mad.lo.s32 %0, %1, %2, %3;" : "=r"(h) : "r"(__float_as_int(x)), "r"(bl_ce_k[0]), "r"(t));
        y = __int_as_float(h);
    } else {
        y = fmaxf(x, y);
    }
    x = lo;
}
#define CE(a, b) bl_ce<MIX, __COUNTER__>(v[a], v[b]);

// Rows are sanitised where they are written (wgrad / BatchNorm / bias epilogues, fused diffs, attack kernels -- the
// reference's nan_to_num in save_update, client.py:198).  The consumer only has to stay correct if a non-finite value
// shows up anyway: the running total (needed for the attack statistics; FMA pipe) is NaN / inf exactly then, and the
// warp takes the slow path that applies nan_to_num to every value.  Saves ~4 ALU-pipe instructions per value.
__device__ __forceinline__ bool bl_nonfinite(float total) { return !(fabsf(total) <= FLT_MAX); }
#include "gen/sortnet_gen.cuh"
#include "select_part_core.cuh"
#undef CE

struct SelectParams {
    const float* rows[128];   // real rows: honest first (stat rows), then other real rows
    int n_real;               // number of real rows (<= NP)
    int n_stat;               // first n_stat rows enter the attack statistics
    int n_virtual;            // multiplicity f of the virtual row
    int virt_kind;            // 0 none, 1 ALIE (mean - p*std_unbiased), 2 IPM (-p*mean), 3 sign (mean - p*sign(mean))
    float virt_param;
    int mode;                 // 0 trimmed mean, 1 median
    int trim_b;
    long long c0, c1;         // coordinate range owned by this launch
    BlEpilogue ep;
    const float* virt_param_ptr;   // non-null: p is read from device memory (Min-Max / Min-Sum scale solver)
};

// the virtual row's parameter: the launch's constant, or the value a solver left in device memory
template <class P>
__device__ __forceinline__ float bl_virt_param(const P& p) { return p.virt_param_ptr ? __ldg(p.virt_param_ptr) : p.virt_param; }

// Pipe balance (ncu: the ALU pipe -- FMNMX/ISETP/SEL, 16 lanes/clk/SMSP -- is the limiter): the sorting
// network has to live on the ALU pipe, so everything else is written as FFMA / FADD.SAT arithmetic for
// the otherwise idle FMA pipe: masks are 0/1 floats, rank tests are saturating adds.
// Block size: the straight-line network is ~30-50 KB of SASS, more than the 32 KB L1.5 instruction cache, and ncu
// showed "no_instruction" as the top stall with 128-thread blocks (20 independent warps per SM each streaming
// the code at a different position).  Large blocks keep the warps of an SM roughly in lockstep so they share
// instruction-cache lines; two resident blocks per SM still overlap one block's load phase with the other's sort.
template <int NP> struct SelectBlock { static constexpr int kMax = NP <= 80 ? 640 : (NP <= 104 ? 512 : 384); };

template <int NP, int MODE, int MIX>
__global__ void __launch_bounds__(SelectBlock<NP>::kMax)
coord_select_kernel(const __grid_constant__ SelectParams p) {
    const long long c = p.c0 + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.c1) return;
    float v[NP];
    const int n = p.n_real;
    // Issue ALL row loads back to back before the first use (rows[i >= n] alias row 0 on the host
    // side, so no load is predicated): one DRAM/NVLink round trip per thread instead of NP.
    // 32-bit element offset from the (uniform) row base: no per-load 64-bit address arithmetic on the ALU pipe.
    const unsigned cu = (unsigned)c;
#pragma unroll
    for (int i = 0; i < NP; ++i) v[i] = __ldcs(p.rows[i] + cu);      // ld.global.cs: streaming, evict-first
    {
        float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
#pragma unroll
        for (int i = 0; i + 3 < NP; i += 4) { t0 += v[i]; t1 += v[i + 1]; t2 += v[i + 2]; t3 += v[i + 3]; }
        if (bl_nonfinite((t0 + t1) + (t2 + t3))) {
#pragma unroll
            for (int i = 0; i < NP; ++i) v[i] = bl_sanitize(v[i]);
        }
    }

    // ---- attack prologue (K7): statistics of the honest rows (= the first n_stat slots), load order
    float m = 0.f;
    const int f = p.n_virtual;
    const float fstat = (float)p.n_stat;
    if (f > 0) {
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < NP; ++i) s = fmaf(v[i], __saturatef(fstat - (float)i), s);     // mask = [i < n_stat]
        const float mu = s / fstat;
        const float param = bl_virt_param(p);
        if (p.virt_kind == 1) {
            float q = 0.f;
#pragma unroll
            for (int i = 0; i < NP; ++i) {
                const float d = (v[i] - mu) * __saturatef(fstat - (float)i);
                q = fmaf(d, d, q);
            }
            m = mu - param * sqrtf(q / (fstat - 1.f));
        } else if (p.virt_kind == 3) {
            m = mu - param * bl_sign(mu);
        } else {
            m = -param * mu;
        }
    }
    // padding slots sort to the top: FLT_MAX (finite, so 0-weight products stay 0); n > NP - 8 by dispatch,
    // so only the last 7 slots can be padding
#pragma unroll
    for (int i = (NP >= 8 ? NP - 7 : 0); i < NP; ++i) v[i] = (i < n) ? v[i] : FLT_MAX;

    SortNet<NP>::template run<MIX>(v);

    // ---- merge the virtual value with multiplicity f: r = #real values below m
    const int N = n + f;
    float rf = 0.f;
    if (f > 0) {
#pragma unroll
        for (int i = 0; i < NP; ++i) rf += (v[i] < m) ? 1.f : 0.f;
        rf = fminf(rf, (float)n);               // padding (FLT_MAX) never counts as a real value
    }
    const float ff = (float)f;
    float agg;
    if (MODE == 0) {
        const float lo = (float)p.trim_b, hi = (float)(N - p.trim_b);   // keep merged ranks [lo, hi)
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            const float pos = fmaf(ff, __saturatef((float)(i + 1) - rf), (float)i);       // i + f*[i >= r]
            const float keep = __saturatef(pos - lo + 1.f) * __saturatef(hi - pos);      // [lo <= pos < hi]
            s = fmaf(keep, v[i], s);
        }
        if (f > 0) {
            const float a = fmaxf(rf, lo), b = fminf(rf + ff, hi);
            s = fmaf(m, fmaxf(b - a, 0.f), s);
        }
        agg = s / (hi - lo);
    } else {
        const float k0 = (float)((N - 1) >> 1), k1 = (float)(N >> 1);
        float a0 = 0.f, a1 = 0.f;
        if (f > 0) {
            a0 = m * __saturatef(k0 - rf + 1.f) * __saturatef(rf + ff - k0);
            a1 = m * __saturatef(k1 - rf + 1.f) * __saturatef(rf + ff - k1);
        }
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            const float pos = fmaf(ff, __saturatef((float)(i + 1) - rf), (float)i);
            a0 = fmaf(__saturatef(pos - k0 + 1.f) * __saturatef(k0 + 1.f - pos), v[i], a0);
            a1 = fmaf(__saturatef(pos - k1 + 1.f) * __saturatef(k1 + 1.f - pos), v[i], a1);
        }
        agg = 0.5f * (a0 + a1);
    }
    bl_epilogue_store(p.ep, c, agg);
}

// ---------------------------------------------------------------------------------------------
// Partition-only trimmed mean (select_part_core.cuh): n_real == NP == 4 * trim_b and (no virtual rows or f >= b)
// -- the "20 % attackers, Trimmedmean(nb = f)" family (N = 10k clients: 8k honest rows, b = 2k).  Two half-size
// sorts + two bitonic splits instead of one full network: ~21 % fewer FMNMX on the pipe that bounds this kernel.
// select_part_core.cuh can run the two half sorts as ONE rolled code copy (ncu's top stall of this kernel is
// "no_instruction"); with the exchange of the halves between the passes and the 128-register budget it then needs,
// that form measured slower (1.02 vs 0.95 ms at the headline shape), so it stays off.
constexpr bool kSelectRollHalves = false;

template <int NP, int MIX>
__global__ void __launch_bounds__(SelectBlock<NP>::kMax)
coord_select_part_kernel(const __grid_constant__ SelectParams p) {
    const long long c = p.c0 + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.c1) return;
    constexpr int H = NP / 2;
    float a[H], b[H];
    const unsigned cu = (unsigned)c;
#pragma unroll
    for (int i = 0; i < H; ++i) a[i] = __ldcs(p.rows[i] + cu);
#pragma unroll
    for (int i = 0; i < H; ++i) b[i] = __ldcs(p.rows[H + i] + cu);
    float total = bl_total<NP>(a, b);
    if (bl_nonfinite(total)) {
#pragma unroll
        for (int i = 0; i < H; ++i) { a[i] = bl_sanitize(a[i]); b[i] = bl_sanitize(b[i]); }
        total = bl_total<NP>(a, b);
    }
    const int f = p.n_virtual;
    float m = 0.f;
    if (f > 0) m = p.n_stat == NP ? bl_virtual_value_all<NP>(a, b, total, p.virt_kind, bl_virt_param(p))
                                  : bl_virtual_value<NP>(a, b, p.n_stat, p.virt_kind, bl_virt_param(p));
    bl_epilogue_store(p.ep, c, bl_trimmed_partition<NP, MIX, kSelectRollHalves>(a, b, m, f));
}

// ---------------------------------------------------------------------------------------------
// Partition-only trimmed mean fed by bulk copies (the TMA engine's 1-D form, cp.async.bulk): a persistent CTA walks
// tiles of 128 coordinates; warp 0 issues one 512 B bulk copy per client row (local HBM or a peer's rows over NVLink)
// into a [NP][128] shared-memory tile, completion is counted on an mbarrier, every thread then takes its coordinate's
// NP values with immediate-offset LDS.  The per-row 64-bit address arithmetic (2 ALU-pipe IADD3 per row and THREAD in
// the LDG form -- 15 % of the pipe that bounds this kernel) is done once per row and TILE by the issuing lanes, and
// the next tile's copies fly while the current one is sorted (registers hold the values, so one buffer suffices).
constexpr int kStageTile = 128;
static_assert(kStageTile == 128, "stage_issue hard-codes the tile width");

// warp 0, all lanes: bulk copies of rows lane, lane + 32, ... of tile t into the shared tile
template <int NP>
__device__ __forceinline__ void stage_issue(const SelectParams& p, float* tile, uint64_t* full, long long t, int tid) {
    const long long c = p.c0 + t * 128;
    if (tid == 0) bl::mbar_arrive_expect_tx(full, (uint32_t)(NP * 128 * sizeof(float)));
    __syncwarp();
    for (int i = tid; i < NP; i += 32) {
        asm volatile(
            "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
            :: "r"(bl::smem_u32(tile + i * 128)), "l"(p.rows[i] + c), "r"((uint32_t)(128 * sizeof(float))),
               "r"(bl::smem_u32(full)) : "memory");
    }
}

template <int NP> struct StageBlocks { static constexpr int kPerSM = NP <= 48 ? 4 : 3; };   // register budget without spills

template <int NP, int MIX>
__global__ void __launch_bounds__(kStageTile, StageBlocks<NP>::kPerSM)
coord_select_part_stage_kernel(const __grid_constant__ SelectParams p) {
    extern __shared__ __align__(128) unsigned char stage_smem[];
    float* tile = reinterpret_cast<float*>(stage_smem);                              // [NP][kStageTile]
    uint64_t* full = reinterpret_cast<uint64_t*>(stage_smem + (size_t)NP * kStageTile * sizeof(float));
    constexpr int H = NP / 2;
    const int tid = threadIdx.x;
    const long long n_tiles = (p.c1 - p.c0) / kStageTile;                            // whole tiles only (launcher)
    if (tid == 0) { bl::mbar_init(full, 1); bl::fence_barrier_init(); }
    __syncthreads();

    long long t = blockIdx.x;
    if (t < n_tiles && tid < 32) stage_issue<NP>(p, tile, full, t, tid);
    uint32_t parity = 0;
    const int f = p.n_virtual;
    for (; t < n_tiles; t += gridDim.x) {
        float a[H], b[H];
        bl::mbar_wait(full, parity);
        parity ^= 1u;
#pragma unroll
        for (int i = 0; i < H; ++i) a[i] = tile[i * kStageTile + tid];
#pragma unroll
        for (int i = 0; i < H; ++i) b[i] = tile[(H + i) * kStageTile + tid];
        __syncthreads();                                                             // everyone has its values
        const long long tn = t + gridDim.x;
        if (tn < n_tiles && tid < 32) stage_issue<NP>(p, tile, full, tn, tid);       // refill while this tile is sorted
        float total = bl_total<NP>(a, b);
        if (bl_nonfinite(total)) {
#pragma unroll
            for (int i = 0; i < H; ++i) { a[i] = bl_sanitize(a[i]); b[i] = bl_sanitize(b[i]); }
            total = bl_total<NP>(a, b);
        }
        float m = 0.f;
        if (f > 0) m = p.n_stat == NP ? bl_virtual_value_all<NP>(a, b, total, p.virt_kind, bl_virt_param(p))
                                      : bl_virtual_value<NP>(a, b, p.n_stat, p.virt_kind, bl_virt_param(p));
        bl_epilogue_store(p.ep, p.c0 + t * kStageTile + tid, bl_trimmed_partition<NP, MIX>(a, b, m, f));
    }
}

static int select_block_size(int kmax, bool partition) {
    static int forced = -1;
    if (forced < 0) {
        const char* e = getenv("BLADES_SELECT_BLOCK");
        forced = e ? atoi(e) : 0;
    }
    // measured (profiles/kernel_bench_r2.txt): the partition kernel (two half sorts) is fastest with 128-thread
    // blocks, the full networks (more straight-line code per warp) with 256
    int b = forced > 0 ? forced : (partition ? 128 : 256);
    if (b > kmax) b = kmax;
    return (b / 32) * 32;
}

static bool select_partition_enabled() {
    static const bool on = [] { const char* e = getenv("BLADES_SELECT_PARTITION"); return !(e && e[0] == '0'); }();
    return on;
}

// The partition-only kernel applies when the real rows fill the padded size exactly, the trim count is a quarter of
// them and a virtual row (if any) has multiplicity >= the trim count (select_part_core.cuh).  Its virtual value needs
// n_stat >= 2 only for the ALIE form (kind 1: the unbiased std); IPM (2) and sign (3) need the mean alone.
static bool partition_applies(const SelectParams& p, int NP) {
    return p.mode == 0 && p.n_real == NP && p.trim_b * 4 == NP && (p.n_virtual == 0 || p.n_virtual >= p.trim_b)
           && (p.n_virtual == 0 || p.n_stat >= 2 || p.virt_kind == 2 || p.virt_kind == 3) && select_partition_enabled();
}

// Compare-exchange mix (see bl_ce): BLADES_SELECT_CE = 0 plain FMNMX pairs, otherwise kSelectMix
constexpr int kSelectMix = 5;         // measured best of {0..6} on the headline shape (profiles/kernel_bench_r2.txt)
static int select_ce_mix() {
    static const int v = [] { const char* e = getenv("BLADES_SELECT_CE"); return e ? atoi(e) : kSelectMix; }();
    return v;
}
static bool select_imad_enabled() { return select_ce_mix() != 0; }

static bool select_staged_enabled() {
    // opt-in: measured SLOWER than the LDG form on B200 so far (1.23 vs 0.95 ms at the headline shape,
    // profiles/kernel_bench_r2.txt) -- kept for the ncu comparison, BLADES_SELECT_STAGED=1 enables it
    static const bool on = [] { const char* e = getenv("BLADES_SELECT_STAGED"); return e && e[0] == '1'; }();
    return on;
}

// Bulk-copy staged form: whole 128-coordinate tiles whose row segments are 16 B aligned; the launcher hands the
// remaining (< 128, or misaligned) coordinates to the LDG form.  Returns the number of coordinates it covered.
template <int NP>
static long long launch_partition_staged(const SelectParams& p, cudaStream_t st) {
    if constexpr (NP > 80) return 0;     // experimental form: instantiated up to the headline size only
    else {
    if (!select_staged_enabled() || select_ce_mix() == 0 || (p.c0 % 4) != 0) return 0;
    for (int i = 0; i < NP; ++i)
        if ((uintptr_t)p.rows[i] % 16 != 0) return 0;
    const long long n_tiles = (p.c1 - p.c0) / kStageTile;
    if (n_tiles < 1) return 0;
    const size_t smem = (size_t)NP * kStageTile * sizeof(float) + 16;
    static int sms = 0;
    static bool attr = false;
    if (!attr) {
        if (cudaFuncSetAttribute(coord_select_part_stage_kernel<NP, kSelectMix>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)smem) != cudaSuccess) return 0;
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        attr = true;
    }
    int per_sm = (int)((227 * 1024) / (smem + 1024));
    if (per_sm > StageBlocks<NP>::kPerSM) per_sm = StageBlocks<NP>::kPerSM;
    if (per_sm < 1) return 0;
    long long grid = (long long)sms * per_sm;
    if (grid > n_tiles) grid = n_tiles;
    SelectParams q = p;
    q.c1 = p.c0 + n_tiles * kStageTile;
    coord_select_part_stage_kernel<NP, kSelectMix><<<(unsigned)grid, kStageTile, smem, st>>>(q);
    return n_tiles * kStageTile;
    }
}

template <int NP>
static bool launch_partition(const SelectParams& p, unsigned grid, int block, cudaStream_t st) {
    if constexpr (NP % 8 == 0) {
        if (partition_applies(p, NP)) {
            const int mix = select_ce_mix();
            if constexpr (NP == 80) {          // headline shape: the other mixes stay selectable for A/B runs
                if (mix == 3) { coord_select_part_kernel<NP, 3><<<grid, block, 0, st>>>(p); return true; }
                if (mix == 4) { coord_select_part_kernel<NP, 4><<<grid, block, 0, st>>>(p); return true; }
                if (mix == 2) { coord_select_part_kernel<NP, 2><<<grid, block, 0, st>>>(p); return true; }
                if (mix == 6) { coord_select_part_kernel<NP, 6><<<grid, block, 0, st>>>(p); return true; }
                if (mix == 1) { coord_select_part_kernel<NP, 1><<<grid, block, 0, st>>>(p); return true; }
            }
            if (mix != 0) coord_select_part_kernel<NP, kSelectMix><<<grid, block, 0, st>>>(p);
            else coord_select_part_kernel<NP, 0><<<grid, block, 0, st>>>(p);
            return true;
        }
    }
    return false;
}

template <int NP>
static cudaError_t launch_small(const SelectParams& p, cudaStream_t st) {
    const long long cols = p.c1 - p.c0;
    if (cols <= 0) return cudaSuccess;
    if (p.c1 > 0xFFFFFFFFLL) return cudaErrorInvalidValue;      // 32-bit element offsets
    if constexpr (NP % 8 == 0) {
        if (partition_applies(p, NP)) {
            SelectParams q = p;
            q.c0 += launch_partition_staged<NP>(p, st);            // whole aligned tiles through the bulk-copy form
            if (q.c0 >= q.c1) return cudaGetLastError();
            const int pblock = select_block_size(SelectBlock<NP>::kMax, true);
            launch_partition<NP>(q, (unsigned)((q.c1 - q.c0 + pblock - 1) / pblock), pblock, st);
            return cudaGetLastError();
        }
    }
    const int block = select_block_size(SelectBlock<NP>::kMax, false);
    const unsigned grid = (unsigned)((cols + block - 1) / block);
    if (select_imad_enabled()) {
        if (p.mode == 0) coord_select_kernel<NP, 0, kSelectMix><<<grid, block, 0, st>>>(p);
        else coord_select_kernel<NP, 1, kSelectMix><<<grid, block, 0, st>>>(p);
    } else {
        if (p.mode == 0) coord_select_kernel<NP, 0, 0><<<grid, block, 0, st>>>(p);
        else coord_select_kernel<NP, 1, 0><<<grid, block, 0, st>>>(p);
    }
    return cudaGetLastError();
}


// One translation unit per group of padded sizes (coord_select_p*.cu) so the straight-line networks compile in parallel;
// each defines the launchers of its sizes, the dispatcher (coord_select.cu) switches over them.
#define BL_SELECT_LAUNCHER(K) \
    extern "C" int bl_select_launch_k##K(const SelectParams* p, void* stream) { \
        return (int)launch_small<8 * K>(*p, (cudaStream_t)stream); }
