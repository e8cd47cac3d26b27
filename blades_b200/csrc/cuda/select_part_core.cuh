// Partition-only trimmed mean (per coordinate, in registers) -- the core shared by coord_select_part_kernel and by
// the host-side checker (csrc/host/select_core_check.cu compiles this very file for the CPU).
//
// The trimmed mean does not need the NP values sorted, only partitioned into bottom-b | middle | top-b.  For
// NP = 4Q real values held as two halves a[2Q], b[2Q] and trim count b = Q:
//   1. sort each half (2 x SortNet<2Q>: 610 compare-exchanges for NP = 80, vs 849 for SortNet<80>);
//   2. one bitonic split per end: the Q smallest of the union are {min(a[i], b[Q-1-i])}, the Q largest are
//      {max(a[Q+i], b[2Q-1-i])}; the 2Q losers of the two splits ARE the middle.
// A virtual value m of multiplicity f >= Q (ALIE / IPM rows, SURVEY K7) merges analytically: the lowest Q of the
// merged multiset are the bottom-set members below m plus copies of m, so every bottom-set member x >= m stays
// (contributing x) while a copy of m is trimmed instead -- and symmetrically at the top:
//   kept = sum(middle) + sum_{x in Bot} max(x - m, 0) + sum_{x in Top} min(x - m, 0) + f*m,   N - 2Q values kept
//        (= sum(middle) + sum_{x in Bot} max(x, m) + sum_{x in Top} min(x, m) + (f - 2Q)*m).
// No large-minus-large cancellation: the middle is summed directly and the corrections are differences to m.
#pragma once

#ifndef BL_CORE_FN
#define BL_CORE_FN __device__ __forceinline__
#endif

BL_CORE_FN float bl_sat01(float x) {
#ifdef __CUDA_ARCH__
    return __saturatef(x);
#else
    return fminf(fmaxf(x, 0.f), 1.f);
#endif
}

// sign(x) with sign(0) = 0
BL_CORE_FN float bl_sign(float x) { return (float)((x > 0.f) - (x < 0.f)); }

// Virtual value from the statistics of the first n_stat values in LOAD order (a[0..H) are rows 0..H-1, b[0..H) rows
// H..NP-1): kind 1 = ALIE mean - p * std_unbiased, kind 2 = IPM -p * mean, kind 3 = mean - p * sign(mean) (Min-Max /
// Min-Sum with the sign deviation; same arithmetic as coord_select_kernel).
template <int NP>
BL_CORE_FN float bl_virtual_value(const float (&a)[NP / 2], const float (&b)[NP / 2], int n_stat, int kind, float param) {
    constexpr int H = NP / 2;
    const float fstat = (float)n_stat;
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < H; ++i) s = fmaf(a[i], bl_sat01(fstat - (float)i), s);
#pragma unroll
    for (int i = 0; i < H; ++i) s = fmaf(b[i], bl_sat01(fstat - (float)(H + i)), s);
    const float mu = s / fstat;
    if (kind == 3) return mu - param * bl_sign(mu);
    if (kind != 1) return -param * mu;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < H; ++i) { const float d = (a[i] - mu) * bl_sat01(fstat - (float)i); q = fmaf(d, d, q); }
#pragma unroll
    for (int i = 0; i < H; ++i) { const float d = (b[i] - mu) * bl_sat01(fstat - (float)(H + i)); q = fmaf(d, d, q); }
    return mu - param * sqrtf(q / (fstat - 1.f));
}

// Sum of all NP values (four independent chains).  NaN / +-inf exactly when some value is non-finite (or the finite sum
// overflows): the kernel's cue for the nan_to_num slow path; the mean of the attack statistics when every row is honest.
template <int NP>
BL_CORE_FN float bl_total(const float (&a)[NP / 2], const float (&b)[NP / 2]) {
    constexpr int H = NP / 2;
    float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
#pragma unroll
    for (int i = 0; i + 1 < H; i += 2) { t0 += a[i]; t1 += a[i + 1]; t2 += b[i]; t3 += b[i + 1]; }
    if (H % 2) { t0 += a[H - 1]; t2 += b[H - 1]; }
    return (t0 + t1) + (t2 + t3);
}

// bl_virtual_value when all NP rows are honest (n_stat == NP): no rank masks, the mean comes from the total.
template <int NP>
BL_CORE_FN float bl_virtual_value_all(const float (&a)[NP / 2], const float (&b)[NP / 2], float total, int kind, float param) {
    constexpr int H = NP / 2;
    const float mu = total / (float)NP;
    if (kind == 3) return mu - param * bl_sign(mu);
    if (kind != 1) return -param * mu;
    float q0 = 0.f, q1 = 0.f;
#pragma unroll
    for (int i = 0; i < H; ++i) {
        const float da = a[i] - mu, db = b[i] - mu;
        q0 = fmaf(da, da, q0);
        q1 = fmaf(db, db, q1);
    }
    return mu - param * sqrtf((q0 + q1) / (float)(NP - 1));
}

// Trimmed mean of the NP real values (+ f copies of m), trimming Q = NP/4 from each end.  Requires f == 0 or f >= Q.
// Destroys a and b (sorted in place).
template <int NP, int MIX = 0, bool ROLL = false>
BL_CORE_FN float bl_trimmed_partition(float (&a)[NP / 2], float (&b)[NP / 2], float m, int f) {
    static_assert(NP % 8 == 0 && NP >= 8 && NP <= 128, "halves must be SortNet sizes (multiples of 4)");
    constexpr int H = NP / 2, Q = NP / 4;
    if (ROLL) {
    // ONE copy of the half-size network in the instruction stream, executed twice: ncu's top stall of the unrolled
    // form was "no_instruction" (the two inlined 305-comparator networks are ~27 KB of SASS, the whole kernel ~45 KB
    // against a 32 KB L1.5 instruction cache, and 128-thread blocks run out of phase).  The halves trade places
    // between the passes (register moves); the splits below are symmetric in (a, b), so no second exchange.
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
        SortNet<H>::template run<MIX>(a);
        if (h == 0) {
#pragma unroll
            for (int i = 0; i < H; ++i) { const float t = a[i]; a[i] = b[i]; b[i] = t; }
        }
    }
    } else {
    SortNet<H>::template run<MIX>(a);
    SortNet<H>::template run<MIX>(b);
    }
    float mid0 = 0.f, mid1 = 0.f, ext0 = 0.f, ext1 = 0.f;
    if (f > 0) {                                               // uniform branch (kernel parameter)
#pragma unroll
        for (int i = 0; i < Q; ++i) {
            const float x = a[i], y = b[Q - 1 - i];
            mid0 += fmaxf(x, y);                               // loser of the bottom split -> middle
            ext0 += fmaxf(fminf(x, y), m) - m;                 // bottom-set member above m stays (as x - m + m)
        }
#pragma unroll
        for (int i = 0; i < Q; ++i) {
            const float x = a[Q + i], y = b[H - 1 - i];
            mid1 += fminf(x, y);                               // loser of the top split -> middle
            ext1 += fminf(fmaxf(x, y), m) - m;                 // top-set member below m stays
        }
    } else {
#pragma unroll
        for (int i = 0; i < Q; ++i) mid0 += fmaxf(a[i], b[Q - 1 - i]);
#pragma unroll
        for (int i = 0; i < Q; ++i) mid1 += fminf(a[Q + i], b[H - 1 - i]);
    }
    // (hoisting the "- m" out of the sums -- sum clip + (f - 2Q) m -- saves 2Q FADDs but lengthens live ranges enough
    // to spill at several sizes; kept in the per-element form)
    const float kept = (mid0 + mid1) + (ext0 + ext1) + (float)f * (f > 0 ? m : 0.f);
    return kept / (float)(NP + f - 2 * Q);
}
