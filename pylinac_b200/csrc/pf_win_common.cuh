// Device pieces shared by the PicketFence window kernels (pf_windows.cu, pf_windows2.cu): packed u16x2 sorting-network medians and
// the serial integer FWXM analysis of one window's median profile.
#pragma once
#include <utility>

#include "pf_common.cuh"

namespace epid {

// a * b + c with a 64-bit accumulator in ONE instruction (IMAD.WIDE.U32); the compiler emits IMAD + IADD3 + IADD3.X for the C form
__device__ __forceinline__ unsigned long long mad_wide_u32(uint32_t a, uint32_t b, unsigned long long c) {
    unsigned long long d;
    asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(d) : "r"(a), "r"(b), "l"(c));
    return d;
}

// Batcher merge-exchange network (valid for any N) as a compile-time comparator list.  The list is applied through template
// arguments, so every array index is a constant and the sorted values stay in registers (written as nested loops the compiler left
// the array in local memory: LDL / STL around every comparator).
struct NetList {
    int n;
    short a[640], b[640];
};
constexpr NetList batcher_net(int N) {
    NetList L{};
    for (int p = 1; p < N; p <<= 1)
        for (int k = p; k >= 1; k >>= 1)
            for (int j = k % p; j <= N - 1 - k; j += 2 * k)
                for (int i = 0; i < k; i++)
                    if (i <= N - j - k - 1 && (i + j) / (2 * p) == (i + j + k) / (2 * p)) {
                        L.a[L.n] = (short)(i + j);
                        L.b[L.n] = (short)(i + j + k);
                        L.n++;
                    }
    return L;
}
template <int N>
struct BatcherNet {
    static constexpr NetList L = batcher_net(N);
};

template <int A, int B, int N>
__device__ __forceinline__ void cmpswap_u16x2(uint32_t (&r)[N]) {
    const uint32_t a = r[A], b = r[B];
    r[A] = __vminu2(a, b);
    r[B] = __vmaxu2(a, b);
}
template <int N, int... I>
__device__ __forceinline__ void apply_net_u16x2(uint32_t (&r)[N], std::integer_sequence<int, I...>) {
    (cmpswap_u16x2<BatcherNet<N>::L.a[I], BatcherNet<N>::L.b[I], N>(r), ...);
}
// ascending in both 16-bit halves independently
template <int N>
__device__ __forceinline__ void sort_net_u16x2(uint32_t (&r)[N]) {
    apply_net_u16x2<N>(r, std::make_integer_sequence<int, BatcherNet<N>::L.n>{});
}

template <int A, int B, int N>
__device__ __forceinline__ void cmpswap_u64(unsigned long long (&r)[N]) {
    const unsigned long long a = r[A], b = r[B];
    r[A] = a < b ? a : b;
    r[B] = a < b ? b : a;
}
template <int N, int... I>
__device__ __forceinline__ void apply_net_u64(unsigned long long (&r)[N], std::integer_sequence<int, I...>) {
    (cmpswap_u64<BatcherNet<N>::L.a[I], BatcherNet<N>::L.b[I], N>(r), ...);
}
template <int N>
__device__ __forceinline__ void sort_net_u64(unsigned long long (&r)[N]) {
    apply_net_u64<N>(r, std::make_integer_sequence<int, BatcherNet<N>::L.n>{});
}

// 2 * median over exactly N rows of the travel-sample pair in word `t`: (va + vb) per half
template <int N>
__device__ __forceinline__ void pair_median_exact(const uint16_t* __restrict__ px, int S, int t, uint32_t& m_lo, uint32_t& m_hi) {
    uint32_t r[N];
#pragma unroll
    for (int i = 0; i < N; i++) r[i] = *reinterpret_cast<const uint32_t*>(px + i * S + 2 * t);
    sort_net_u16x2<N>(r);
    const uint32_t va = r[(N - 1) / 2], vb = r[N / 2];
    m_lo = (va & 0xffffu) + (vb & 0xffffu);
    m_hi = (va >> 16) + (vb >> 16);
}

// padded variant for row counts without an exact instantiation
template <int NRP>
__device__ __forceinline__ void pair_median_padded(const uint16_t* __restrict__ px, int S, int nr, int t, uint32_t& m_lo, uint32_t& m_hi) {
    uint32_t r[NRP];
#pragma unroll
    for (int i = 0; i < NRP; i++)
        r[i] = i < nr ? *reinterpret_cast<const uint32_t*>(px + i * S + 2 * t) : 0xffffffffu;
    sort_net_u16x2<NRP>(r);
    const int k1 = (nr - 1) / 2, k2 = nr / 2;
    uint32_t va = 0, vb = 0;
#pragma unroll
    for (int i = 0; i < NRP; i++) {
        if (i == k1) va = r[i];
        if (i == k2) vb = r[i];
    }
    m_lo = (va & 0xffffu) + (vb & 0xffffu);
    m_hi = (va >> 16) + (vb >> 16);
}

static __device__ __noinline__ uint2 pair_median_any(const uint16_t* __restrict__ px, int S, int nr, int t) {
    uint32_t m_lo = 0, m_hi = 0;
    switch (nr) {
#define EPID_MED_CASE(N) case N: pair_median_exact<N>(px, S, t, m_lo, m_hi); break;
        EPID_MED_CASE(6) EPID_MED_CASE(7) EPID_MED_CASE(8) EPID_MED_CASE(9) EPID_MED_CASE(10) EPID_MED_CASE(11)
        EPID_MED_CASE(12) EPID_MED_CASE(13) EPID_MED_CASE(14) EPID_MED_CASE(15) EPID_MED_CASE(16) EPID_MED_CASE(17)
        EPID_MED_CASE(18) EPID_MED_CASE(19) EPID_MED_CASE(20) EPID_MED_CASE(21) EPID_MED_CASE(22) EPID_MED_CASE(23)
        EPID_MED_CASE(24) EPID_MED_CASE(25) EPID_MED_CASE(26) EPID_MED_CASE(27) EPID_MED_CASE(28) EPID_MED_CASE(29)
        EPID_MED_CASE(30) EPID_MED_CASE(31) EPID_MED_CASE(32)
#undef EPID_MED_CASE
        default:
            if (nr < 6) pair_median_padded<8>(px, S, nr, t, m_lo, m_hi);
            else if (nr <= 48) pair_median_padded<48>(px, S, nr, t, m_lo, m_hi);
            else pair_median_padded<64>(px, S, nr, t, m_lo, m_hi);
    }
    return make_uint2(m_lo, m_hi);
}

// serial FWXM analysis of one window's median profile m[0..nc) (2 * median in g units), lane-private.
// Mirrors find_peaks(values, fwxm_height=0.5, max_number=1) on xs = (m - min) / (max - min) and scipy's _peak_widths.
// returns valid (1), 0 = no peak / flat (the caller raises EPID_PF_WINDOW_NO_PEAK)
template <int ST = 1>
__device__ inline int window_fwxm(const uint32_t* __restrict__ mbase, int nc, double& out_l, double& out_r) {
    auto M = [&](int j) { return mbase[j * ST]; };
    // one branch-light pass (the lanes of the warp -- one window each -- stay in lockstep): min, max and the two highest local
    // maxima (scipy _local_maxima_1d: rise, plateau, fall; midpoint of the plateau), key = height << 8 | position
    uint32_t lmin, lmax, best1 = 0, best2 = 0;
    {
        int start = -1;
        uint32_t prev = M(0);
        lmin = lmax = prev;
        for (int i = 1; i < nc; i++) {
            const uint32_t v = M(i);
            lmin = min(lmin, v);
            lmax = max(lmax, v);
            if (v < prev && start >= 0) {
                const uint32_t key = (prev << 8) | (uint32_t)((start + i - 1) >> 1);
                if (key > best1) { best2 = best1; best1 = key; }
                else if (key > best2) best2 = key;
            }
            start = v > prev ? i : (v < prev ? -1 : start);
            prev = v;
        }
    }
    if (lmax == lmin || best1 == 0) return 0;
    const double den = (double)(lmax - lmin);
    auto xs = [&](int j) { return (double)(M(j) - lmin) / den; };
    double best_prom = -1.0;
    int best_idx = -1, best_lb = 0, best_rb = 0, best_int = -1;
    auto evaluate = [&](uint32_t key) {
        const uint32_t hp = key >> 8;
        const int p = (int)(key & 255u);
        int k = p, lb = p, rb = p;
        uint32_t lm = hp, rm = hp;
        while (k >= 0 && M(k) <= hp) { if (M(k) < lm) { lm = M(k); lb = k; } k--; }
        k = p;
        while (k <= nc - 1 && M(k) <= hp) { if (M(k) < rm) { rm = M(k); rb = k; } k++; }
        const double prom = xs(p) - xs(lm > rm ? lb : rb);      // fmax(xs[lb], xs[rb]): xs is monotone in m
        if (prom > best_prom || (prom == best_prom && p > best_idx)) { best_prom = prom; best_idx = p; best_lb = lb; best_rb = rb; }
        best_int = max(best_int, (int)(hp - max(lm, rm)));
    };
    // candidates from the highest down: one of height hp cannot have a prominence above hp - min(profile)
    evaluate(best1);
    if (best2 != 0 && (int)((best2 >> 8) - lmin) >= best_int) {      // rare: the runner-up could still win
        uint32_t bound = best1;
        while (true) {
            uint32_t key = 0;
            int start = -1;
            uint32_t prev = M(0);
            for (int i = 1; i < nc; i++) {
                const uint32_t v = M(i);
                if (v < prev && start >= 0) {
                    const uint32_t kk = (prev << 8) | (uint32_t)((start + i - 1) >> 1);
                    if (kk < bound && kk > key) key = kk;
                }
                start = v > prev ? i : (v < prev ? -1 : start);
                prev = v;
            }
            if (key == 0 || (int)((key >> 8) - lmin) < best_int) break;
            bound = key;
            evaluate(key);
        }
    }
    const int p = best_idx;
    const double h = xs(p) - best_prom * 0.5;
    // integer pre-filter for "h < xs[k]": xs is a monotone map of m, T = h * den + min is h in integer units up to ~1e-10
    const double T = h * den + (double)lmin;
    auto above = [&](int k) {
        const double mk = (double)M(k);
        if (mk > T + 0.5) return true;
        if (mk < T - 0.5) return false;
        return h < xs(k);
    };
    int kl = p;
    while (kl > best_lb && above(kl)) kl--;
    double l = (double)kl;
    {
        const double xk = xs(kl);
        if (xk < h) l += (h - xk) / (xs(kl + 1) - xk);
    }
    int kr = p;
    while (kr < best_rb && above(kr)) kr++;
    double r = (double)kr;
    {
        const double xk = xs(kr);
        if (xk < h) r -= (h - xk) / (xs(kr - 1) - xk);
    }
    out_l = l;
    out_r = r;
    return 1;
}


}  // namespace epid
