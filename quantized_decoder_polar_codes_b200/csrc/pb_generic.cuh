// Generic schedule-driven decoder kernel: one CTA decodes one frame at a time, all L paths in lock-step.
// Covers all 15 decoder kinds (every row of SURVEY.md 8a).  The specialised kernels in pb_scl_lut.cuh
// take over the LUT SC/SCL family when the shape allows; this one is the always-available CUDA path
// (there is no CPU fallback anywhere in the library).
//
// Per-path state is never copied on a list permutation.  Instead every path slot owns one physical buffer
// per tree level and a tiny pointer row says which physical slot currently holds level d of logical path i
// ("lazy copy").  Because all paths write level d+1 in the same step, ownership of that level snaps back
// to the writer's own slot, so a permutation only shuffles the pointer rows:
//   observationally identical to the reference's eager whole-state copies (PD/src/SCLLUTDecoder.cpp:132-144).
//
// Level layout inside a slot (N = code length):
//   V  (values: uint8 symbols or fp64 LLRs)  level d in [1,n] at offset N-(N>>(d-1)), N>>d live elements
//   UL (partial sums returned by LEFT children) same offsets, level d in [1,n], pointer-tracked
//   UR (partial sums returned by RIGHT children / the root) level d in [0,n] at N + 2N-2(N>>d), own slot only
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>

#include <algorithm>
#include <vector>

#include "pb_internal.h"

namespace pb {

// ------------------------------------------------------------------------------------------------
// libstdc++ std::sort on an index array with comparator key[a] < key[b] (GCC 13 bits/stl_algo.h:1848-1950),
// run by ONE thread.  n <= 16 is a plain insertion sort (stable); above that the introsort phases are
// reproduced so that the order of equal keys matches the reference build bit for bit (SURVEY App. B1).
// Sub-ranges produced by the partition step are disjoint, so processing them from an explicit stack in a
// different order than the recursion does not change the result.
// The algorithm is written once over an accessor (get/set of element i) and a strict-weak `less` on element VALUES,
// so that the same code sorts an index array through a key table (PtrAcc/KeyLess, below) and the packed, lane-strided
// shared-memory arrays of the warp kernels.
template <class A, class Less>
__device__ inline void ss_unguarded_linear_insert(A a, int last, Less less) {
    const typename A::V val = a.get(last);
    int next = last - 1;
    for (;;) {
        const typename A::V nv = a.get(next);
        if (!less(val, nv)) break;
        a.set(last, nv);
        last = next;
        --next;
    }
    a.set(last, val);
}
template <class A, class Less>
__device__ inline void ss_insertion_sort(A a, int first, int last, Less less) {
    if (first == last) return;
    for (int i = first + 1; i != last; ++i) {
        const typename A::V val = a.get(i);
        if (less(val, a.get(first))) {
            for (int k = i; k > first; --k) a.set(k, a.get(k - 1));
            a.set(first, val);
        } else {
            ss_unguarded_linear_insert(a, i, less);
        }
    }
}
template <class A, class Less>
__device__ inline void ss_push_heap(A a, int first, int hole, int top, typename A::V value, Less less) {
    int parent = (hole - 1) / 2;
    while (hole > top && less(a.get(first + parent), value)) {
        a.set(first + hole, a.get(first + parent));
        hole = parent;
        parent = (hole - 1) / 2;
    }
    a.set(first + hole, value);
}
template <class A, class Less>
__device__ inline void ss_adjust_heap(A a, int first, int hole, int len, typename A::V value, Less less) {
    const int top = hole;
    int child = hole;
    while (child < (len - 1) / 2) {
        child = 2 * (child + 1);
        if (less(a.get(first + child), a.get(first + child - 1))) child--;
        a.set(first + hole, a.get(first + child));
        hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
        child = 2 * (child + 1);
        a.set(first + hole, a.get(first + child - 1));
        hole = child - 1;
    }
    ss_push_heap(a, first, hole, top, value, less);
}
template <class A, class Less>
__device__ inline void ss_heapsort(A a, int first, int last, Less less) {
    int len = last - first;
    if (len >= 2) {
        int parent = (len - 2) / 2;
        for (;;) {
            const typename A::V value = a.get(first + parent);
            ss_adjust_heap(a, first, parent, len, value, less);
            if (parent == 0) break;
            parent--;
        }
    }
    while (last - first > 1) {
        --last;
        const typename A::V value = a.get(last);
        a.set(last, a.get(first));
        ss_adjust_heap(a, first, 0, last - first, value, less);
    }
}
template <class A>
__device__ inline void ss_swap(A a, int i, int j) { const typename A::V t = a.get(i); a.set(i, a.get(j)); a.set(j, t); }

// STK: capacity of the explicit range stack (one entry per pending right-hand partition: <= 2*log2(n) + 1)
template <int STK, class A, class Less>
__device__ inline void std_sort_acc(A a, int n, Less less) {
    if (n <= 1) return;
    if (n > 16) {
        int lg = 0;
        for (int t = n; t > 1; t >>= 1) lg++;
        int stk_f[STK], stk_l[STK], stk_d[STK];
        int sp = 0;
        stk_f[0] = 0; stk_l[0] = n; stk_d[0] = 2 * lg; sp = 1;
        while (sp > 0) {
            --sp;
            int first = stk_f[sp], last = stk_l[sp], depth = stk_d[sp];
            while (last - first > 16) {
                if (depth == 0) { ss_heapsort(a, first, last, less); break; }
                --depth;
                int mid = first + (last - first) / 2;
                // __move_median_to_first(first, first+1, mid, last-1)
                int ia = first + 1, ib = mid, ic = last - 1;
                const typename A::V ka = a.get(ia), kb = a.get(ib), kc = a.get(ic);
                if (less(ka, kb)) {
                    if (less(kb, kc)) ss_swap(a, first, ib);
                    else if (less(ka, kc)) ss_swap(a, first, ic);
                    else ss_swap(a, first, ia);
                } else if (less(ka, kc)) ss_swap(a, first, ia);
                else if (less(kb, kc)) ss_swap(a, first, ic);
                else ss_swap(a, first, ib);
                // __unguarded_partition(first+1, last, pivot = first)
                int lo = first + 1, hi = last;
                const typename A::V kp = a.get(first);
                for (;;) {
                    while (less(a.get(lo), kp)) ++lo;
                    --hi;
                    while (less(kp, a.get(hi))) --hi;
                    if (!(lo < hi)) break;
                    ss_swap(a, lo, hi);
                    ++lo;
                }
                // recurse on [lo,last), continue with [first,lo)
                stk_f[sp] = lo; stk_l[sp] = last; stk_d[sp] = depth; ++sp;
                last = lo;
            }
        }
        ss_insertion_sort(a, 0, 16, less);
        for (int i = 16; i < n; ++i) ss_unguarded_linear_insert(a, i, less);
    } else {
        ss_insertion_sort(a, 0, n, less);
    }
}

template <typename IdxT>
struct PtrAcc {
    using V = IdxT;
    IdxT *p;
    __device__ __forceinline__ V get(int i) const { return p[i]; }
    __device__ __forceinline__ void set(int i, V v) const { p[i] = v; }
};
template <typename IdxT>
struct KeyLess {
    const double *key;
    __device__ __forceinline__ bool operator()(IdxT x, IdxT y) const { return key[x] < key[y]; }
};
// index array `a` sorted by key[a[i]]
template <typename IdxT>
__device__ void std_sort_idx(IdxT *a, int n, const double *key) {
    std_sort_acc<40>(PtrAcc<IdxT>{a}, n, KeyLess<IdxT>{key});
}

// ------------------------------------------------------------------------------------------------
template <int DOM> struct Val { using T = double; };
template <> struct Val<DOM_LUT> { using T = uint8_t; };

#define PB_SGN(x) (((x) < 0) ? -1 : ((x) > 0))

__device__ __forceinline__ double dev_minsum(double a, double b) {  // PD/src/utils.cpp:26-30
    double fa = fabs(a), fb = fabs(b);
    return (double)(PB_SGN(a) * PB_SGN(b)) * (fa < fb ? fa : fb);
}
__device__ __forceinline__ double dev_g(double a, double b, int u) {  // utils.cpp:32-36
    return (double)(1 - 2 * u) * a + b;
}
__device__ __forceinline__ double dev_Q(double x, double r, double M) {  // utils.cpp:8-10
    return fabs(x) > M ? (double)PB_SGN(x) * (M - 0.5 * r) : (floor(x / r) + 0.5) * r;
}
__device__ __forceinline__ double dev_bisect(double a, const double *boundary, int nb, const double *rec) {
    int lo = 0, hi = nb;  // utils.cpp:12-24
    while (lo < hi) {
        int mid = (lo + hi) / 2;
        if (boundary[mid] < a) lo = mid + 1; else hi = mid;
    }
    return rec[lo > 0 ? lo - 1 : 0];   // (pd_create guarantees boundary[0] = -inf-like and nr >= nb-1; NaN input: first cell)
}

struct Ctl {
    double PM[kMaxL];
    double PM2[2 * kMaxL];
    int sidx[2 * kMaxL];
    uint8_t parent[kMaxL], flip[kMaxL], dec[kMaxL], rowp[kMaxL];
    int qsel[kMaxL];
    uint8_t ptrV[kMaxL][kMaxLog + 2];
    uint8_t ptrU[kMaxL][kMaxLog + 2];
    int winner;
    int pass;
    double dmetric;   // PD_BD_DMETRIC accumulator (DMetric.cpp:35,61,93)
    double bd_pm;     // PD_BD_CASCL: the PM value the reference returns
};

template <bool WARP>
__device__ __forceinline__ void gsync() {
    if (WARP) __syncwarp(); else __syncthreads();
}

// mink (PD/src/SCLLUTDecoder.cpp:8-22): L smallest of PM2[0..2L) in std::sort order -> parent/flip/PM.
template <bool WARP>
__device__ __forceinline__ void fork_select(Ctl &c, int L, int tid) {
    gsync<WARP>();
    if (2 * L <= 16) {
        if (tid < 2 * L) {
            double k = c.PM2[tid];
            int rank = 0;
            for (int j = 0; j < 2 * L; ++j) {
                double kj = c.PM2[j];
                rank += (kj < k) || (kj == k && j < tid);
            }
            c.sidx[rank] = tid;
        }
    } else if (tid == 0) {
        for (int j = 0; j < 2 * L; ++j) c.sidx[j] = j;
        std_sort_idx(c.sidx, 2 * L, c.PM2);
    }
    gsync<WARP>();
    if (tid < L) {
        int idx = c.sidx[tid];
        c.PM[tid] = c.PM2[idx];
        c.flip[tid] = idx >= L;
        c.parent[tid] = (uint8_t)(idx >= L ? idx - L : idx);
    }
    gsync<WARP>();
}

// slot i <- slot parent[i] for the pointer rows (the whole "copy" of a list permutation)
template <bool WARP>
__device__ __forceinline__ void permute_rows(Ctl &c, int L, int n, int tid, bool with_rowp) {
    uint8_t nv[kMaxLog + 2], nu[kMaxLog + 2];
    uint8_t nr = 0;
    if (tid < L) {
        int p = c.parent[tid];
#pragma unroll
        for (int lv = 0; lv < kMaxLog + 2; ++lv) { nv[lv] = c.ptrV[p][lv]; nu[lv] = c.ptrU[p][lv]; }
        nr = c.rowp[p];
    }
    gsync<WARP>();
    if (tid < L) {
#pragma unroll
        for (int lv = 0; lv < kMaxLog + 2; ++lv) { c.ptrV[tid][lv] = nv[lv]; c.ptrU[tid][lv] = nu[lv]; }
        if (with_rowp) c.rowp[tid] = nr;
    }
    gsync<WARP>();
}

template <int DOM, bool LIST, bool WARP>
__global__ void __launch_bounds__(256)
generic_decode_kernel(const Dev d, const void *__restrict__ in, int in_dtype, uint8_t *__restrict__ out,
                      long long B, char *ws, size_t ws_stride, int use_smem, int *err_flag,
                      double *dbg_pm, int *dbg_win) {
    using T = typename Val<DOM>::T;
    PB_DYN_SMEM(char, dyn_smem);
    __shared__ Ctl c;

    const int tid = threadIdx.x, nth = blockDim.x;
    const int N = d.N, n = d.n, L = LIST ? d.L : 1;
    const int VS = N, US = 3 * N;

    // carve the per-CTA workspace
    char *base = use_smem ? dyn_smem : ws + (size_t)blockIdx.x * ws_stride;
    T *V = reinterpret_cast<T *>(base);
    size_t off = ((size_t)L * VS * sizeof(T) + 15) & ~(size_t)15;   // (uint8 values: keep the fp64 scratch behind them aligned)
    double *AL = reinterpret_cast<double *>(base + off);       // R1 scratch: |llr| rows
    off += (size_t)L * d.r1_tmax * sizeof(double);
    int *SI = reinterpret_cast<int *>(base + off);              // R1 scratch: argsort rows
    off += (size_t)L * d.r1_tmax * sizeof(int);
    uint8_t *U = reinterpret_cast<uint8_t *>(base + off);
    off += (size_t)L * US;
    uint8_t *DEC = reinterpret_cast<uint8_t *>(base + off);     // R1 scratch: decisions, double buffered
    off += (size_t)2 * L * d.r1_tmax;
    uint8_t *X = reinterpret_cast<uint8_t *>(base + off);       // epilogue scratch [N]

#define OFFV(dd) (N - (N >> ((dd)-1)))
#define OFFUR(dd) (N + 2 * N - 2 * (N >> (dd)))

    for (long long frame = blockIdx.x; frame < B; frame += gridDim.x) {
        const uint8_t *in8 = reinterpret_cast<const uint8_t *>(in) + (size_t)frame * N;
        const int32_t *in32 = reinterpret_cast<const int32_t *>(in) + (size_t)frame * N;
        const double *in64 = reinterpret_cast<const double *>(in) + (size_t)frame * N;

        auto in0 = [&](int j) -> T {
            if (DOM == DOM_LUT) {
                int s = (in_dtype == 0) ? (int)in8[j] : in32[j];
                int bound = (j < N / 2) ? d.root_qa : d.root_qb;
                if (s < 0 || s >= bound) { *err_flag = 1; s = 0; }
                return (T)s;
            } else {
                return (T)in64[j];
            }
        };
        auto readV = [&](int i, int dd, int idx) -> T {
            if (dd == 0) return in0(idx);
            return V[(size_t)c.ptrV[i][dd] * VS + OFFV(dd) + idx];
        };
        // LLR seen at depth dd (>=1), node `node`, element j of path i
        auto elem_llr = [&](int i, int dd, unsigned node, int j) -> double {
            T v = readV(i, dd, j);
            if (DOM == DOM_LUT) {
                int pos = (int)(node << (n - dd)) + j;
                return d.llr[d.llr_off[(size_t)(dd - 1) * N + pos] + (int)v];
            } else {
                return (double)v;
            }
        };
        // destination of the partial sums a node at (dd,node) returns; marks ownership for left children
        auto result_ptr = [&](int i, int dd, unsigned node) -> uint8_t * {
            if (dd > 0 && (node & 1) == 0) return U + (size_t)i * US + OFFV(dd);
            return U + (size_t)i * US + OFFUR(dd);
        };

        if (tid < L) {
            c.PM[tid] = (tid == 0) ? 0.0 : d.pm_init;
            if (tid == 0) c.dmetric = 0.0;
            c.rowp[tid] = (uint8_t)tid;
            for (int lv = 0; lv < kMaxLog + 2; ++lv) { c.ptrV[tid][lv] = (uint8_t)tid; c.ptrU[tid][lv] = (uint8_t)tid; }
        }
        gsync<WARP>();

        for (int s = 0; s < d.n_steps; ++s) {
            const Step st = d.steps[s];
            const int dd = st.depth;
            const unsigned node = st.node;
            const int temp = N >> dd;
            switch (st.op) {
            case OP_F:
            case OP_G: {
                const int ct = temp >> 1, lct = n - dd - 1;
                const int p = (1 << dd) + (int)node - 1;
                const bool isg = st.op == OP_G;
                NodeTab tb;
                if (DOM == DOM_LUT) tb = d.tabs[p];
                double r = 0, M = 0;
                const double *bnd = nullptr, *rec = nullptr;
                if (DOM == DOM_UNIFORM) {
                    r = isg ? d.r_g[p] : d.r_f[p];
                    M = (isg ? d.mg_mul : d.mf_mul) * r;
                }
                if (DOM == DOM_LLOYD) {
                    bnd = (isg ? d.bnd_g : d.bnd_f) + (size_t)p * d.nb;
                    rec = (isg ? d.rec_g : d.rec_f) + (size_t)p * d.nr;
                }
                for (int it = tid; it < (L << lct); it += nth) {
                    const int i = it >> lct, j = it & (ct - 1);
                    T a = readV(i, dd, j), b = readV(i, dd, j + ct);
                    int u = 0;
                    if (isg) u = U[(size_t)c.ptrU[i][dd + 1] * US + OFFV(dd + 1) + j];
                    T o;
                    if (DOM == DOM_LUT) {
                        if (!isg) o = (T)d.lut[tb.f_off + (size_t)j * tb.f_pstride + (unsigned)a * tb.f_qb + (unsigned)b];
                        else o = (T)d.lut[tb.g_off + (size_t)j * tb.g_pstride + (unsigned)u * tb.g_sz + (unsigned)a * tb.g_qb + (unsigned)b];
                    } else {
                        double x = isg ? dev_g((double)a, (double)b, u) : dev_minsum((double)a, (double)b);
                        if (DOM == DOM_UNIFORM) x = dev_Q(x, r, M);
                        if (DOM == DOM_LLOYD) x = dev_bisect(x, bnd, d.nb, rec);
                        o = (T)x;
                    }
                    V[(size_t)i * VS + OFFV(dd + 1) + j] = o;
                }
                gsync<WARP>();   // all reads through ptrV[.][dd] done (dd+1 rows are not read in this step)
                if (tid < L) c.ptrV[tid][dd + 1] = (uint8_t)tid;
                break;
            }
            case OP_C: {
                const int ct = temp >> 1, lct = n - dd - 1;
                for (int it = tid; it < (L << lct); it += nth) {
                    const int i = it >> lct, j = it & (ct - 1);
                    uint8_t ul = U[(size_t)c.ptrU[i][dd + 1] * US + OFFV(dd + 1) + j];
                    uint8_t ur = U[(size_t)i * US + OFFUR(dd + 1) + j];
                    uint8_t *dst = result_ptr(i, dd, node);
                    dst[j] = ul ^ ur;
                    dst[j + ct] = ur;
                }
                gsync<WARP>();
                if (tid < L && dd > 0 && (node & 1) == 0) c.ptrU[tid][dd] = (uint8_t)tid;
                break;
            }
            case OP_LEAF: {
                if (!LIST) {
                    if (tid == 0) {
                        uint8_t bit = 0;
                        if (!st.flag) bit = (uint8_t)(elem_llr(0, n, node, 0) <= 0);  // PD/src/SCDecoder.cpp:31
                        result_ptr(0, n, node)[0] = bit;
                    }
                } else if (st.flag) {
                    if (tid < L) {   // PD/src/SCLLUTDecoder.cpp:99-104
                        double DM = elem_llr(tid, n, node, 0);
                        c.PM[tid] += fabs(DM) * (double)(DM < 0);
                        result_ptr(tid, n, node)[0] = 0;
                        if ((node & 1) == 0) c.ptrU[tid][n] = (uint8_t)tid;
                    }
                } else {
                    if (tid < L) {   // PD/src/SCLLUTDecoder.cpp:105-115
                        double DM = elem_llr(tid, n, node, 0);
                        c.dec[tid] = (uint8_t)(DM < 0);
                        c.PM2[tid] = c.PM[tid];
                        c.PM2[tid + L] = c.PM[tid] + fabs(DM);
                    }
                    fork_select<WARP>(c, L, tid);
                    permute_rows<WARP>(c, L, n, tid, false);
                    if (tid < L) {
                        uint8_t bit = c.dec[c.parent[tid]];
                        if (c.flip[tid]) bit = 1 - bit;
                        result_ptr(tid, n, node)[0] = bit;
                        if ((node & 1) == 0) c.ptrU[tid][n] = (uint8_t)tid;
                    }
                }
                break;
            }
            case OP_R0: {
                if (LIST) {
                    if (tid < L) {   // PD/src/FastSCLLUTDecoder.cpp:83-93, serial fp64 order
                        double pm = c.PM[tid];
                        for (int j = 0; j < temp; ++j) {
                            double l = elem_llr(tid, dd, node, j);
                            pm += (double)(float)(l < 0) * fabs(l);
                        }
                        c.PM[tid] = pm;
                    }
                }
                if (!LIST && d.bd == 1 && tid == 0) {   // DMetric.cpp:56-61: DMetric += (sum of the node's LLRs) / temp
                    double tmp = 0;
                    for (int j = 0; j < temp; ++j) tmp += elem_llr(0, dd, node, j);
                    c.dmetric += tmp / temp;
                }
                for (int it = tid; it < L * temp; it += nth) {
                    const int i = it / temp, j = it - i * temp;
                    result_ptr(i, dd, node)[j] = 0;
                }
                gsync<WARP>();
                if (tid < L && (node & 1) == 0) c.ptrU[tid][dd] = (uint8_t)tid;
                break;
            }
            case OP_REP: {
                if (!LIST) {
                    if (tid == 0) {   // PD/src/FastSCLUT.cpp:67-79
                        double S = 0;
                        for (int j = 0; j < temp; ++j) S += elem_llr(0, dd, node, j);
                        c.dec[0] = (uint8_t)(S <= 0);
                        if (d.bd == 1) c.dmetric += fabs(S) / temp;   // DMetric.cpp:87-93
                    }
                    gsync<WARP>();
                    for (int j = tid; j < temp; j += nth) result_ptr(0, dd, node)[j] = c.dec[0];
                } else {
                    if (tid < L) {   // PD/src/FastSCLLUTDecoder.cpp:169-184
                        double a0 = c.PM[tid], a1 = c.PM[tid];
                        for (int j = 0; j < temp; ++j) {
                            double l = elem_llr(tid, dd, node, j);
                            a0 += (double)(l < 0) * fabs(l);
                            a1 += (double)(l >= 0) * fabs(l);
                        }
                        c.PM2[tid] = a0;
                        c.PM2[tid + L] = a1;
                    }
                    fork_select<WARP>(c, L, tid);
                    permute_rows<WARP>(c, L, n, tid, false);
                    for (int it = tid; it < L * temp; it += nth) {
                        const int i = it / temp, j = it - i * temp;
                        result_ptr(i, dd, node)[j] = c.flip[i];
                    }
                }
                gsync<WARP>();
                if (tid < L && (node & 1) == 0) c.ptrU[tid][dd] = (uint8_t)tid;
                break;
            }
            case OP_R1: {
                if (!LIST) {   // PD/src/FastSCLUT.cpp:54-66
                    for (int j = tid; j < temp; j += nth) result_ptr(0, dd, node)[j] = (uint8_t)(elem_llr(0, dd, node, j) <= 0);
                } else {       // PD/src/FastSCLLUTDecoder.cpp:98-165 incl. the flip-index quirk (SURVEY App. B4)
                    const int TM = d.r1_tmax;
                    const int rounds = (L - 1 < temp) ? L - 1 : temp;
                    int cur = 0;
                    for (int it = tid; it < L * temp; it += nth) {
                        const int i = it / temp, j = it - i * temp;
                        double l = elem_llr(i, dd, node, j);
                        DEC[(size_t)i * TM + j] = (uint8_t)(l < 0);
                        AL[(size_t)i * TM + j] = fabs(l);
                        SI[(size_t)i * TM + j] = j;
                    }
                    if (tid < L) c.rowp[tid] = (uint8_t)tid;
                    gsync<WARP>();
                    if (tid < L) std_sort_idx(SI + (size_t)tid * TM, temp, AL + (size_t)tid * TM);
                    gsync<WARP>();
                    for (int layer = 0; layer < rounds; ++layer) {
                        if (tid < L) {
                            int row = c.rowp[tid];
                            int q = SI[(size_t)row * TM + layer];
                            c.qsel[tid] = q;
                            c.PM2[tid] = c.PM[tid];
                            c.PM2[tid + L] = c.PM[tid] + AL[(size_t)row * TM + q];
                        }
                        fork_select<WARP>(c, L, tid);
                        uint8_t *src = DEC + (size_t)cur * L * TM, *dst = DEC + (size_t)(cur ^ 1) * L * TM;
                        for (int it = tid; it < L * temp; it += nth) {
                            const int i = it / temp, j = it - i * temp;
                            uint8_t b = src[(size_t)c.parent[i] * TM + j];
                            if (c.flip[i] && j == c.qsel[i]) b = 1 - b;   // slot i's OWN pre-permutation index
                            dst[(size_t)i * TM + j] = b;
                        }
                        permute_rows<WARP>(c, L, n, tid, true);
                        cur ^= 1;
                    }
                    const uint8_t *src = DEC + (size_t)cur * L * TM;
                    for (int it = tid; it < L * temp; it += nth) {
                        const int i = it / temp, j = it - i * temp;
                        result_ptr(i, dd, node)[j] = src[(size_t)i * TM + j];
                    }
                }
                gsync<WARP>();
                if (tid < L && (node & 1) == 0) c.ptrU[tid][dd] = (uint8_t)tid;
                break;
            }
            case OP_SPC: {   // non-list only (PD/src/FastSCLUT.cpp:80-106): Wagner, first arg-min |llr|
                for (int j = tid; j < temp; j += nth) result_ptr(0, dd, node)[j] = (uint8_t)(elem_llr(0, dd, node, j) <= 0);
                gsync<WARP>();
                if (tid == 0) {
                    uint8_t *r = result_ptr(0, dd, node);
                    int parity = 0, amin = 0;
                    double best = 0;
                    for (int j = 0; j < temp; ++j) {
                        double al = fabs(elem_llr(0, dd, node, j));
                        parity += r[j];
                        if (j == 0 || al < best) { best = al; amin = j; }
                    }
                    if (parity & 1) r[amin] = 1 - r[amin];
                }
                gsync<WARP>();
                if (tid < L && (node & 1) == 0) c.ptrU[tid][dd] = (uint8_t)tid;
                break;
            }
            }
            gsync<WARP>();
        }

        // ---------------- epilogue: pick the path, recover u = x F^{(x)n}, gather ----------------
        auto load_transform = [&](int slot) {
            const uint8_t *x = U + (size_t)slot * US + OFFUR(0);
            for (int j = tid; j < N; j += nth) X[j] = x[j];
            gsync<WARP>();
            for (int m = 1; m < N; m <<= 1) {
                for (int t = tid; t < N / 2; t += nth) {
                    int blk = t / m, jj = t - blk * m;
                    int i0 = blk * 2 * m + jj;
                    X[i0] ^= X[i0 + m];
                }
                gsync<WARP>();
            }
        };
        if (tid == 0) {
            int w = 0;
            if (LIST) {
                if (!d.ca) {
                    for (int i = 1; i < L; ++i) if (c.PM[i] < c.PM[w]) w = i;   // std::min_element
                } else {
                    for (int i = 0; i < L; ++i) c.sidx[i] = i;
                    std_sort_idx(c.sidx, L, c.PM);                              // argsort(PML)
                    w = c.sidx[0];
                }
            }
            c.winner = w;
            c.pass = 0;
            c.bd_pm = LIST ? c.PM[0] : 0.0;   // CASCLWithRNTI.cpp:205: PM = PML[0]
        }
        gsync<WARP>();
        if (LIST && d.ca) {
            for (int t = 0; t < L; ++t) {   // PD/src/CASCLLUTDecoder.cpp:264-289
                int cand = c.sidx[t];
                load_transform(cand);
                if (tid == 0) {
                    uint32_t reg = 0;
                    const uint32_t msb = 1u << (d.crc_n - 1);
                    const uint32_t mask = (d.crc_n >= 32) ? 0xffffffffu : ((1u << d.crc_n) - 1u);
                    for (int k = 0; k < d.A; ++k) {
                        uint32_t top = ((reg & msb) ? 1u : 0u) ^ (uint32_t)X[d.info_pos[k]];
                        reg = (reg << 1) & mask;
                        if (top) reg ^= d.crc_taps;
                    }
                    int ok = 1;
                    for (int k = 0; k < d.crc_check; ++k) {
                        uint32_t bit = (reg >> (d.crc_n - 1 - k)) & 1u;
                        // CASCLWithRNTI.cpp:224-226: the RNTI is added onto the last RNTILength check bits
                        if (d.bd_rnti_len > 0 && k >= d.crc_n - d.bd_rnti_len) bit ^= (uint32_t)(d.bd_rnti[k - (d.crc_n - d.bd_rnti_len)] & 1);
                        if (bit != (uint32_t)X[d.info_pos[d.A + k]]) { ok = 0; break; }
                    }
                    if (ok) { c.winner = cand; c.pass = 1; c.bd_pm = c.PM[t]; }   // :236 PM = PML[i] (slot i, not the candidate's)
                }
                gsync<WARP>();
                if (c.pass) break;
            }
            if (!c.pass) load_transform(c.winner);
        } else {
            load_transform(c.winner);
        }
        if (out) for (int k = tid; k < d.Kout; k += nth) out[(size_t)frame * d.Kout + k] = X[d.info_pos[k]];
        if (d.bd_metric && tid == 0) d.bd_metric[frame] = d.bd == 1 ? c.dmetric : c.bd_pm;
        if (d.bd_pass && tid == 0) d.bd_pass[frame] = (uint8_t)c.pass;
        if (dbg_pm && tid < L) dbg_pm[(size_t)frame * L + tid] = LIST ? c.PM[tid] : 0.0;
        if (dbg_win && tid == 0) dbg_win[frame] = c.winner;
        gsync<WARP>();
    }
#undef OFFV
#undef OFFUR
}

const void *generic_kernel_fn(int dom, bool list, bool warp);   // instantiations: pb_kernels.cu

// ------------------------------------------------------------------------------------------------
// host side

// Copies n elements of h into a new device buffer (at least 16 bytes) and records it in `allocs`, whose owner frees it.
template <typename T>
inline cudaError_t upload(std::vector<void *> &allocs, const T *h, size_t n, const T **out) {
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, std::max<size_t>(n * sizeof(T), 16));
    if (e != cudaSuccess) return e;
    allocs.push_back(p);
    if (n && (e = cudaMemcpy(p, h, n * sizeof(T), cudaMemcpyHostToDevice)) != cudaSuccess) return e;
    *out = reinterpret_cast<const T *>(p);
    return cudaSuccess;
}

struct GenericPlan {
    int threads = 32;
    size_t ws_bytes = 0;   // per-CTA workspace
    int use_smem = 0;      // the workspace lives in dynamic shared memory, else in global memory
    int ctas_per_sm = 1;
};

// Block size and workspace of the CTA-per-frame kernel; ctas_per_sm < 1 when it does not fit on the device.
inline cudaError_t plan_generic(const Dev &d, GenericPlan *pl) {
    const int L = d.list ? d.L : 1;
    const size_t vsz = d.domain == DOM_LUT ? 1 : 8;
    size_t ws = (((size_t)L * d.N * vsz + 15) & ~(size_t)15) + (size_t)L * d.r1_tmax * (8 + 4) + (size_t)L * 3 * d.N + (size_t)2 * L * d.r1_tmax + d.N;
    ws = (ws + 15) & ~(size_t)15;
    pl->ws_bytes = ws;
    const int64_t work = (int64_t)L * d.N / 2;
    int th = 32;
    while (th < 256 && th * 8 < work) th *= 2;
    pl->threads = th;
    pl->use_smem = ws <= 96 * 1024;
    const void *fn = generic_kernel_fn(d.domain, d.list != 0, th == 32);
    // (the attribute belongs to the kernel function, which every decoder of the same domain shares: always the cap, never
    //  this decoder's own size -- a smaller decoder created later must not shrink it under a live larger one)
    if (pl->use_smem) {
        const cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
        if (e != cudaSuccess) return e;
    }
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(&pl->ctas_per_sm, fn, th, pl->use_smem ? ws : 0);
}

inline int generic_grid(const GenericPlan &pl, long long B, int sm_count) {
    return (int)std::max<long long>(1, std::min<long long>((long long)sm_count * pl.ctas_per_sm, B));
}

inline int launch_generic(const Dev &d, const GenericPlan &pl, const void *d_in, int dtype, long long B, uint8_t *d_out,
                          cudaStream_t s, char *ws, int *d_err, double *dbg_pm, int *dbg_win, int sm_count) {
    const int grid = generic_grid(pl, B, sm_count);
    void *args[] = {(void *)&d, (void *)&d_in, (void *)&dtype, (void *)&d_out, (void *)&B, (void *)&ws, (void *)&pl.ws_bytes,
                    (void *)&pl.use_smem, (void *)&d_err, (void *)&dbg_pm, (void *)&dbg_win};
    cudaError_t e = cudaLaunchKernel(generic_kernel_fn(d.domain, d.list != 0, pl.threads == 32), dim3(grid), dim3(pl.threads), args,
                                     pl.use_smem ? pl.ws_bytes : 0, s);
    if (e != cudaSuccess) return (int)e;
    return (int)cudaGetLastError();
}

}  // namespace pb
