// beam_search.cu — batched beam-search decode for sm_100a.
//
// Replaces simple_beam_search(log_probs[T,V], beam_width, blank) (/root/reference/beam_search.py:2-42),
// which the reference calls once per utterance from a Python loop (model/trainer.py:229-242) at a cost
// of one torch.topk launch and 2*k*n_beams .item() host syncs per frame.
//
// Exact semantics kept (SURVEY.md §8 a13):
//   * per frame: torch.topk(row, k) INCLUDING the CPU kernel's tie order (libstdc++ std::partial_sort
//     with the comparator of ATen/native/TopKImpl.h:56-58, used when k*64 <= V)
//   * every beam extended by the k tokens in order; scores are fp64 = score + double(log_p)
//   * prune = stable sort by score descending (ties keep insertion order: beam-major, k-minor)
//   * result = CTC collapse of beams[0] where `prev` is updated on every frame, blank included
//
// Three routes over the same building blocks (DESIGN.md §4.9):
//   * beam_fused_kernel   V in 513..832, <= 32 candidates, short utterances, up to 16 x SMs of them per call: persistent
//                         CTAs, top-k warps feed recurrence warps through shared memory
//   * beam_topk_kernel + beam_recur_kernel   V <= 1024: top-k of all N*T rows (one warp per row, row in registers), then
//                         one warp per utterance over the [T,beam] lists
//   * beam_search_kernel  any V: one warp per utterance does both, rows staged through a 3-deep cp.async ring
// Per row the warp (1) finds the top-(k+1) with a threshold pass (lane maxima -> (k+1)-th largest -> compaction ->
// rank); when those k+1 values are pairwise distinct and NaN-free the top-k is unique and any algorithm agrees with
// torch.  Otherwise (2) it runs the literal libstdc++ heap-select/sort-heap (or nth_element + sort) on the
// shared-memory row (one lane owns the heap, the warp scans ahead with ballots).  (3) Only the (b+1)(j+1) <= beam
// candidates can survive the prune (every (b',j') <= (b,j) sorts first), so <= ~beam*ln(beam) candidates are ranked by
// counting, scores in fp64, back-pointers kept per frame.
#include "common.cuh"
#include "beam_internal.h"

namespace avctc {

constexpr int kBeamMax = 32;       // beam widths supported by the kernel
constexpr int kCandMax = 64;       // fast-path candidate list
constexpr int kCandPad = kCandMax + 4;   // + one 16-byte group of padding for the vector rank loop (two-phase kernel)
constexpr int kRowBufs = 3;
constexpr int kBpSmemBytes = 24 * 1024;

struct BeamParams {
    const float* lp; int64_t stride_n, stride_t;
    int N, T, V;
    const int64_t* lengths;
    int beam, blank, fast;
    int32_t* out_ids; int32_t* out_len; double* dbg_scores; int32_t* dbg_paths;
    uint32_t* bp_global;   // [N][T][beam] when back-pointers do not fit shared memory, else nullptr
    int32_t* path_ws;      // [N][T]
    int* status;           // device int error channel (0 = ok)
    int row_floats;        // smem floats per staged row
    int n_enum;            // number of (b,j) candidate pairs
    int use_nth;           // k*64 > V: torch.topk's nth_element + sort route for tied rows
    int prefetch;          // top-k kernel: L2-prefetch the warp's next row (tuning knob "beam_pf")
    float* tk_val;         // [N][T][beam] per-frame top-k values (two-phase path)
    int32_t* tk_idx;       // [N][T][beam] per-frame top-k indices
};

__device__ __forceinline__ bool ranks_before(float x, float y) {  // TopKImpl.h:56-58
    return ((x != x) && !(y != y)) || (x > y);
}

// libstdc++ std::__adjust_heap + std::__push_heap on (value,index) pairs with comp = ranks_before.
__device__ void adjust_heap(volatile float* hv, volatile int* hi, int hole, int len, float val, int vidx) {
    const int top = hole;
    int child = hole;
    while (child < (len - 1) / 2) {
        child = 2 * (child + 1);
        if (ranks_before(hv[child], hv[child - 1])) child--;
        hv[hole] = hv[child]; hi[hole] = hi[child];
        hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
        child = 2 * (child + 1);
        hv[hole] = hv[child - 1]; hi[hole] = hi[child - 1];
        hole = child - 1;
    }
    int parent = (hole - 1) / 2;
    while (hole > top && ranks_before(hv[parent], val)) {
        hv[hole] = hv[parent]; hi[hole] = hi[parent];
        hole = parent;
        parent = (hole - 1) / 2;
    }
    hv[hole] = val; hi[hole] = vidx;
}

// exact std::partial_sort(queue, queue+k, queue+V, ranks_before) -> (tv,ti)[0..k)
__device__ void topk_exact(const float* row, int V, int k, volatile float* tv, volatile int* ti, int lane) {
    if (lane == 0) {
        for (int j = 0; j < k; ++j) { tv[j] = row[j]; ti[j] = j; }
        if (k >= 2) {  // std::__make_heap
            int parent = (k - 2) / 2;
            while (true) {
                const float v = tv[parent]; const int vi = ti[parent];
                adjust_heap(tv, ti, parent, k, v, vi);
                if (parent == 0) break;
                parent--;
            }
        }
    }
    __syncwarp();
    for (int i0 = k; i0 < V; i0 += 32) {  // std::__heap_select, warp looks 32 elements ahead
        const int i = i0 + lane;
        const float v = (i < V) ? row[i] : 0.f;
        float top = tv[0];
        unsigned m = __ballot_sync(kFullMask, i < V && ranks_before(v, top));
        while (m) {
            const int l = __ffs(m) - 1;
            const float pv = __shfl_sync(kFullMask, v, l);
            if (lane == 0) adjust_heap(tv, ti, 0, k, pv, i0 + l);   // std::__pop_heap(first, middle, i)
            __syncwarp();
            top = tv[0];
            m = __ballot_sync(kFullMask, i < V && lane > l && ranks_before(v, top));
        }
    }
    if (lane == 0) {  // std::__sort_heap
        int last = k;
        while (last > 1) {
            --last;
            const float v = tv[last]; const int vi = ti[last];
            tv[last] = tv[0]; ti[last] = ti[0];
            adjust_heap(tv, ti, 0, last, v, vi);
        }
    }
    __syncwarp();
}


// ---- literal libstdc++ (GCC 13) std::nth_element + std::sort on (value,index) pairs, one lane, in place.
// torch.topk takes this route when k*64 > V (TopKImpl.h:45,66-76); only reached when the fast path saw ties.
struct PairQ { volatile float* v; volatile int* i; };
__device__ __forceinline__ bool q_cmp(const PairQ& q, int a, int b) { return ranks_before(q.v[a], q.v[b]); }
__device__ __forceinline__ void q_swap(const PairQ& q, int a, int b) {
    const float x = q.v[a]; const int xi = q.i[a];
    q.v[a] = q.v[b]; q.i[a] = q.i[b];
    q.v[b] = x; q.i[b] = xi;
}
__device__ void q_make_heap(const PairQ& q, int first, int last) {
    const int len = last - first;
    if (len < 2) return;
    int parent = (len - 2) / 2;
    while (true) {
        const float v = q.v[first + parent]; const int vi = q.i[first + parent];
        adjust_heap(q.v + first, q.i + first, parent, len, v, vi);
        if (parent == 0) return;
        parent--;
    }
}
__device__ void q_pop_heap(const PairQ& q, int first, int last, int result) {
    const float v = q.v[result]; const int vi = q.i[result];
    q.v[result] = q.v[first]; q.i[result] = q.i[first];
    adjust_heap(q.v + first, q.i + first, 0, last - first, v, vi);
}
__device__ void q_heap_select(const PairQ& q, int first, int middle, int last) {
    q_make_heap(q, first, middle);
    for (int i = middle; i < last; ++i)
        if (q_cmp(q, i, first)) q_pop_heap(q, first, middle, i);
}
__device__ void q_sort_heap(const PairQ& q, int first, int last) {
    while (last - first > 1) { --last; q_pop_heap(q, first, last, last); }
}
__device__ void q_move_median_to_first(const PairQ& q, int result, int a, int b, int c) {
    if (q_cmp(q, a, b)) {
        if (q_cmp(q, b, c)) q_swap(q, result, b);
        else if (q_cmp(q, a, c)) q_swap(q, result, c);
        else q_swap(q, result, a);
    } else if (q_cmp(q, a, c)) q_swap(q, result, a);
    else if (q_cmp(q, b, c)) q_swap(q, result, c);
    else q_swap(q, result, b);
}
__device__ int q_unguarded_partition(const PairQ& q, int first, int last, int pivot) {
    while (true) {
        while (q_cmp(q, first, pivot)) ++first;
        --last;
        while (q_cmp(q, pivot, last)) --last;
        if (!(first < last)) return first;
        q_swap(q, first, last);
        ++first;
    }
}
__device__ int q_partition_pivot(const PairQ& q, int first, int last) {
    const int mid = first + (last - first) / 2;
    q_move_median_to_first(q, first, first + 1, mid, last - 1);
    return q_unguarded_partition(q, first + 1, last, first);
}
__device__ void q_unguarded_linear_insert(const PairQ& q, int last) {
    const float v = q.v[last]; const int vi = q.i[last];
    int next = last - 1;
    while (ranks_before(v, q.v[next])) {
        q.v[last] = q.v[next]; q.i[last] = q.i[next];
        last = next; --next;
    }
    q.v[last] = v; q.i[last] = vi;
}
__device__ void q_insertion_sort(const PairQ& q, int first, int last) {
    if (first == last) return;
    for (int i = first + 1; i != last; ++i) {
        if (q_cmp(q, i, first)) {
            const float v = q.v[i]; const int vi = q.i[i];
            for (int j = i; j > first; --j) { q.v[j] = q.v[j - 1]; q.i[j] = q.i[j - 1]; }
            q.v[first] = v; q.i[first] = vi;
        } else {
            q_unguarded_linear_insert(q, i);
        }
    }
}
__device__ __forceinline__ int q_lg(int n) { return 31 - __clz(n); }
__device__ void q_nth_element(const PairQ& q, int first, int nth, int last) {
    if (first == last || nth == last) return;
    int depth = q_lg(last - first) * 2;
    while (last - first > 3) {
        if (depth == 0) {
            q_heap_select(q, first, nth + 1, last);
            q_swap(q, first, nth);
            return;
        }
        --depth;
        const int cut = q_partition_pivot(q, first, last);
        if (cut <= nth) first = cut; else last = cut;
    }
    q_insertion_sort(q, first, last);
}
__device__ void q_sort(const PairQ& q, int first, int last) {
    if (first == last) return;
    // std::__introsort_loop with an explicit stack (the recursive call handles [cut,last))
    int stk_f[40], stk_l[40], stk_d[40];
    int sp = 0;
    stk_f[0] = first; stk_l[0] = last; stk_d[0] = q_lg(last - first) * 2; sp = 1;
    while (sp > 0) {
        --sp;
        int f = stk_f[sp], l = stk_l[sp], d = stk_d[sp];
        while (l - f > 16) {
            if (d == 0) { q_heap_select(q, f, l, l); q_sort_heap(q, f, l); break; }
            --d;
            const int cut = q_partition_pivot(q, f, l);
            if (sp < 40) { stk_f[sp] = cut; stk_l[sp] = l; stk_d[sp] = d; ++sp; }
            l = cut;
        }
    }
    // std::__final_insertion_sort
    if (last - first > 16) {
        q_insertion_sort(q, first, first + 16);
        for (int i = first + 16; i != last; ++i) q_unguarded_linear_insert(q, i);
    } else {
        q_insertion_sort(q, first, last);
    }
}
// exact nth_element(queue, queue+k-1, queue+V) + sort(queue, queue+k-1); mutates the staged row.
__device__ void topk_nth_exact(float* row, int* qi, int V, int k, volatile float* tv, volatile int* ti, int lane) {
    for (int c = lane; c < V; c += 32) qi[c] = c;
    __syncwarp();
    if (lane == 0) {
        PairQ q{row, qi};
        q_nth_element(q, 0, k - 1, V);
        q_sort(q, 0, k - 1);
        for (int j = 0; j < k; ++j) { tv[j] = q.v[j]; ti[j] = q.i[j]; }
    }
    __syncwarp();
}

// threshold top-k; returns false when the result is not provably tie-free (caller runs topk_exact)
__device__ bool topk_fast(const float* row, int V, int k, float* cv, int* ci, volatile float* tv,
                          volatile int* ti, int lane) {
    if (k + 1 > 32 || V < k + 1) return false;
    float ml = AVCTC_NEG_INF;
    bool bad = false;
    for (int c = lane; c < V; c += 32) {
        const float v = row[c];
        bad |= (v != v);
        ml = fmaxf(ml, v);
    }
    if (__any_sync(kFullMask, bad)) return false;
    // (k+1)-th largest lane maximum: a lower bound of the (k+1)-th largest element
    int rank = 0;
#pragma unroll 8
    for (int j = 0; j < 32; ++j) {
        const float o = __shfl_sync(kFullMask, ml, j);
        rank += (o > ml) || (o == ml && j < lane);
    }
    const unsigned who = __ballot_sync(kFullMask, rank == k);
    const float tau = __shfl_sync(kFullMask, ml, __ffs(who) - 1);
    // compaction of everything >= tau
    int count = 0;
    for (int c0 = 0; c0 < V; c0 += 32) {
        const int c = c0 + lane;
        const float v = (c < V) ? row[c] : AVCTC_NEG_INF;
        const bool take = (c < V) && (v >= tau);
        const unsigned m = __ballot_sync(kFullMask, take);
        const int pos = count + __popc(m & ((1u << lane) - 1));
        if (take && pos < kCandMax) { cv[pos] = v; ci[pos] = c; }
        count += __popc(m);
    }
    if (count > kCandMax || count < k + 1) return false;
    __syncwarp();
    // rank the candidates (value desc, index asc); keep ranks 0..k
    for (int i = lane; i < count; i += 32) {
        const float v = cv[i]; const int idx = ci[i];
        int r = 0;
        for (int j = 0; j < count; ++j) {
            const float o = cv[j];
            r += (o > v) || (o == v && ci[j] < idx);
        }
        if (r <= k) { tv[r] = v; ti[r] = idx; }
    }
    __syncwarp();
    const bool tie = (lane < k) && (tv[lane] == tv[lane + 1]);
    if (__any_sync(kFullMask, tie)) return false;
    return true;
}

// 32-bit shared-window accessors: the recurrence's scratch is addressed without the generic-pointer conversion the
// compiler would otherwise re-derive (S2UR + ULEA) every frame
__device__ __forceinline__ uint32_t smem_addr(const void* ptr) { return (uint32_t)__cvta_generic_to_shared(ptr); }
__device__ __forceinline__ double lds_f64(uint32_t a) { double v; asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void sts_f64(uint32_t a, double v) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory"); }
__device__ __forceinline__ double2 lds_v2f64(uint32_t a) {
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ int lds_s32(uint32_t a) { int v; asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void sts_s32(uint32_t a, int v) { asm volatile("st.shared.s32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_u16(uint32_t a, unsigned v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"((unsigned short)v) : "memory"); }

// One frame of the prune when the (b+1)(j+1) <= beam candidates fit one warp: lane m IS candidate m = (my_b, my_j).
// (tvv, tii) = this frame's top-k list (lane j holds entry j).  Shared addresses: sc_a / sn_a = scores of the current /
// next beams (kBeamMax doubles each), cand_a = 32 candidate scores, bp16_a = this frame's 16-bit back-pointer row (0:
// 32-bit entries through bp_t).  Rank = number of strictly greater scores; equal scores give equal ranks: two survivors
// that share a rank store to the same slot, which each detects by reading back the lane tag it left beside its score
// (the tags live in the current-score row, dead once the candidates are built) -> stable (insertion-order) ranks and a
// second store.  (A match.any on the ranks costs several hundred cycles of latency per frame: ncu, round 2.)
// Returns the number of beams kept.
__device__ __forceinline__ int recur_step_enum32(const float tvv, const int tii, const int my_b, const int my_j,
                                                 const int n_enum, const int nb, const int k, const uint32_t sc_a,
                                                 const uint32_t sn_a, const uint32_t cand_a, const uint32_t bp16_a,
                                                 uint32_t* bp_t, const int lane) {
    const bool in = (lane < n_enum) && (my_b < nb);
    const int M = __popc(__ballot_sync(kFullMask, in));        // candidates are ordered by beam: `in` is a prefix
    const float lpv = __shfl_sync(kFullMask, tvv, my_j);
    const int tok = __shfl_sync(kFullMask, tii, my_j);
    const double s = in ? lds_f64(sc_a + my_b * 8) + (double)lpv : __longlong_as_double(0x7ff8000000000000ll);
    sts_f64(cand_a + lane * 8, s);
    __syncwarp();
    const int keep = min(k, M);
    // every lane wrote its slot (NaN where it holds no candidate), so the 32 slots are compared in two unrolled halves:
    // eight 16-byte loads in flight, four chains of predicated increments (DSETP + @p IADD per compare), no loop tail
    int r = 0;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        if (h == 0 || M > 16) {
            int ra = 0, rb = 0, rc = 0, rd = 0;
            double2 o[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) o[q] = lds_v2f64(cand_a + (8 * h + q) * 16);
#pragma unroll
            for (int q = 0; q < 8; q += 2) {
                asm("{\n\t.reg .pred p;\n\tsetp.gt.f64 p, %1, %2;\n\t@p add.s32 %0, %0, 1;\n\t}" : "+r"(ra) : "d"(o[q].x), "d"(s));
                asm("{\n\t.reg .pred p;\n\tsetp.gt.f64 p, %1, %2;\n\t@p add.s32 %0, %0, 1;\n\t}" : "+r"(rb) : "d"(o[q].y), "d"(s));
                asm("{\n\t.reg .pred p;\n\tsetp.gt.f64 p, %1, %2;\n\t@p add.s32 %0, %0, 1;\n\t}" : "+r"(rc) : "d"(o[q + 1].x), "d"(s));
                asm("{\n\t.reg .pred p;\n\tsetp.gt.f64 p, %1, %2;\n\t@p add.s32 %0, %0, 1;\n\t}" : "+r"(rd) : "d"(o[q + 1].y), "d"(s));
            }
            r += (ra + rb) + (rc + rd);
        }
    }
    const unsigned bpe16 = (unsigned)((my_b << 10) | tok);
    const uint32_t bpe32 = ((uint32_t)my_b << 24) | (uint32_t)tok;
    const bool wr = in && r < keep;
    if (wr) {
        sts_f64(sn_a + r * 8, s);
        sts_s32(sc_a + r * 4, lane);
        if (bp16_a) sts_u16(bp16_a + r * 2, bpe16);
        else bp_t[r] = bpe32;
    }
    __syncwarp();
    const int tag = lds_s32(sc_a + r * 4);             // r <= 32: inside the row for every lane, no branch around the load
    const bool clash = (wr & (tag != lane)) | (in & (s != s));
    if (__any_sync(kFullMask, clash)) {                // ties (or NaNs): insertion-order tie-break, as the reference's stable sort
        r = 0;
        for (int q = 0; q < M; ++q) {
            const double o = lds_f64(cand_a + q * 8);
            r += (o > s) || (o == s && q < lane);
        }
        if (in && r < keep) {
            sts_f64(sn_a + r * 8, s);
            if (bp16_a) sts_u16(bp16_a + r * 2, bpe16);
            else bp_t[r] = bpe32;
        }
        __syncwarp();
    }
    return keep;
}

// After the last frame: back-track beams[0] (lane i walks beam i for the debug export), CTC-collapse it (`prev` follows
// every frame, blank included: beam_search.py:33-40) and write the token list.  Back-pointers: 16-bit (parent << 10 |
// token) in shared memory (bp16) or 32-bit (parent << 24 | token) entries (bp); sc = scores of the surviving beams.
__device__ __forceinline__ void beam_finish(const BeamParams& p, const int n, const int k, const int frames, const int nb,
                                            const uint32_t* bp, const uint16_t* bp16, const int bp_is16, const double* sc,
                                            int32_t* path, const int lane) {
    if (frames > 0) {
        const bool dbg = (p.dbg_paths != nullptr);
        if (lane == 0 || (dbg && lane < nb)) {
            int32_t* dst = dbg ? p.dbg_paths + ((size_t)n * k + lane) * p.T : path;
            int idx = lane;
            for (int t = frames - 1; t >= 0; --t) {
                if (bp_is16) {
                    const unsigned e = bp16[(size_t)t * k + idx];
                    dst[t] = (int32_t)(e & 0x3ffu);
                    idx = (int)(e >> 10);
                } else {
                    const uint32_t e = bp[(size_t)t * k + idx];
                    dst[t] = (int32_t)(e & 0xffffffu);
                    idx = (int)(e >> 24);
                }
            }
            if (dbg && lane == 0)
                for (int t = 0; t < frames; ++t) path[t] = dst[t];
        }
        if (p.dbg_scores && lane < nb) p.dbg_scores[(size_t)n * k + lane] = sc[lane];
    }
    __syncwarp();
    __threadfence_block();
    int count = 0;
    int32_t* out = p.out_ids + (size_t)n * p.T;
    for (int t0 = 0; t0 < frames; t0 += 32) {
        const int t = t0 + lane;
        bool keepit = false;
        int c = 0;
        if (t < frames) {
            c = path[t];
            keepit = (c != p.blank) && (t == 0 || path[t - 1] != c);
        }
        const unsigned m = __ballot_sync(kFullMask, keepit);
        if (keepit) out[count + __popc(m & ((1u << lane) - 1))] = c;
        count += __popc(m);
    }
    if (lane == 0) p.out_len[n] = count;
}

__global__ void __launch_bounds__(32) beam_search_kernel(const BeamParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = blockIdx.x, lane = threadIdx.x;
    const int k = p.beam;
    // ---- shared memory carve-up
    float* rows = reinterpret_cast<float*>(smem_raw);                       // kRowBufs * row_floats
    double* score = reinterpret_cast<double*>(rows + kRowBufs * p.row_floats);  // 2 * kBeamMax
    double* cand_s = score + 2 * kBeamMax;                                  // n_enum
    float* cv = reinterpret_cast<float*>(cand_s + p.n_enum);               // kCandMax
    int* ci = reinterpret_cast<int*>(cv + kCandMax);                        // kCandMax
    float* tv = reinterpret_cast<float*>(ci + kCandMax);                    // kBeamMax + 1
    int* ti = reinterpret_cast<int*>(tv + kBeamMax + 1);                    // kBeamMax + 1
    unsigned char* en_b = reinterpret_cast<unsigned char*>(ti + kBeamMax + 1);  // n_enum
    unsigned char* en_j = en_b + p.n_enum;                                  // n_enum
    int* qi = reinterpret_cast<int*>((reinterpret_cast<uintptr_t>(en_j + p.n_enum) + 15) & ~(uintptr_t)15);
    uint32_t* bp_s = reinterpret_cast<uint32_t*>(qi + (p.use_nth ? p.row_floats : 0));

    long long fl = p.lengths ? p.lengths[n] : p.T;
    const int frames = (int)(fl < 0 ? 0 : (fl > p.T ? p.T : fl));
    uint32_t* bp = p.bp_global ? p.bp_global + (size_t)n * p.T * k : bp_s;
    int32_t* path = p.path_ws + (size_t)n * p.T;
    const float* base = p.lp + (int64_t)n * p.stride_n;

    // candidate enumeration in insertion order (beam-major, k-minor); (b+1)(j+1) <= beam
    if (lane == 0) {
        int m = 0;
        for (int b = 0; b < k; ++b)
            for (int j = 0; j < k; ++j)
                if ((b + 1) * (j + 1) <= k) { en_b[m] = (unsigned char)b; en_j[m] = (unsigned char)j; ++m; }
        score[0] = 0.0;
    }
    int nb = 1, cur = 0;
    int o_in[kRowBufs];
#pragma unroll
    for (int i = 0; i < kRowBufs; ++i) o_in[i] = 0;
#pragma unroll
    for (int i = 0; i < kRowBufs - 1; ++i) {
        if (i < frames) o_in[i] = stage_row(base + (int64_t)i * p.stride_t, p.V, rows + i * p.row_floats, lane);
        else cp_async_commit();
    }
    __syncwarp();

    for (int t = 0; t < frames; ++t) {
        // prefetch frame t + kRowBufs - 1 into the buffer frame t-1 just vacated
        {
            const int tn = t + kRowBufs - 1;
            const int bi = tn % kRowBufs;
            int o = 0;
            if (tn < frames) o = stage_row(base + (int64_t)tn * p.stride_t, p.V, rows + bi * p.row_floats, lane);
            else cp_async_commit();
#pragma unroll
            for (int i = 0; i < kRowBufs; ++i) if (i == bi) o_in[i] = o;
        }
        cp_async_wait<kRowBufs - 1>();
        __syncwarp();
        int ob = 0;
#pragma unroll
        for (int i = 0; i < kRowBufs; ++i) if (i == t % kRowBufs) ob = o_in[i];
        float* row = rows + (t % kRowBufs) * p.row_floats + ob;

        bool ok = false;
        if (p.fast) ok = topk_fast(row, p.V, k, cv, ci, tv, ti, lane);
        if (!ok) {
            if (p.use_nth) topk_nth_exact(row, qi, p.V, k, tv, ti, lane);
            else topk_exact(row, p.V, k, tv, ti, lane);
        }
        // ---- expand + prune
        int M = 0;  // candidates: prefix of the enumeration with b < nb
        for (int m0 = 0; m0 < p.n_enum; m0 += 32) {
            const int m = m0 + lane;
            const bool in = (m < p.n_enum) && (en_b[m] < nb);
            M += __popc(__ballot_sync(kFullMask, in));
        }
        // enumeration is beam-major, so the b < nb entries are exactly the first M
        const double* sc = score + cur * kBeamMax;
        double* sn = score + (cur ^ 1) * kBeamMax;
        for (int m = lane; m < M; m += 32) cand_s[m] = sc[en_b[m]] + (double)tv[en_j[m]];
        __syncwarp();
        const int keep = min(k, M);
        for (int m = lane; m < M; m += 32) {
            const double s = cand_s[m];
            int r = 0;
            for (int q = 0; q < M; ++q) {
                const double o = cand_s[q];
                r += (o > s) || (o == s && q < m);
            }
            if (r < keep) {
                sn[r] = s;
                bp[(size_t)t * k + r] = ((uint32_t)en_b[m] << 24) | (uint32_t)ti[en_j[m]];
            }
        }
        __syncwarp();
        cur ^= 1;
        nb = keep;
    }
    cp_async_wait<0>();

    beam_finish(p, n, k, frames, nb, bp, nullptr, 0, score + cur * kBeamMax, path, lane);
}

// ------------------------------------------------------------------------------------------------
// Two-phase decode (default): the per-frame torch.topk does not depend on the beam state, so it runs for ALL
// N*T rows at once, HBM-bound (phase 1: one warp per row, the row lives in registers); the beam recurrence then
// only touches the [N,T,beam] top-k lists (phase 2: one warp per utterance, fp64 scores, back-pointers).
// Algorithmic traffic: one read of log_probs (T*V*4 bytes per utterance).
constexpr int kTopkWarps = 8;

__device__ __forceinline__ unsigned f2key(float v) {       // order-preserving float -> uint (no NaNs here)
    const unsigned b = __float_as_uint(v);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__host__ __device__ inline size_t topk_smem_per_warp(int row_floats, int use_nth) {
    const size_t b = (size_t)kCandPad * 8 + (size_t)(kBeamMax + 1) * 8 + (size_t)row_floats * 4 * (use_nth ? 2 : 1);
    return (b + 15) / 16 * 16;
}

__device__ __forceinline__ float fmax_nan(float a, float b) {      // NaN-propagating maximum (FMNMX.NAN)
    float d;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
    return d;
}

// MODE 0: V == 32*NV (no bounds predicates at all), MODE 1: only slot NV-1 is ragged, MODE 2: any V <= 32*NV.
// Per row (fast route, ~350 warp instructions): NV coalesced loads; the lane maxima with NaN propagation; a lower
// bound tau of the (k+1)-th largest element from k+1 rounds of redux.max over the lane maxima (equal maxima retire
// together, which only lowers tau); a per-lane bitmask of the elements >= tau, compacted into shared memory through
// a prefix sum of the lane counts (no per-slot votes or branches); ranks by counting greater candidates with 16-byte
// shared loads.  Any tie inside the first k+1 ranks, a NaN, or a candidate list outside [k+1, kCandMax] sends the row
// to the literal libstdc++ order of torch.topk (topk_exact / topk_nth_exact).
// One row of torch.topk for the warp.  row = first class of the row + lane; pf = this lane's 128-byte line of the warp's
// NEXT row (L2 prefetch) or nullptr.  On return (tv, ti)[0..k) in the warp's shared scratch hold the result, visible to
// every lane.
template <int NV, int MODE>
__device__ __forceinline__ void topk_row(const BeamParams& p, const float* __restrict__ row, const float* pf,
                                         const bool can_fast, const int k, const int lane, float* cv, float* tv, int* ti,
                                         float* srow, int* qi, int* slow_lock = nullptr) {
    const int full_slots = (MODE == 0) ? NV : (MODE == 1) ? NV - 1 : p.V / 32;
    const bool tail_ok = lane + 32 * (NV - 1) < p.V;           // MODE 1: the one ragged slot
    auto valid = [&](int j) -> bool {
        if (MODE == 0) return true;
        if (MODE == 1) return j < NV - 1 || tail_ok;
        return j < full_slots || lane + 32 * j < p.V;
    };
    float x[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) x[j] = valid(j) ? __ldcs(row + 32 * j) : AVCTC_NEG_INF;
    if (pf) asm volatile("prefetch.global.L2 [%0];" ::"l"(pf));
    float ml = x[0];
#pragma unroll
    for (int j = 1; j < NV; ++j) ml = fmax_nan(ml, x[j]);
    bool ok = can_fast && !__any_sync(kFullMask, ml != ml);
    if (ok) {
        unsigned key = f2key(ml), m = 0;
        for (int i = 0; i <= k; ++i) {
            m = __reduce_max_sync(kFullMask, key);
            if (key == m) key = 0u;
        }
        const float tau = __uint_as_float((m & 0x80000000u) ? (m & 0x7fffffffu) : ~m);   // inverse of f2key (m = 0 -> NaN)
        int c = 0, c1 = 0;
#pragma unroll
        for (int j = 0; j < NV; ++j) {      // FSETP + predicated IADD per slot, two chains (set.ge.u32 would be FSETP + SEL + IADD)
            if (valid(j)) {
                if (j & 1) asm("{\n\t.reg .pred p;\n\tsetp.ge.f32 p, %1, %2;\n\t@p add.s32 %0, %0, 1;\n\t}" : "+r"(c1) : "f"(x[j]), "f"(tau));
                else asm("{\n\t.reg .pred p;\n\tsetp.ge.f32 p, %1, %2;\n\t@p add.s32 %0, %0, 1;\n\t}" : "+r"(c) : "f"(x[j]), "f"(tau));
            }
        }
        c += c1;
        int inc = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int up = __shfl_up_sync(kFullMask, inc, d);
            if (lane >= d) inc += up;
        }
        const int count = __shfl_sync(kFullMask, inc, 31);
        ok = (count <= kCandMax) && (count >= k + 1);
        if (ok) {
            float2* cand = reinterpret_cast<float2*>(cv);          // (value, index bits) pairs, dense
            uint32_t dst = (uint32_t)__cvta_generic_to_shared(cand + (inc - c));
#pragma unroll
            for (int j = 0; j < NV; ++j) {      // 4 instructions per slot: setp, index, predicated 8-byte store + bump
                if (valid(j))
                    asm volatile("{\n\t.reg .pred p;\n\t"
                                 "setp.ge.f32 p, %1, %2;\n\t"
                                 "@p st.shared.v2.b32 [%0], {%4, %3};\n\t"
                                 "@p add.u32 %0, %0, 8;\n\t}"
                                 : "+r"(dst) : "f"(x[j]), "f"(tau), "r"(lane + 32 * j), "r"(__float_as_uint(x[j])) : "memory");
            }
            // pad: one candidate per lane when count <= 32 (slots [count, 32) = -inf), else the last 16-byte group
            if (count <= 32) { if (lane >= count) cand[lane] = make_float2(AVCTC_NEG_INF, 0.f); }
            else if (lane == 0) cand[count] = make_float2(AVCTC_NEG_INF, 0.f);
            __syncwarp();
            bool tie = false;
            if (count <= 32) {
                // one candidate per lane: rank = number of greater values, counted over the 32 slots in two unrolled halves
                // (eight 16-byte loads in flight, four chains of FSETP + predicated IADD); equal values collide on the rank
                const float2 me = cand[lane];
                const float4* c4 = reinterpret_cast<const float4*>(cand);
                int gt = 0;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    if (h == 0 || count > 16) {
                        int ga = 0, gb = 0, gc = 0, gd = 0;
                        float4 o[8];
#pragma unroll
                        for (int q = 0; q < 8; ++q) o[q] = c4[8 * h + q];
#pragma unroll
                        for (int q = 0; q < 8; q += 2) {
                            asm("{\n\t.reg .pred p;\n\tsetp.gt.f32 p, %1, %2;\n\t@p add.s32 %0, %0, 1;\n\t}" : "+r"(ga) : "f"(o[q].x), "f"(me.x));
                            asm("{\n\t.reg .pred p;\n\tsetp.gt.f32 p, %1, %2;\n\t@p add.s32 %0, %0, 1;\n\t}" : "+r"(gb) : "f"(o[q].z), "f"(me.x));
                            asm("{\n\t.reg .pred p;\n\tsetp.gt.f32 p, %1, %2;\n\t@p add.s32 %0, %0, 1;\n\t}" : "+r"(gc) : "f"(o[q + 1].x), "f"(me.x));
                            asm("{\n\t.reg .pred p;\n\tsetp.gt.f32 p, %1, %2;\n\t@p add.s32 %0, %0, 1;\n\t}" : "+r"(gd) : "f"(o[q + 1].z), "f"(me.x));
                        }
                        gt += (ga + gb) + (gc + gd);
                    }
                }
                // equal values collide on the rank: both store to slot gt, and the one whose (unique) class index did not
                // survive sees it (a match.any on the ranks is several hundred cycles of latency)
                const bool top = (lane < count) && gt <= k;
                if (top) { tv[gt] = me.x; ti[gt] = __float_as_int(me.y); }
                __syncwarp();
                tie = top && ti[gt] != __float_as_int(me.y);
            } else {
                for (int i = lane; i < count; i += 32) {
                    const float2 me = cand[i];
                    int gt = 0, eq = 0;
                    for (int j = 0; j < count; j += 2) {
                        const float4 o = *reinterpret_cast<const float4*>(cand + j);
                        gt += (o.x > me.x) + (o.z > me.x);
                        eq += (o.x == me.x) + (o.z == me.x);
                    }
                    if (gt <= k) { tv[gt] = me.x; ti[gt] = __float_as_int(me.y); tie = tie || (eq > 1); }
                }
            }
            ok = !__any_sync(kFullMask, tie);      // the first k+1 ranks hold distinct values: any algorithm agrees
        }
    }
    if (!ok) {     // ties / NaNs: literal libstdc++ order on a staged copy of the row
        __syncwarp();
        if (slow_lock) {        // the staging buffer is shared by the CTA's top-k warps (fused kernel): one row at a time
            if (lane == 0)
                while (atomicCAS(slow_lock, 0, 1) != 0) __nanosleep(200);
            __syncwarp();
        }
#pragma unroll
        for (int j = 0; j < NV; ++j) { const int c = lane + 32 * j; if (c < p.V) srow[c] = x[j]; }
        __syncwarp();
        if (p.use_nth) topk_nth_exact(srow, qi, p.V, k, tv, ti, lane);
        else topk_exact(srow, p.V, k, tv, ti, lane);
        if (slow_lock) {
            __syncwarp();
            if (lane == 0) { __threadfence_block(); atomicExch(slow_lock, 0); }
        }
    }
    __syncwarp();
}

template <int NV, int MODE>
__global__ void __launch_bounds__(kTopkWarps * 32) beam_topk_kernel(const BeamParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int k = p.beam;
    // per-warp scratch: candidates (+4 floats of padding), sorted top-(k+1), and (slow path only) a staged row + queue
    const size_t per_warp = topk_smem_per_warp(p.row_floats, p.use_nth);        // multiple of 16 bytes
    unsigned char* mine = smem_raw + (size_t)warp * per_warp;
    float* cv = reinterpret_cast<float*>(mine);                                 // 16-byte aligned (float4 rank loop)
    int* ci = reinterpret_cast<int*>(cv + kCandPad);
    float* tv = reinterpret_cast<float*>(ci + kCandPad);
    int* ti = reinterpret_cast<int*>(tv + kBeamMax + 1);
    float* srow = reinterpret_cast<float*>(ti + kBeamMax + 1);
    int* qi = reinterpret_cast<int*>(srow + p.row_floats);
    const unsigned rows = (unsigned)p.N * (unsigned)p.T;       // host guarantees N*T < 2^31
    const unsigned uT = (unsigned)p.T;
    const bool can_fast = p.fast && (k + 1 <= 32) && (p.V >= k + 1);
    for (unsigned r = blockIdx.x * kTopkWarps + warp; r < rows; r += gridDim.x * kTopkWarps) {
        if (p.lengths) {
            const unsigned n = r / uT, t = r - n * uT;
            const long long fl = p.lengths[n];
            if ((long long)t >= fl) continue;
        }
        const float* row;
        const bool dense = p.stride_n == (int64_t)uT * p.stride_t;
        if (dense) row = p.lp + (int64_t)r * p.stride_t + lane;     // dense [N,T,V]
        else { const unsigned n = r / uT, t = r - n * uT; row = p.lp + (int64_t)n * p.stride_n + (int64_t)t * p.stride_t + lane; }
        const float* pf = nullptr;
        if (p.prefetch && dense) {       // the warp's next row: one 128-byte line per lane into L2
            const unsigned rn = r + gridDim.x * kTopkWarps;
            if (rn < rows && lane * 32 < p.V) pf = p.lp + (int64_t)rn * p.stride_t + lane * 32;
        }
        topk_row<NV, MODE>(p, row, pf, can_fast, k, lane, cv, tv, ti, srow, qi);
        if (lane < k) {
            p.tk_val[(size_t)r * k + lane] = tv[lane];
            p.tk_idx[(size_t)r * k + lane] = ti[lane];
        }
        __syncwarp();
    }
}

// phase 2: beam recurrence over the top-k lists; one warp per utterance, kRecurWarps utterances per CTA
constexpr int kRecurWarps = 4;

__global__ void __launch_bounds__(kRecurWarps * 32) beam_recur_kernel(const BeamParams p, const int per_warp_bytes,
                                                                      const int bp_in_smem) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = blockIdx.x * kRecurWarps + warp;
    if (n >= p.N) return;
    const int k = p.beam;
    unsigned char* mine = smem_raw + (size_t)warp * per_warp_bytes;
    double* score = reinterpret_cast<double*>(mine);                        // 2 * kBeamMax
    double* cand_s = score + 2 * kBeamMax;                                  // max(n_enum, 32), 16-byte aligned
    unsigned char* en_b = reinterpret_cast<unsigned char*>(cand_s + (p.n_enum > 32 ? p.n_enum : 32));
    unsigned char* en_j = en_b + p.n_enum;
    uint32_t* bp_s = reinterpret_cast<uint32_t*>((reinterpret_cast<uintptr_t>(en_j + p.n_enum) + 15) & ~(uintptr_t)15);

    long long fl = p.lengths ? p.lengths[n] : p.T;
    const int frames = (int)(fl < 0 ? 0 : (fl > p.T ? p.T : fl));
    // back-pointers: in shared memory as 16-bit (parent << 10 | token; the two-phase path has V <= 1024, beam <= 32),
    // which doubles the resident warps per SM of this latency-bound kernel; the global spill keeps 32-bit entries
    uint32_t* bp = bp_in_smem ? bp_s : p.bp_global + (size_t)n * p.T * k;
    uint16_t* bp16 = reinterpret_cast<uint16_t*>(bp_s);
    int32_t* path = p.path_ws + (size_t)n * p.T;
    if (lane == 0) {
        int m = 0;
        for (int b = 0; b < k; ++b)
            for (int j = 0; j < k; ++j)
                if ((b + 1) * (j + 1) <= k) { en_b[m] = (unsigned char)b; en_j[m] = (unsigned char)j; ++m; }
        score[0] = 0.0;
    }
    __syncwarp();
    int nb = 1, cur = 0;
    const bool fast_enum = p.n_enum <= 32;
    const int my_b = (lane < p.n_enum) ? en_b[lane] : 0, my_j = (lane < p.n_enum) ? en_j[lane] : 0;
    const float* tvp = p.tk_val + (size_t)n * p.T * k;
    const int32_t* tip = p.tk_idx + (size_t)n * p.T * k;
    float tv_n = 0.f; int ti_n = 0;
    if (frames > 0 && lane < k) { tv_n = tvp[lane]; ti_n = tip[lane]; }
    const float* tv_nx = tvp + lane;           // running pointers: the next frame's list / this frame's back-pointer row
    const int32_t* ti_nx = tip + lane;
    uint32_t* bp_t = bp;
    uint16_t* bp16_t = bp16;
    const uint32_t score_a = smem_addr(score), cand_a = smem_addr(cand_s), bp16_a = smem_addr(bp16);
    for (int t = 0; t < frames; ++t, bp_t += k, bp16_t += k) {
        const float tvv = tv_n; const int tii = ti_n;
        tv_nx += k; ti_nx += k;
        if (t + 1 < frames && lane < k) { tv_n = *tv_nx; ti_n = *ti_nx; }
        if (fast_enum) {
            nb = recur_step_enum32(tvv, tii, my_b, my_j, p.n_enum, nb, k, score_a + cur * (kBeamMax * 8),
                                   score_a + (cur ^ 1) * (kBeamMax * 8), cand_a, bp_in_smem ? bp16_a + t * k * 2 : 0u, bp_t, lane);
            cur ^= 1;
            continue;
        }
        int M = 0;
        for (int m0 = 0; m0 < p.n_enum; m0 += 32) {
            const int m = m0 + lane;
            const bool in = (m < p.n_enum) && (en_b[m] < nb);
            M += __popc(__ballot_sync(kFullMask, in));
        }
        const double* sc = score + cur * kBeamMax;
        double* sn = score + (cur ^ 1) * kBeamMax;
        for (int m0 = 0; m0 < M; m0 += 32) {
            const int m = m0 + lane;
            const int jj = (m < M) ? en_j[m] : 0;
            const float lpv = __shfl_sync(kFullMask, tvv, jj);
            if (m < M) cand_s[m] = sc[en_b[m]] + (double)lpv;
        }
        __syncwarp();
        const int keep = min(k, M);
        for (int m0 = 0; m0 < M; m0 += 32) {
            const int m = m0 + lane;
            const int jj = (m < M) ? en_j[m] : 0;
            const int tok = __shfl_sync(kFullMask, tii, jj);
            if (m < M) {
                const double s = cand_s[m];
                int r = 0;
                for (int q = 0; q < M; ++q) {
                    const double o = cand_s[q];
                    r += (o > s) || (o == s && q < m);
                }
                if (r < keep) {
                    sn[r] = s;
                    if (bp_in_smem) bp16_t[r] = (uint16_t)(((int)en_b[m] << 10) | tok);
                    else bp_t[r] = ((uint32_t)en_b[m] << 24) | (uint32_t)tok;
                }
            }
        }
        __syncwarp();
        cur ^= 1;
        nb = keep;
    }
    beam_finish(p, n, k, frames, nb, bp, bp16, bp_in_smem, score + cur * kBeamMax, path, lane);
}

// ------------------------------------------------------------------------------------------------
// Fused decode (large batches of short utterances): a persistent CTA owns WHOLE utterances.  TW top-k warps take the
// rows of the CTA's current utterance (warp w: frames w, w+TW, ...) and leave the [T,beam] lists in SHARED memory; RW
// recurrence warps (utterances alternate between them) follow frame by frame, as soon as the leading frames of their
// utterance are complete, while the top-k warps already read the next utterance.  Against the two-phase path: the
// lists never travel through HBM (-2 x N*T*beam*8 bytes), and the latency-bound recurrence runs in the issue slots
// the HBM-bound top-k warps leave idle instead of after them.
//
// Hand-off, all in shared memory (no block-wide barrier after start-up):
//   prog[buf][w]  = (sequence << 12) | rows finished by top-k warp w for the utterance that occupies list buffer buf
//                   (written by lane 0 after __syncwarp + fence; stale values carry an older sequence number);
//   rdone[buf]    = number of sequences whose recurrence has read the last list of buffer buf (top-k warps wait for
//                   sequence i - NBUF before they overwrite it).
// Utterance i of a CTA (n = blockIdx.x + i*gridDim.x) uses buffer i % NBUF and recurrence warp i % RW.  No wait can
// deadlock: top-k warps only wait for recurrences of OLDER sequences, a recurrence only for top-k rows of its own.
__device__ __forceinline__ void fence_acq_rel_cta() { asm volatile("fence.acq_rel.cta;" ::: "memory"); }

__device__ __forceinline__ void fused_wait_ge(const int* word, int need) {
    int spins = 0;
    while (ld_volatile_shared_s32(word) < need) {
        __nanosleep(64);
        if (++spins > (1 << 24)) __trap();      // never hang the GPU on a protocol bug
    }
    fence_acq_rel_cta();
}

// leading frames of the utterance whose top-k lists are complete (warp-uniform)
template <int TW>
__device__ __forceinline__ int fused_frames_ready(const int* prog_buf, const int seq, const int lane) {
    int c = 0x7fffffff;
    if (lane < TW) {
        const int v = ld_volatile_shared_s32(prog_buf + lane);
        const int cnt = ((v >> 12) == seq) ? (v & 0xfff) : 0;
        c = lane + cnt * TW;                    // first frame of warp `lane` that is not finished
    }
    return __reduce_min_sync(kFullMask, c);
}

constexpr int kFusedCtrlBytes = 256;            // prog[NBUF][8] + rdone[NBUF] ints + the slow-path lock
constexpr int kFusedScratch = (kCandPad * 8 + (kBeamMax + 1) * 8 + 15) / 16 * 16;   // per top-k warp: candidates + sorted top-(k+1)
__host__ __device__ inline size_t fused_list_bytes(int T, int beam) { return ((size_t)T * beam * 6 + 15) / 16 * 16; }
__host__ __device__ inline size_t fused_slow_bytes(int row_floats, int use_nth) {
    return ((size_t)row_floats * 4 * (use_nth ? 2 : 1) + 15) / 16 * 16;
}
__host__ __device__ inline size_t fused_recur_bytes(int T, int beam) {
    return (2 * kBeamMax * 8 + 32 * 8 + (size_t)T * beam * 2 + 15) / 16 * 16;
}

// 8 warps per CTA, four CTAs per SM: the 64 registers per thread the top-k rows need (63) fill the register file
template <int NV, int MODE, int TW, int RW, int NBUF>
__global__ void __launch_bounds__((TW + RW) * 32, 2048 / ((TW + RW) * 32) < 4 ? 2048 / ((TW + RW) * 32) : 4)
beam_fused_kernel(const BeamParams p) {
    static_assert(TW <= 8 && (NBUF * 9 + 1) * 4 <= kFusedCtrlBytes && RW <= NBUF, "control block layout");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int k = p.beam;
    int* prog = reinterpret_cast<int*>(smem_raw);
    int* rdone = prog + NBUF * 8;
    int* slow_lock = rdone + NBUF;
    const size_t list_bytes = fused_list_bytes(p.T, k);
    float* srow = reinterpret_cast<float*>(smem_raw + kFusedCtrlBytes + (size_t)TW * kFusedScratch);   // shared slow-path row (+ queue)
    unsigned char* lists = reinterpret_cast<unsigned char*>(srow) + fused_slow_bytes(p.row_floats, p.use_nth);
    unsigned char* recur = lists + (size_t)NBUF * list_bytes;
    if (threadIdx.x < NBUF * 9 + 1) prog[threadIdx.x] = 0;
    __syncthreads();
    const int n_seq = (p.N - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;      // host: gridDim.x <= N

    if (warp < TW) {
        // ==================================================================== top-k warps
        unsigned char* mine = smem_raw + kFusedCtrlBytes + (size_t)warp * kFusedScratch;
        float* cv = reinterpret_cast<float*>(mine);
        int* ci = reinterpret_cast<int*>(cv + kCandPad);
        float* tv = reinterpret_cast<float*>(ci + kCandPad);
        int* ti = reinterpret_cast<int*>(tv + kBeamMax + 1);
        int* qi = reinterpret_cast<int*>(srow + p.row_floats);
        const bool can_fast = p.fast && (k + 1 <= 32) && (p.V >= k + 1);
        const bool pf_lane = p.prefetch && (lane * 32 < p.V);
        for (int i = 0; i < n_seq; ++i) {
            const int n = (int)blockIdx.x + i * (int)gridDim.x;
            const int buf = i % NBUF;
            const long long fl = p.lengths ? p.lengths[n] : p.T;
            const int frames = (int)(fl < 0 ? 0 : (fl > p.T ? p.T : fl));
            if (i >= NBUF) fused_wait_ge(&rdone[buf], i - NBUF + 1);
            float* lv = reinterpret_cast<float*>(lists + (size_t)buf * list_bytes);
            uint16_t* li = reinterpret_cast<uint16_t*>(lv + (size_t)p.T * k);
            const float* base = p.lp + (int64_t)n * p.stride_n;
            int done = 0;
            for (int t = warp; t < frames; t += TW) {
                const float* pf = nullptr;      // the warp's next row (same utterance, else its first row of the next one)
                if (pf_lane) {
                    if (t + TW < frames) pf = base + (int64_t)(t + TW) * p.stride_t + lane * 32;
                    else if (i + 1 < n_seq && warp < p.T) pf = base + (int64_t)gridDim.x * p.stride_n + (int64_t)warp * p.stride_t + lane * 32;
                }
                topk_row<NV, MODE>(p, base + (int64_t)t * p.stride_t + lane, pf, can_fast, k, lane, cv, tv, ti, srow, qi, slow_lock);
                if (lane < k) {
                    lv[t * k + lane] = tv[lane];
                    li[t * k + lane] = (uint16_t)ti[lane];
                }
                __syncwarp();
                ++done;
                if (lane == 0) {
                    fence_acq_rel_cta();
                    st_volatile_shared_s32(&prog[buf * 8 + warp], (i << 12) | done);
                }
            }
        }
        return;
    }

    // ======================================================================== recurrence warps
    const int rw = warp - TW;
    unsigned char* mine = recur + (size_t)rw * fused_recur_bytes(p.T, k);
    double* score = reinterpret_cast<double*>(mine);                        // 2 * kBeamMax
    double* cand_s = score + 2 * kBeamMax;                                  // 32
    uint16_t* bp16 = reinterpret_cast<uint16_t*>(cand_s + 32);              // T * beam
    const uint32_t score_a = smem_addr(score), cand_a = smem_addr(cand_s), bp16_a = smem_addr(bp16);
    int my_b = 0, my_j = 0;                    // candidate `lane` of the (b+1)(j+1) <= beam enumeration (beam-major)
    {
        int m = 0;
        for (int b = 0; b < k; ++b)
            for (int j = 0; j < k; ++j)
                if ((b + 1) * (j + 1) <= k) { if (m == lane) { my_b = b; my_j = j; } ++m; }
    }
    for (int i = rw; i < n_seq; i += RW) {
        const int n = (int)blockIdx.x + i * (int)gridDim.x;
        const int buf = i % NBUF;
        const long long fl = p.lengths ? p.lengths[n] : p.T;
        const int frames = (int)(fl < 0 ? 0 : (fl > p.T ? p.T : fl));
        const float* lv = reinterpret_cast<const float*>(lists + (size_t)buf * list_bytes);
        const uint16_t* li = reinterpret_cast<const uint16_t*>(lv + (size_t)p.T * k);
        int32_t* path = p.path_ws + (size_t)n * p.T;
        if (lane == 0) score[0] = 0.0;
        __syncwarp();
        int nb = 1, cur = 0, ready = 0;
        for (int t = 0; t < frames; ++t) {
            if (t >= ready) {
                int spins = 0;
                while ((ready = fused_frames_ready<TW>(prog + buf * 8, i, lane)) <= t) {
                    __nanosleep(160);
                    if (++spins > (1 << 24)) __trap();
                }
                fence_acq_rel_cta();
            }
            float tvv = 0.f; int tii = 0;
            if (lane < k) { tvv = lv[t * k + lane]; tii = li[t * k + lane]; }
            nb = recur_step_enum32(tvv, tii, my_b, my_j, p.n_enum, nb, k, score_a + cur * (kBeamMax * 8),
                                   score_a + (cur ^ 1) * (kBeamMax * 8), cand_a, bp16_a + t * k * 2, nullptr, lane);
            cur ^= 1;
        }
        __syncwarp();                          // every lane has read its last list entry
        if (lane == 0) {
            fence_acq_rel_cta();
            st_volatile_shared_s32(&rdone[buf], i + 1);
        }
        beam_finish(p, n, k, frames, nb, nullptr, bp16, 1, score + cur * kBeamMax, path, lane);
        __syncwarp();
    }
}

static int enum_count(int k) {
    int m = 0;
    for (int b = 0; b < k; ++b)
        for (int j = 0; j < k; ++j)
            if ((b + 1) * (j + 1) <= k) ++m;
    return m;
}

struct BeamPlan { size_t off_bp, off_path, off_status, off_tv, off_ti, total; bool bp_in_smem; size_t smem; int row_floats, n_enum, use_nth;
                  bool two_phase; size_t smem_topk, smem_recur_per_warp; bool bp_in_smem2;
                  bool fused_ok; size_t smem_fused; };

// Warp layout of the fused kernel, measured on B200 at config 5 and its shards (profiles/r02_beam_fused_ab*.txt): six
// top-k warps + two recurrence warps, two list buffers.  One recurrence warp per CTA cannot keep up with the top-k warps
// at large batches; 10- and 12-warp CTAs or 48 registers per thread (more resident warps, a few spills) are slower.
constexpr int kFusedTW = 6, kFusedRW = 2, kFusedNBuf = 2;
constexpr int kFusedMaxSmem = 75 * 1024;        // at least three CTAs per SM

static bool beam_plan(int N, int T, int V, int beam, BeamPlan* pl) {
    if (beam < 1 || beam > kBeamMax || beam > V) return false;
    pl->row_floats = (V + 8 + 3) & ~3;
    pl->n_enum = enum_count(beam);
    pl->use_nth = ((long long)beam * 64 > V) ? 1 : 0;
    size_t fixed = (size_t)kRowBufs * pl->row_floats * 4 + 2 * kBeamMax * 8 + (size_t)pl->n_enum * 8 +
                   kCandMax * 8 + (kBeamMax + 1) * 8 + 2 * (size_t)pl->n_enum + 16 +
                   (pl->use_nth ? (size_t)pl->row_floats * 4 : 0);
    const size_t bp_bytes = (size_t)(T > 0 ? T : 1) * beam * 4;
    pl->bp_in_smem = bp_bytes <= (size_t)kBpSmemBytes;
    pl->smem = fixed + (pl->bp_in_smem ? bp_bytes : 0);
    if (pl->smem > 200 * 1024) return false;
    size_t o = 0;
    pl->off_status = o; o += 256;
    pl->off_path = o; o = (o + (size_t)N * (T > 0 ? T : 1) * 4 + 255) / 256 * 256;
    // two-phase path: rows of up to 1024 classes live in registers (32 per lane)
    pl->two_phase = (V <= 1024) && (avctc_tuning_get("beam_two_phase", 1) != 0);
    pl->smem_topk = (size_t)kTopkWarps * topk_smem_per_warp(pl->row_floats, pl->use_nth);
    const size_t recur_fixed = 2 * kBeamMax * 8 + (size_t)(pl->n_enum > 32 ? pl->n_enum : 32) * 8 + 2 * (size_t)pl->n_enum + 16;
    const size_t bp16_bytes = bp_bytes / 2;              // two-phase recurrence: 16-bit entries in shared memory
    pl->bp_in_smem2 = bp16_bytes <= (size_t)kBpSmemBytes / 2;
    pl->smem_recur_per_warp = (recur_fixed + (pl->bp_in_smem2 ? bp16_bytes : 0) + 15) / 16 * 16;
    const bool need_bp_global = pl->two_phase ? !pl->bp_in_smem2 : !pl->bp_in_smem;
    pl->off_bp = o; if (need_bp_global) o = (o + (size_t)N * bp_bytes + 255) / 256 * 256;
    pl->off_tv = o; if (pl->two_phase) o = (o + (size_t)N * (T > 0 ? T : 1) * beam * 4 + 255) / 256 * 256;
    pl->off_ti = o; if (pl->two_phase) o = (o + (size_t)N * (T > 0 ? T : 1) * beam * 4 + 255) / 256 * 256;
    pl->total = o;
    // fused path: vocabularies of 17..26 register slots per lane (513..832 classes), one-warp candidate lists, lists of
    // NBUF utterances + the top-k scratch in shared memory (short utterances)
    pl->smem_fused = kFusedCtrlBytes + (size_t)kFusedTW * kFusedScratch + fused_slow_bytes(pl->row_floats, pl->use_nth) +
                     (size_t)kFusedNBuf * fused_list_bytes(T, beam) + (size_t)kFusedRW * fused_recur_bytes(T, beam);
    const int need = (V + 31) / 32;
    pl->fused_ok = pl->two_phase && pl->n_enum <= 32 && need >= 17 && need <= 26 && T >= 1 && T <= 4095 &&
                   pl->smem_fused <= (size_t)kFusedMaxSmem;
    return true;
}

template <int NV, int MODE>
static int launch_fused(const BeamParams& bp, size_t smem, int sms, cudaStream_t st) {
    auto kern = beam_fused_kernel<NV, MODE, kFusedTW, kFusedRW, kFusedNBuf>;
    constexpr int threads = (kFusedTW + kFusedRW) * 32;
    static size_t configured = 0;
    if (smem > configured) {
        AVCTC_CUDA_RETURN(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kFusedMaxSmem));
        configured = kFusedMaxSmem;
    }
    int occ = 0;
    AVCTC_CUDA_RETURN(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem));
    if (occ < 1) return AVCTC_ERR_UNSUPPORTED;
    long long grid = (long long)sms * occ;
    const int cap = avctc_tuning_get("beam_fused_grid", 0);      // tests: few CTAs, many utterances per CTA
    if (cap > 0 && cap < grid) grid = cap;
    if (grid > bp.N) grid = bp.N;
    kern<<<(unsigned)grid, threads, smem, st>>>(bp);
    return (int)cudaGetLastError();
}

// "beam_fused" = 1 whenever eligible, 0 never, -1 (default) up to four utterances per resident CTA.  Measured
// (profiles/r02_beam_fused_ab.txt): both routes are instruction-issue bound; the fused kernel hides the recurrence's
// latency and saves a launch and the HBM round trip of the lists (1.2x at 1024 utterances, 1.25x at 512), but its
// hand-off polling costs 13 % more instructions once every SM is saturated anyway (0.88x at 4096).
static bool beam_use_fused(const BeamPlan& pl, int N, int sms) {
    const int knob = avctc_tuning_get("beam_fused", -1);
    return pl.fused_ok && (knob > 0 || (knob < 0 && N <= 16 * sms));
}

static int beam_sm_count() {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
        (void)cudaGetLastError();       // no device (host-side planning, tests): plan for a B200
        sms = 148;
    }
    return sms;
}

// beam_topk_kernel over all N*T rows (V <= 1024, N*T < 2^31): bp.beam entries per row into bp.tk_val / bp.tk_idx
static int topk_launch(const BeamParams& bp, size_t smem_topk, int sms, cudaStream_t st) {
    const int V = bp.V;
    const int need = (V + 31) / 32;
    long long blocks = ((long long)bp.N * bp.T + kTopkWarps - 1) / kTopkWarps;
    if (blocks > (long long)sms * 8) blocks = (long long)sms * 8;
    if (blocks < 1) blocks = 1;
#define AVCTC_TOPK(NV, MODE)                                                                                        \
    do {                                                                                                            \
        static bool cfg = false;                                                                                    \
        if (!cfg && smem_topk > 48 * 1024) {                                                                        \
            AVCTC_CUDA_RETURN(cudaFuncSetAttribute(beam_topk_kernel<NV, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                                   200 * 1024));                                                    \
            cfg = true;                                                                                             \
        }                                                                                                           \
        beam_topk_kernel<NV, MODE><<<(unsigned)blocks, kTopkWarps * 32, smem_topk, st>>>(bp);                       \
    } while (0)
#define AVCTC_TOPK_M(NV)                                                                                            \
    do {                                                                                                            \
        if (V == 32 * NV) AVCTC_TOPK(NV, 0);                                                                        \
        else if (V > 32 * (NV - 1)) AVCTC_TOPK(NV, 1);                                                              \
        else AVCTC_TOPK(NV, 2);                                                                                     \
    } while (0)
    if (need <= 4) AVCTC_TOPK(4, 2);
    else if (need <= 8) AVCTC_TOPK(8, 2);
    else if (need <= 16) AVCTC_TOPK(16, 2);
    else if (need <= 25) AVCTC_TOPK_M(25);
    else if (need <= 26) AVCTC_TOPK_M(26);
    else AVCTC_TOPK_M(32);
#undef AVCTC_TOPK_M
#undef AVCTC_TOPK
    return (int)cudaGetLastError();
}

}  // namespace avctc

using namespace avctc;

int avctc_beam_topk_lists(const float* log_probs, int64_t stride_n, int64_t stride_t, int N, int T, int V,
                          const int64_t* lengths, int k, float* tk_val, int32_t* tk_idx, void* stream) {
    if (N < 0 || T < 0 || V < 1 || V > 1024 || k < 1 || k + 1 > 32 || k > V) return AVCTC_ERR_UNSUPPORTED;
    if ((long long)N * T >= (1ll << 31)) return AVCTC_ERR_UNSUPPORTED;
    BeamParams bp = {};
    bp.lp = log_probs; bp.stride_n = stride_n; bp.stride_t = stride_t;
    bp.N = N; bp.T = T; bp.V = V; bp.lengths = lengths; bp.beam = k;
    bp.fast = avctc_tuning_get("beam_fast", 1);
    bp.prefetch = avctc_tuning_get("beam_pf", 1);
    bp.row_floats = (V + 8 + 3) & ~3;
    bp.use_nth = ((long long)k * 64 > V) ? 1 : 0;
    bp.tk_val = tk_val; bp.tk_idx = tk_idx;
    return topk_launch(bp, (size_t)kTopkWarps * topk_smem_per_warp(bp.row_floats, bp.use_nth), beam_sm_count(),
                       reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int avctc_beam_route(int N, int T, int V, int beam) {
    BeamPlan pl;
    if (N <= 0 || T <= 0 || V <= 0 || beam < 1 || beam > V || !beam_plan(N, T, V, beam, &pl)) return AVCTC_BEAM_ROUTE_NONE;
    if (!pl.two_phase) return AVCTC_BEAM_ROUTE_SINGLE;
    if ((long long)N * T >= (1ll << 31)) return AVCTC_BEAM_ROUTE_NONE;
    return beam_use_fused(pl, N, beam_sm_count()) ? AVCTC_BEAM_ROUTE_FUSED : AVCTC_BEAM_ROUTE_TWO_PHASE;
}

extern "C" size_t avctc_beam_workspace_bytes(int N, int T, int V, int beam) {
    BeamPlan pl;
    if (N < 0 || T < 0 || V <= 0) return 0;
    if (!beam_plan(N, T, V, beam, &pl)) return 0;
    return pl.total;
}

extern "C" int avctc_beam_search(const float* log_probs, int64_t stride_n, int64_t stride_t, int N, int T, int V,
                                 const int64_t* lengths, int beam, int blank, int32_t* out_ids,
                                 int32_t* out_len, double* dbg_scores, int32_t* dbg_paths, void* workspace,
                                 size_t workspace_bytes, void* stream) {
    if (N < 0 || T < 0 || V <= 0 || beam < 1) return AVCTC_ERR_BAD_ARG;
    if (beam > V) return AVCTC_ERR_BAD_ARG;   // torch.topk raises "selected index k out of range"
    if (N == 0) return AVCTC_OK;
    if (!out_ids || !out_len || !workspace || (T > 0 && !log_probs)) return AVCTC_ERR_BAD_ARG;
    BeamPlan pl;
    if (!beam_plan(N, T, V, beam, &pl)) return AVCTC_ERR_UNSUPPORTED;
    if (workspace_bytes < pl.total) return AVCTC_ERR_WORKSPACE;
    if (reinterpret_cast<uintptr_t>(workspace) & 255) return AVCTC_ERR_ALIGNMENT;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    char* w = reinterpret_cast<char*>(workspace);
    BeamParams bp;
    bp.lp = log_probs; bp.stride_n = stride_n; bp.stride_t = stride_t;
    bp.N = N; bp.T = T; bp.V = V; bp.lengths = lengths; bp.beam = beam; bp.blank = blank;
    bp.fast = avctc_tuning_get("beam_fast", 1);
    bp.prefetch = avctc_tuning_get("beam_pf", 1);
    bp.out_ids = out_ids; bp.out_len = out_len; bp.dbg_scores = dbg_scores; bp.dbg_paths = dbg_paths;
    bp.bp_global = pl.bp_in_smem ? nullptr : reinterpret_cast<uint32_t*>(w + pl.off_bp);
    bp.path_ws = reinterpret_cast<int32_t*>(w + pl.off_path);
    bp.status = reinterpret_cast<int*>(w + pl.off_status);
    bp.row_floats = pl.row_floats; bp.n_enum = pl.n_enum; bp.use_nth = pl.use_nth;
    bp.tk_val = nullptr; bp.tk_idx = nullptr;
    AVCTC_CUDA_RETURN(cudaMemsetAsync(bp.status, 0, sizeof(int), st));
    if (pl.two_phase && (long long)N * T >= (1ll << 31)) return AVCTC_ERR_UNSUPPORTED;
    if (pl.two_phase) {
        if (T == 0) { AVCTC_CUDA_RETURN(cudaMemsetAsync(out_len, 0, sizeof(int32_t) * N, st)); return AVCTC_OK; }
        bp.tk_val = reinterpret_cast<float*>(w + pl.off_tv);
        bp.tk_idx = reinterpret_cast<int32_t*>(w + pl.off_ti);
        bp.bp_global = pl.bp_in_smem2 ? nullptr : reinterpret_cast<uint32_t*>(w + pl.off_bp);
        const int need = (V + 31) / 32;
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (beam_use_fused(pl, N, sms)) {
            int rc;
            if (need <= 25) {
                if (V == 800) rc = launch_fused<25, 0>(bp, pl.smem_fused, sms, st);
                else if (V > 768) rc = launch_fused<25, 1>(bp, pl.smem_fused, sms, st);
                else rc = launch_fused<25, 2>(bp, pl.smem_fused, sms, st);
            } else {
                if (V == 832) rc = launch_fused<26, 0>(bp, pl.smem_fused, sms, st);
                else rc = launch_fused<26, 1>(bp, pl.smem_fused, sms, st);
            }
            return rc;
        }
        const int rc_topk = topk_launch(bp, pl.smem_topk, sms, st);
        if (rc_topk) return rc_topk;
        const size_t smem2 = pl.smem_recur_per_warp * kRecurWarps;
        static bool cfg2 = false;
        if (!cfg2 && smem2 > 48 * 1024) {
            AVCTC_CUDA_RETURN(cudaFuncSetAttribute(beam_recur_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
            cfg2 = true;
        }
        beam_recur_kernel<<<(N + kRecurWarps - 1) / kRecurWarps, kRecurWarps * 32, smem2, st>>>(
            bp, (int)pl.smem_recur_per_warp, pl.bp_in_smem2 ? 1 : 0);
        return (int)cudaGetLastError();
    }
    static size_t configured = 0;
    if (pl.smem > 48 * 1024 && pl.smem > configured) {
        AVCTC_CUDA_RETURN(cudaFuncSetAttribute(beam_search_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               200 * 1024));
        configured = 200 * 1024;
    }
    beam_search_kernel<<<N, 32, pl.smem, st>>>(bp);
    return (int)cudaGetLastError();
}
