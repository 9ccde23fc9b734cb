// ctc_prefix_beam.cu — batched CTC prefix beam search with N-best hypotheses and scores for sm_100a (DESIGN.md §4.13).
//
// The search and its tie rules are defined once in oracle/prefix_beam_oracle.py; this kernel computes the same fp64
// scores bit for bit.  Two launches:
//   1. beam_topk_kernel (beam_search.cu, through avctc_beam_topk_lists): K_t = torch.topk(lp[n,t], k), k = min(2B+1, V),
//      for every frame, into [N,T,k] lists in the workspace.
//   2. ctc_prefix_beam_kernel: one warp per utterance, kPbWarps utterances per CTA.  Lane i holds beam entry i (pb, pnb,
//      tot, last token, length, trie node).  Per frame: the parent of each entry inside the beam (by content), the stay
//      candidates (lane = source, 2-3 log_adds), the extensions (lane = entry of K_t; only the first B+1 that are not
//      blank and not already in the beam can survive the prune), then a stable rank by counting and the new beam.
// Prefixes are trie nodes (parent << 10 | token) in shared memory, or in the workspace when 1 + T*B of them do not fit.
// A prefix that left the beam and comes back gets a new node, so two nodes can hold the same prefix: identity is
// decided by content, walking both parent chains until the nodes meet (never by a hash).
// ctc_prefix_beam_lm_kernel (below) is the same recurrence with shallow fusion of a token n-gram LM (DESIGN.md §4.14)
// and / or contextual biasing towards a phrase list (§4.15).
#include <cmath>

#include "common.cuh"
#include "beam_internal.h"

namespace avctc {
namespace {

constexpr int kPbMaxBeam = 15;
constexpr int kPbWarps = 4;
constexpr int kPbCand = 256;            // candidate slots: nb * (B + 2) <= 15 * 17
constexpr int kPbSmemNodes = 4096;      // trie nodes per warp kept in shared memory (16 KB)
constexpr int kPbFixedBytes = kPbCand * 8 + kPbCand * 4 + 16 * 8 + 16 * 4 * 2;

// log_add: the fixed IEEE sequence of oracle/prefix_beam_oracle.py::log_add; every operation is an explicit
// round-to-nearest intrinsic, so nothing is contracted into an FMA and no library exp / log1p is involved.
__constant__ double kExpC[14] = {        // 1/n!
    0x1.0000000000000p+0, 0x1.0000000000000p+0, 0x1.0000000000000p-1, 0x1.5555555555555p-3, 0x1.5555555555555p-5,
    0x1.1111111111111p-7, 0x1.6c16c16c16c17p-10, 0x1.a01a01a01a01ap-13, 0x1.a01a01a01a01ap-16, 0x1.71de3a556c734p-19,
    0x1.27e4fb7789f5cp-22, 0x1.ae64567f544e4p-26, 0x1.1eed8eff8d898p-29, 0x1.6124613a86d09p-33};
__constant__ double kLogC[17] = {        // 1/(2n+1)
    0x1.0000000000000p+0, 0x1.5555555555555p-2, 0x1.999999999999ap-3, 0x1.2492492492492p-3, 0x1.c71c71c71c71cp-4,
    0x1.745d1745d1746p-4, 0x1.3b13b13b13b14p-4, 0x1.1111111111111p-4, 0x1.e1e1e1e1e1e1ep-5, 0x1.af286bca1af28p-5,
    0x1.8618618618618p-5, 0x1.642c8590b2164p-5, 0x1.47ae147ae147bp-5, 0x1.2f684bda12f68p-5, 0x1.1a7b9611a7b96p-5,
    0x1.0842108421084p-5, 0x1.f07c1f07c1f08p-6};
constexpr double kInvLn2 = 0x1.71547652b82fep+0;
constexpr double kLn2Hi = 0x1.62e42fee00000p-1;
constexpr double kLn2Lo = 0x1.a39ef35793c76p-33;
#define kNegInfD (-CUDART_INF)

__device__ __forceinline__ double log_add(double a, double b) {
    if (b > a) { const double x = a; a = b; b = x; }
    if (b == kNegInfD) return a;
    const double d = __dsub_rn(b, a);
    if (!(d >= -708.0)) return a;
    const double kd = floor(__dadd_rn(__dmul_rn(d, kInvLn2), 0.5));
    const double r = __dsub_rn(__dsub_rn(d, __dmul_rn(kd, kLn2Hi)), __dmul_rn(kd, kLn2Lo));
    double p = kExpC[13];
#pragma unroll
    for (int i = 12; i >= 0; --i) p = __dadd_rn(__dmul_rn(p, r), kExpC[i]);
    const double e = __dmul_rn(p, __longlong_as_double((long long)((int)kd + 1023) << 52));   // exact: 2^k is normal
    const double s = __ddiv_rn(e, __dadd_rn(2.0, e));
    const double z = __dmul_rn(s, s);
    double q = kLogC[16];
#pragma unroll
    for (int i = 15; i >= 0; --i) q = __dadd_rn(__dmul_rn(q, z), kLogC[i]);
    return __dadd_rn(a, __dmul_rn(__dmul_rn(s, q), 2.0));
}

// Two nodes of equal depth hold the same prefix iff their chains agree token by token until they meet.
__device__ __forceinline__ bool same_prefix(const volatile uint32_t* nodes, int x, int y) {
    while (x != y) {
        const uint32_t u = nodes[x], w = nodes[y];
        if ((u ^ w) & 1023u) return false;
        x = (int)(u >> 10);
        y = (int)(w >> 10);
    }
    return true;
}

}  // namespace

struct PbParams {
    const float* lp; int64_t stride_n, stride_t;
    int N, T, V;
    const int64_t* lengths;
    int beam, nbest, blank, k;
    const float* tk_val; const int32_t* tk_idx;      // [N][T][k] from phase 1
    uint32_t* nodes_g;                                // [N][node_cap] when the trie does not fit shared memory
    int node_cap;
    int32_t* out_tokens; int32_t* out_len; double* out_scores; int32_t* status;
};

__global__ void __launch_bounds__(kPbWarps * 32) ctc_prefix_beam_kernel(const PbParams p, const int per_warp_bytes) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = blockIdx.x * kPbWarps + warp;
    if (n >= p.N) return;
    unsigned char* mine = smem_raw + (size_t)warp * per_warp_bytes;
    double* ctot = reinterpret_cast<double*>(mine);                  // candidate tot', -inf = no candidate
    int* ctok = reinterpret_cast<int*>(ctot + kPbCand);              // candidate token, -1 = stay
    double* nx_tot = reinterpret_cast<double*>(ctok + kPbCand);      // the kept candidates in rank order
    int* nx_src = reinterpret_cast<int*>(nx_tot + 16);
    int* nx_tok = nx_src + 16;
    volatile uint32_t* nodes = p.nodes_g ? p.nodes_g + (size_t)n * p.node_cap
                                         : reinterpret_cast<uint32_t*>(mine + kPbFixedBytes);
    const int B = p.beam, S = B + 2, k = p.k, blank = p.blank;
    int32_t* olen = p.out_len + (size_t)n * p.nbest;
    double* osc = p.out_scores + (size_t)n * p.nbest;
    const long long fl = p.lengths ? p.lengths[n] : p.T;
    if (fl < 0 || fl > p.T) {
        if (lane < p.nbest) { olen[lane] = 0; osc[lane] = kNegInfD; }
        if (lane == 0) p.status[n] = 2;
        return;
    }
    const int frames = (int)fl;
    const float* base = p.lp + (int64_t)n * p.stride_n;
    const float* tkv = p.tk_val + (size_t)n * p.T * k;
    const int32_t* tki = p.tk_idx + (size_t)n * p.T * k;
    const unsigned lt = (1u << lane) - 1u;

    double pb = lane == 0 ? 0.0 : kNegInfD, pnb = kNegInfD, tot = pb;
    int last = -1, len = 0, node = 0, nb = 1, next_node = 1, st = 0;
    float kv = 0.f, lpb = 0.f, lpl = 0.f;      // this frame's K_t entry (lane j), lp[t,blank], lp[t,last]
    int ki = -1;
    if (frames > 0) {
        if (lane < k) { kv = tkv[lane]; ki = tki[lane]; }
        lpb = base[blank];
    }
    for (int t = 0; t < frames; ++t) {
        const float kv_t = kv, lpb_t = lpb, lpl_t = lpl;
        const int ki_t = ki;
        if (t + 1 < frames && lane < k) { kv = tkv[(size_t)(t + 1) * k + lane]; ki = tki[(size_t)(t + 1) * k + lane]; }
        const float k0 = __shfl_sync(kFullMask, kv_t, 0);
        if (k0 != k0) { st = 1; break; }

        // parent inside the beam: the entry j with len_j = len - 1 holding this entry's prefix minus its last token
        const bool mine_live = lane < nb && len > 0;
        const int my_par = mine_live ? (int)(nodes[node] >> 10) : 0;
        int pidx = -1;
        for (int j = 0; j < nb; ++j) {
            const int lj = __shfl_sync(kFullMask, len, j), nj = __shfl_sync(kFullMask, node, j);
            if (mine_live && pidx < 0 && lj == len - 1 && same_prefix(nodes, my_par, nj)) pidx = j;
        }
        // stay candidate of source `lane`: slot lane * S
        const int ps = pidx < 0 ? 0 : pidx;
        const double p_pb = __shfl_sync(kFullMask, pb, ps), p_tot = __shfl_sync(kFullMask, tot, ps);
        const int p_last = __shfl_sync(kFullMask, last, ps);
        double spb = kNegInfD, spnb = kNegInfD;
        if (lane < nb) {
            spb = __dadd_rn(tot, (double)lpb_t);
            if (len > 0) {
                const double lc = (double)lpl_t;
                spnb = __dadd_rn(pnb, lc);
                if (pidx >= 0) spnb = log_add(spnb, __dadd_rn(last == p_last ? p_pb : p_tot, lc));
            }
            const double stot = log_add(spb, spnb);
            ctot[lane * S] = stot > kNegInfD ? stot : kNegInfD;
            ctok[lane * S] = -1;
        }
        // bit s of inbeam: source s + (K_t entry of this lane) is already in the beam
        unsigned inbeam = 0;
        for (int e = 0; e < nb; ++e) {
            const int pe = __shfl_sync(kFullMask, pidx, e), le = __shfl_sync(kFullMask, last, e);
            if (pe >= 0 && le == ki_t) inbeam |= 1u << pe;
        }
        const bool tok_ok = lane < k && ki_t != blank;
        // extensions of source s: slots s*S + 1 .. s*S + B + 1, in K_t order
        for (int s = 0; s < nb; ++s) {
            const double s_tot = __shfl_sync(kFullMask, tot, s), s_pb = __shfl_sync(kFullMask, pb, s);
            const int s_last = __shfl_sync(kFullMask, last, s);
            const bool ok = tok_ok && !((inbeam >> s) & 1u);
            const unsigned m = __ballot_sync(kFullMask, ok);
            const int r = __popc(m & lt);
            const int slot0 = s * S + 1;
            if (ok && r <= B) {
                const double e = __dadd_rn(ki_t == s_last ? s_pb : s_tot, (double)kv_t);
                ctot[slot0 + r] = e > kNegInfD ? e : kNegInfD;
                ctok[slot0 + r] = ki_t;
            }
            const int cnt = min(__popc(m), B + 1);
            if (lane >= cnt && lane <= B) ctot[slot0 + lane] = kNegInfD;
        }
        __syncwarp();
        // stable rank by counting: strictly greater scores, then equal scores at earlier slots
        const int M = nb * S;
        int valid = 0;
        for (int m = lane; m < M; m += 32) {
            const double v = ctot[m];
            if (v > kNegInfD) {
                ++valid;
                int r = 0;
                for (int q = 0; q < M && r < B; ++q) {
                    const double o = ctot[q];
                    r += (o > v) || (o == v && q < m);
                }
                if (r < B) { nx_tot[r] = v; nx_src[r] = m / S; nx_tok[r] = ctok[m]; }
            }
        }
        const int nb_new = min(B, (int)__reduce_add_sync(kFullMask, (unsigned)valid));
        __syncwarp();
        const bool live = lane < nb_new;
        const int src = live ? nx_src[lane] : 0;
        const int tok = live ? nx_tok[lane] : -1;
        const double ntot = live ? nx_tot[lane] : kNegInfD;
        const double o_spb = __shfl_sync(kFullMask, spb, src), o_spnb = __shfl_sync(kFullMask, spnb, src);
        const int o_last = __shfl_sync(kFullMask, last, src), o_len = __shfl_sync(kFullMask, len, src);
        const int o_node = __shfl_sync(kFullMask, node, src);
        const bool is_ext = live && tok >= 0;
        const unsigned em = __ballot_sync(kFullMask, is_ext);
        if (is_ext) {
            const int id = next_node + __popc(em & lt);
            nodes[id] = ((uint32_t)o_node << 10) | (uint32_t)tok;
            pb = kNegInfD; pnb = ntot; last = tok; len = o_len + 1; node = id;
        } else if (live) {
            pb = o_spb; pnb = o_spnb; last = o_last; len = o_len; node = o_node;
        } else {
            pb = kNegInfD; pnb = kNegInfD; last = -1; len = 0; node = 0;
        }
        tot = ntot;
        next_node += __popc(em);
        nb = nb_new;
        __syncwarp();
        if (t + 1 < frames) {           // the next frame's gathers go out before its top-k list is needed
            const float* row = base + (int64_t)(t + 1) * p.stride_t;
            lpb = row[blank];
            if (live && len > 0) lpl = row[last];
        }
    }
    if (lane < p.nbest) {
        const bool have = st == 0 && lane < nb;
        olen[lane] = have ? len : 0;
        osc[lane] = have ? tot : kNegInfD;
        if (have) {
            int32_t* dst = p.out_tokens + ((size_t)n * p.nbest + lane) * p.T;
            int x = node;
            for (int j = len - 1; j >= 0; --j) {
                const uint32_t u = nodes[x];
                dst[j] = (int32_t)(u & 1023u);
                x = (int)(u >> 10);
            }
        }
    }
    if (lane == 0) p.status[n] = st;
}

// ---------------------------------------------------------------------------------------------------------------
// Shallow fusion with a token n-gram LM (DESIGN.md §4.14; oracle/prefix_beam_lm_oracle.py).  The recurrence above
// with, per lane, the entry's LM history (the last order-1 LM words of <s> + prefix, 11 bits each) and LM score L.
// Candidates are ranked by key = tot' + L'.  Per source, all admissible K_t entries are scored and the source's B best
// by (key descending, K_t position ascending) are kept: B of them precede any later one in the global stable order.

constexpr int kPbLmFixedBytes = kPbCand * (8 + 8 + 8 + 4) + 16 * (8 + 8 + 4 + 4);
constexpr double kLn10 = 0x1.26bb1bbb55516p+1;
constexpr unsigned long long kLmEmpty = ~0ull;
constexpr unsigned long long kLmHashMul = 0x9E3779B97F4A7C15ull;

struct PbLm {
    const int32_t* token_word;
    const float2* unigram;                 // (log10 p, log10 bow) per word id
    const ulonglong2* tab[4];              // orders 2..5: {key, logp | bow << 32}
    unsigned long long mask[4];            // capacity - 1
    int order, bos, eos;
    double alpha, beta;
};

// Open addressing, linear probing: the n-gram `key` is present -> its (logp, bow).
__device__ __forceinline__ bool lm_probe(const ulonglong2* tab, unsigned long long mask, unsigned long long key,
                                         float* logp, float* bow) {
    unsigned long long h = key * kLmHashMul;
    h ^= h >> 29;
    for (unsigned long long i = h & mask;; i = (i + 1) & mask) {
        const ulonglong2 e = __ldg(tab + i);
        if (e.x == key) {
            *logp = __uint_as_float((unsigned)e.y);
            *bow = __uint_as_float((unsigned)(e.y >> 32));
            return true;
        }
        if (e.x == kLmEmpty) return false;
    }
}

// log10 P(w | the hlen <= order-1 words packed in hist), the back-off walk of §4.14 summed in its order.
__device__ __forceinline__ double lm10(const PbLm& lm, unsigned long long hist, int hlen, int w) {
    double acc = 0.0;
#pragma unroll
    for (int m = 4; m >= 1; --m) {       // static table indices; m > hlen is skipped
        if (m > hlen) continue;
        const unsigned long long ctx = hist & ((1ull << (11 * m)) - 1ull);
        float lp, bw = 0.f;
        if (lm_probe(lm.tab[m - 1], lm.mask[m - 1], (ctx << 11) | (unsigned)w, &lp, &bw)) return __dadd_rn(acc, (double)lp);
        bw = 0.f;
        if (m == 1) bw = __ldg(lm.unigram + ctx).y;
        else if (!lm_probe(lm.tab[m - 2], lm.mask[m - 2], ctx, &lp, &bw)) bw = 0.f;
        acc = __dadd_rn(acc, (double)bw);
    }
    return __dadd_rn(acc, (double)__ldg(lm.unigram + w).x);
}

// Contextual biasing (DESIGN.md §4.15; oracle/context_graph_oracle.py): each entry also carries its node u in the
// phrase automaton and an fp64 bias score G.  An extension s+c moves to v = delta(u, c) and adds
// (phi(v) - phi(u)) + omega(v); the key gains + G'.  After the last frame G - phi(u) withdraws an unfinished match.
struct PbCtx {
    const int32_t* token_sym;              // [V]: context-alphabet symbol of a token, -1 = not in any phrase
    const int32_t* delta;                  // [num_nodes][alphabet]
    const double2* node;                   // [num_nodes]: (phi, omega)
    int alphabet;
};

// Per-warp shared memory of the biased instances: kPbLmFixedBytes, then cG[kPbCand], nx_G[16], cctx[kPbCand], nx_ctx[16].
constexpr int kPbBiasFixedBytes = kPbLmFixedBytes + kPbCand * (8 + 4) + 16 * (8 + 4);

// kLm: n-gram fusion (§4.14); kBias: contextual biasing (§4.15).  <true, false> is the LM search of §4.14; its
// parameters come first so that the instance compiles to the same code as before the biasing was added.
template <bool kLm, bool kBias>
__global__ void __launch_bounds__(kPbWarps * 32) ctc_prefix_beam_lm_kernel(const PbParams p, const PbLm lm,
                                                                          double* out_ac, double* out_lm,
                                                                          const int per_warp_bytes, const PbCtx cx,
                                                                          double* out_bias) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = blockIdx.x * kPbWarps + warp;
    if (n >= p.N) return;
    unsigned char* mine = smem_raw + (size_t)warp * per_warp_bytes;
    double* ckey = reinterpret_cast<double*>(mine);                  // candidate tot' + L', NaN = no candidate
    double* ctot = ckey + kPbCand;                                   // candidate tot', -inf = no candidate
    double* cL = ctot + kPbCand;                                     // candidate L'
    int* ctok = reinterpret_cast<int*>(cL + kPbCand);                // candidate token, -1 = stay
    double* nx_tot = reinterpret_cast<double*>(ctok + kPbCand);      // the kept candidates in rank order
    double* nx_L = nx_tot + 16;
    int* nx_src = reinterpret_cast<int*>(nx_L + 16);
    int* nx_tok = nx_src + 16;
    double* cG = reinterpret_cast<double*>(nx_tok + 16);             // candidate G' and context node (biasing only)
    double* nx_G = cG + kPbCand;
    int* cctx = reinterpret_cast<int*>(nx_G + 16);
    int* nx_ctx = cctx + kPbCand;
    volatile uint32_t* nodes = p.nodes_g ? p.nodes_g + (size_t)n * p.node_cap
                                         : reinterpret_cast<uint32_t*>(mine + (kBias ? kPbBiasFixedBytes : kPbLmFixedBytes));
    const int B = p.beam, S = B + 1, k = p.k, blank = p.blank;
    const size_t o0 = (size_t)n * p.nbest;
    int32_t* olen = p.out_len + o0;
    double* osc = p.out_scores + o0;
    double* oac = out_ac + o0;
    double* olm = out_lm + o0;
    double* obias = kBias ? out_bias + o0 : nullptr;
    const long long fl = p.lengths ? p.lengths[n] : p.T;
    if (fl < 0 || fl > p.T) {
        if (lane < p.nbest) {
            olen[lane] = 0; osc[lane] = kNegInfD; oac[lane] = kNegInfD; olm[lane] = kNegInfD;
            if constexpr (kBias) obias[lane] = kNegInfD;
        }
        if (lane == 0) p.status[n] = 2;
        return;
    }
    const int frames = (int)fl;
    const float* base = p.lp + (int64_t)n * p.stride_n;
    const float* tkv = p.tk_val + (size_t)n * p.T * k;
    const int32_t* tki = p.tk_idx + (size_t)n * p.T * k;
    const unsigned lt = (1u << lane) - 1u;
    const int hmax = lm.order - 1;
    const unsigned long long hmask = (1ull << (11 * hmax)) - 1ull;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);

    double pb = lane == 0 ? 0.0 : kNegInfD, pnb = kNegInfD, tot = pb, L = 0.0;
    int last = -1, len = 0, node = 0, nb = 1, next_node = 1, st = 0;
    unsigned long long hist = hmax > 0 ? (unsigned long long)lm.bos : 0ull;
    int hlen = hmax > 0 ? 1 : 0;
    double G = 0.0, phi = 0.0;                 // bias score and phi of the entry's context node ctx (root: 0)
    int ctx = 0;
    float kv = 0.f, lpb = 0.f, lpl = 0.f;      // this frame's K_t entry (lane j), lp[t,blank], lp[t,last]
    int ki = -1, kw = 0, ks = -1;              // its class, LM word and context symbol
    if (frames > 0) {
        if (lane < k) {
            kv = tkv[lane]; ki = tki[lane];
            if constexpr (kLm) kw = ki >= 0 && ki < p.V ? lm.token_word[ki] : 0;
            if constexpr (kBias) ks = ki >= 0 && ki < p.V ? __ldg(cx.token_sym + ki) : -1;
        }
        lpb = base[blank];
    }
    for (int t = 0; t < frames; ++t) {
        const float kv_t = kv, lpb_t = lpb, lpl_t = lpl;
        const int ki_t = ki, kw_t = kw, ks_t = ks;
        if (t + 1 < frames && lane < k) {
            kv = tkv[(size_t)(t + 1) * k + lane];
            ki = tki[(size_t)(t + 1) * k + lane];
            if constexpr (kLm) kw = ki >= 0 && ki < p.V ? lm.token_word[ki] : 0;
            if constexpr (kBias) ks = ki >= 0 && ki < p.V ? __ldg(cx.token_sym + ki) : -1;
        }
        const float k0 = __shfl_sync(kFullMask, kv_t, 0);
        if (k0 != k0) { st = 1; break; }

        const bool mine_live = lane < nb && len > 0;
        const int my_par = mine_live ? (int)(nodes[node] >> 10) : 0;
        int pidx = -1;
        for (int j = 0; j < nb; ++j) {
            const int lj = __shfl_sync(kFullMask, len, j), nj = __shfl_sync(kFullMask, node, j);
            if (mine_live && pidx < 0 && lj == len - 1 && same_prefix(nodes, my_par, nj)) pidx = j;
        }
        // stay candidate of source `lane`: slot lane * S, L unchanged
        const int ps = pidx < 0 ? 0 : pidx;
        const double p_pb = __shfl_sync(kFullMask, pb, ps), p_tot = __shfl_sync(kFullMask, tot, ps);
        const int p_last = __shfl_sync(kFullMask, last, ps);
        double spb = kNegInfD, spnb = kNegInfD;
        if (lane < nb) {
            spb = __dadd_rn(tot, (double)lpb_t);
            if (len > 0) {
                const double lc = (double)lpl_t;
                spnb = __dadd_rn(pnb, lc);
                if (pidx >= 0) spnb = log_add(spnb, __dadd_rn(last == p_last ? p_pb : p_tot, lc));
            }
            const double stot = log_add(spb, spnb);
            const bool ok = stot > kNegInfD;
            ctot[lane * S] = ok ? stot : kNegInfD;
            if constexpr (kBias) {
                ckey[lane * S] = ok ? __dadd_rn(kLm ? __dadd_rn(stot, L) : stot, G) : nan;
                cG[lane * S] = G;
                cctx[lane * S] = ctx;
            } else {
                ckey[lane * S] = ok ? __dadd_rn(stot, L) : nan;
            }
            if constexpr (kLm) cL[lane * S] = L;
            ctok[lane * S] = -1;
        }
        unsigned inbeam = 0;
        for (int e = 0; e < nb; ++e) {
            const int pe = __shfl_sync(kFullMask, pidx, e), le = __shfl_sync(kFullMask, last, e);
            if (pe >= 0 && le == ki_t) inbeam |= 1u << pe;
        }
        const bool tok_ok = lane < k && ki_t != blank;
        // extensions of source s: every admissible K_t entry is scored, the B best by (key, K_t position) kept in
        // slots s*S + 1 .. s*S + B
        for (int s = 0; s < nb; ++s) {
            const double s_tot = __shfl_sync(kFullMask, tot, s), s_pb = __shfl_sync(kFullMask, pb, s);
            const double s_L = kLm ? __shfl_sync(kFullMask, L, s) : 0.0;
            const unsigned long long s_hist = kLm ? __shfl_sync(kFullMask, hist, s) : 0ull;
            const int s_last = __shfl_sync(kFullMask, last, s), s_hlen = kLm ? __shfl_sync(kFullMask, hlen, s) : 0;
            const double e = __dadd_rn(ki_t == s_last ? s_pb : s_tot, (double)kv_t);
            const bool ok = tok_ok && !((inbeam >> s) & 1u) && e > kNegInfD;
            double Lc = 0.0, key = 0.0;
            if (ok) {
                if constexpr (kLm) {
                    const double d = __dadd_rn(__dmul_rn(lm.alpha, __dmul_rn(lm10(lm, s_hist, s_hlen, kw_t), kLn10)), lm.beta);
                    Lc = __dadd_rn(s_L, d);
                    key = __dadd_rn(e, Lc);
                } else {
                    key = e;
                }
            }
            double Gc = 0.0;
            int vc = 0;
            if constexpr (kBias) {
                // v = delta(u_s, c): a token outside every phrase returns to the root
                const double s_G = __shfl_sync(kFullMask, G, s), s_phi = __shfl_sync(kFullMask, phi, s);
                const int s_ctx = __shfl_sync(kFullMask, ctx, s);
                if (ok) {
                    vc = ks_t < 0 ? 0 : __ldg(cx.delta + (size_t)s_ctx * cx.alphabet + ks_t);
                    const double2 nv = __ldg(cx.node + vc);
                    Gc = __dadd_rn(s_G, __dadd_rn(__dsub_rn(nv.x, s_phi), nv.y));
                    key = __dadd_rn(key, Gc);
                }
            }
            const unsigned m = __ballot_sync(kFullMask, ok);
            int r = 0;
            for (int i = 0; i < k; ++i) {
                const double o = __shfl_sync(kFullMask, key, i);
                r += ((m >> i) & 1u) && (o > key || (o == key && i < lane));
            }
            const int slot0 = s * S + 1;
            if (ok && r < B) {
                ckey[slot0 + r] = key;
                ctot[slot0 + r] = e;
                if constexpr (kLm) cL[slot0 + r] = Lc;
                if constexpr (kBias) { cG[slot0 + r] = Gc; cctx[slot0 + r] = vc; }
                ctok[slot0 + r] = ki_t;
            }
            const int cnt = min(__popc(m), B);
            if (lane >= cnt && lane < B) { ctot[slot0 + lane] = kNegInfD; ckey[slot0 + lane] = nan; }
        }
        __syncwarp();
        // stable rank by counting: strictly greater keys, then equal keys at earlier slots (NaN never counts)
        const int M = nb * S;
        int valid = 0;
        for (int m = lane; m < M; m += 32) {
            if (ctot[m] > kNegInfD) {
                const double v = ckey[m];
                ++valid;
                int r = 0;
                for (int q = 0; q < M && r < B; ++q) {
                    const double o = ckey[q];
                    r += (o > v) || (o == v && q < m);
                }
                if (r < B) {
                    nx_tot[r] = ctot[m];
                    if constexpr (kLm) nx_L[r] = cL[m];
                    if constexpr (kBias) { nx_G[r] = cG[m]; nx_ctx[r] = cctx[m]; }
                    nx_src[r] = m / S; nx_tok[r] = ctok[m];
                }
            }
        }
        const int nb_new = min(B, (int)__reduce_add_sync(kFullMask, (unsigned)valid));
        __syncwarp();
        const bool live = lane < nb_new;
        const int src = live ? nx_src[lane] : 0;
        const int tok = live ? nx_tok[lane] : -1;
        const double ntot = live ? nx_tot[lane] : kNegInfD;
        const double nL = kLm && live ? nx_L[lane] : 0.0;
        const double o_spb = __shfl_sync(kFullMask, spb, src), o_spnb = __shfl_sync(kFullMask, spnb, src);
        const int o_last = __shfl_sync(kFullMask, last, src), o_len = __shfl_sync(kFullMask, len, src);
        const int o_node = __shfl_sync(kFullMask, node, src), o_hlen = kLm ? __shfl_sync(kFullMask, hlen, src) : 0;
        const unsigned long long o_hist = kLm ? __shfl_sync(kFullMask, hist, src) : 0ull;
        const bool is_ext = live && tok >= 0;
        const unsigned em = __ballot_sync(kFullMask, is_ext);
        if (is_ext) {
            const int id = next_node + __popc(em & lt);
            nodes[id] = ((uint32_t)o_node << 10) | (uint32_t)tok;
            pb = kNegInfD; pnb = ntot; last = tok; len = o_len + 1; node = id;
            if constexpr (kLm) {
                hist = ((o_hist << 11) | (unsigned)lm.token_word[tok]) & hmask;
                hlen = min(o_hlen + 1, hmax);
            }
        } else if (live) {
            pb = o_spb; pnb = o_spnb; last = o_last; len = o_len; node = o_node;
            hist = o_hist; hlen = o_hlen;
        } else {
            pb = kNegInfD; pnb = kNegInfD; last = -1; len = 0; node = 0;
            hist = 0ull; hlen = 0;
        }
        tot = ntot;
        L = nL;
        if constexpr (kBias) {
            G = live ? nx_G[lane] : 0.0;
            ctx = live ? nx_ctx[lane] : 0;
            phi = live ? __ldg(&cx.node[ctx].x) : 0.0;
        }
        next_node += __popc(em);
        nb = nb_new;
        __syncwarp();
        if (t + 1 < frames) {
            const float* row = base + (int64_t)(t + 1) * p.stride_t;
            lpb = row[blank];
            if (live && len > 0) lpl = row[last];
        }
    }
    // end of sentence: E = alpha * ln P(</s> | history) (0 without an LM) and bias = G - phi(u), then a stable
    // re-rank by (tot + (L + E)) + bias
    const bool have = st == 0 && lane < nb;
    double lms = kNegInfD, fin = kNegInfD, bias = kNegInfD;
    if (have) {
        if constexpr (kLm) {
            lms = __dadd_rn(L, __dmul_rn(lm.alpha, __dmul_rn(lm10(lm, hist, hlen, lm.eos), kLn10)));
            fin = __dadd_rn(tot, lms);
        } else {
            lms = 0.0;
            fin = __dadd_rn(tot, lms);
        }
        if constexpr (kBias) {
            bias = __dsub_rn(G, phi);
            fin = __dadd_rn(fin, bias);
        }
    }
    int r = 0;
    for (int j = 0; j < nb; ++j) {
        const double o = __shfl_sync(kFullMask, fin, j);
        r += (o > fin) || (o == fin && j < lane);
    }
    if (have && r < p.nbest) {
        olen[r] = len; osc[r] = fin; oac[r] = tot; olm[r] = lms;
        if constexpr (kBias) obias[r] = bias;
        int32_t* dst = p.out_tokens + (o0 + r) * p.T;
        int x = node;
        for (int j = len - 1; j >= 0; --j) {
            const uint32_t u = nodes[x];
            dst[j] = (int32_t)(u & 1023u);
            x = (int)(u >> 10);
        }
    }
    const int used = st == 0 ? min(nb, p.nbest) : 0;
    if (lane >= used && lane < p.nbest) {
        olen[lane] = 0; osc[lane] = kNegInfD; oac[lane] = kNegInfD; olm[lane] = kNegInfD;
        if constexpr (kBias) obias[lane] = kNegInfD;
    }
    if (lane == 0) p.status[n] = st;
}

namespace {

struct PbPlan { int k, node_cap; bool smem_nodes; size_t per_warp, off_tv, off_ti, off_nodes, total; };

inline size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

bool pb_plan(int N, int T, int V, int beam, PbPlan* pl) {
    if (N < 0 || T < 0 || V < 1 || V > 1024 || beam < 1 || beam > kPbMaxBeam) return false;
    if ((long long)N * T >= (1ll << 31)) return false;
    const long long cap = 1 + (long long)T * beam;           // root + at most B new prefixes per frame
    if (cap >= (1ll << 22)) return false;                    // parent field of a node: 22 bits
    pl->k = 2 * beam + 1 < V ? 2 * beam + 1 : V;
    pl->node_cap = (int)cap;
    pl->smem_nodes = cap <= kPbSmemNodes;
    pl->per_warp = round_up(kPbFixedBytes + (pl->smem_nodes ? (size_t)cap * 4 : 0), 16);
    const size_t lists = (size_t)N * T * pl->k * 4;
    size_t o = 0;
    pl->off_tv = o; o += round_up(lists, 256);
    pl->off_ti = o; o += round_up(lists, 256);
    pl->off_nodes = o; if (!pl->smem_nodes) o += round_up((size_t)N * cap * 4, 256);
    pl->total = o > 256 ? o : 256;
    return true;
}

}  // namespace
}  // namespace avctc

using namespace avctc;

extern "C" size_t avctc_ctc_prefix_beam_workspace_bytes(int N, int T, int V, int beam) {
    PbPlan pl;
    return pb_plan(N, T, V, beam, &pl) ? pl.total : 0;
}

extern "C" int avctc_ctc_prefix_beam(const float* log_probs, int64_t stride_n, int64_t stride_t, int N, int T, int V,
                                     const int64_t* lengths, int beam, int nbest, int blank, int32_t* out_tokens,
                                     int32_t* out_len, double* out_scores, int32_t* status, void* workspace,
                                     size_t workspace_bytes, void* stream) {
    if (N < 0 || T < 0 || V < 1 || beam < 1 || nbest < 1 || nbest > beam || blank < 0 || blank >= V)
        return AVCTC_ERR_BAD_ARG;
    PbPlan pl;
    if (!pb_plan(N, T, V, beam, &pl)) return AVCTC_ERR_UNSUPPORTED;
    if (N == 0) return AVCTC_OK;
    if (!out_len || !out_scores || !status || !workspace || (T > 0 && (!log_probs || !out_tokens)))
        return AVCTC_ERR_BAD_ARG;
    if (workspace_bytes < pl.total) return AVCTC_ERR_WORKSPACE;
    if (reinterpret_cast<uintptr_t>(workspace) & 255) return AVCTC_ERR_ALIGNMENT;
    char* w = reinterpret_cast<char*>(workspace);
    PbParams p;
    p.lp = log_probs; p.stride_n = stride_n; p.stride_t = stride_t;
    p.N = N; p.T = T; p.V = V; p.lengths = lengths;
    p.beam = beam; p.nbest = nbest; p.blank = blank; p.k = pl.k;
    p.tk_val = reinterpret_cast<float*>(w + pl.off_tv);
    p.tk_idx = reinterpret_cast<int32_t*>(w + pl.off_ti);
    p.nodes_g = pl.smem_nodes ? nullptr : reinterpret_cast<uint32_t*>(w + pl.off_nodes);
    p.node_cap = pl.node_cap;
    p.out_tokens = out_tokens; p.out_len = out_len; p.out_scores = out_scores; p.status = status;
    const int rc = avctc_beam_topk_lists(log_probs, stride_n, stride_t, N, T, V, lengths, pl.k,
                                         reinterpret_cast<float*>(w + pl.off_tv),
                                         reinterpret_cast<int32_t*>(w + pl.off_ti), stream);
    if (rc) return rc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const size_t smem = pl.per_warp * kPbWarps;
    static bool configured = false;
    if (!configured && smem > 48 * 1024) {
        AVCTC_CUDA_RETURN(cudaFuncSetAttribute(ctc_prefix_beam_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               (int)round_up((size_t)kPbFixedBytes + (size_t)kPbSmemNodes * 4, 16) * kPbWarps));
        configured = true;
    }
    ctc_prefix_beam_kernel<<<(N + kPbWarps - 1) / kPbWarps, kPbWarps * 32, smem, st>>>(p, (int)pl.per_warp);
    return (int)cudaGetLastError();
}

namespace {

// §4.14's checks of an LM descriptor and its weights.
bool lm_args_ok(const avctc_ngram_lm* lm, int V, double lm_weight, double token_bonus) {
    if (!lm || lm->order < 1 || lm->order > 5 || lm->map_len != V || !std::isfinite(lm_weight) || lm_weight < 0.0 ||
        !std::isfinite(token_bonus) || lm->num_words < 3 || lm->num_words > 2048 || lm->bos < 0 ||
        lm->bos >= lm->num_words || lm->eos < 0 || lm->eos >= lm->num_words || !lm->token_word || !lm->unigram)
        return false;
    for (int o = 2; o <= lm->order; ++o) {
        const uint64_t cap = lm->capacity[o - 2];
        if (!lm->table[o - 2] || cap < 2 || (cap & (cap - 1))) return false;
    }
    return true;
}

// Both launches of the LM and / or biased search; the arguments are checked by the caller.  lm = NULL gives an
// unused PbLm of order 1, cx = NULL an unused PbCtx.
template <bool kLm, bool kBias>
int launch_lm_search(const float* log_probs, int64_t stride_n, int64_t stride_t, int N, int T, int V,
                     const int64_t* lengths, int beam, int nbest, int blank, const avctc_ngram_lm* lm,
                     double lm_weight, double token_bonus, const avctc_context_graph* cx, int32_t* out_tokens,
                     int32_t* out_len, double* out_scores, double* out_acoustic, double* out_lm, double* out_bias,
                     int32_t* status, void* workspace, size_t workspace_bytes, void* stream) {
    PbPlan pl;
    if (!pb_plan(N, T, V, beam, &pl)) return AVCTC_ERR_UNSUPPORTED;
    if (N == 0) return AVCTC_OK;
    if (!out_len || !out_scores || !out_acoustic || !out_lm || (kBias && !out_bias) || !status || !workspace ||
        (T > 0 && (!log_probs || !out_tokens)))
        return AVCTC_ERR_BAD_ARG;
    if (workspace_bytes < pl.total) return AVCTC_ERR_WORKSPACE;
    if (reinterpret_cast<uintptr_t>(workspace) & 255) return AVCTC_ERR_ALIGNMENT;
    char* w = reinterpret_cast<char*>(workspace);
    PbParams p;
    p.lp = log_probs; p.stride_n = stride_n; p.stride_t = stride_t;
    p.N = N; p.T = T; p.V = V; p.lengths = lengths;
    p.beam = beam; p.nbest = nbest; p.blank = blank; p.k = pl.k;
    p.tk_val = reinterpret_cast<float*>(w + pl.off_tv);
    p.tk_idx = reinterpret_cast<int32_t*>(w + pl.off_ti);
    p.nodes_g = pl.smem_nodes ? nullptr : reinterpret_cast<uint32_t*>(w + pl.off_nodes);
    p.node_cap = pl.node_cap;
    p.out_tokens = out_tokens; p.out_len = out_len; p.out_scores = out_scores; p.status = status;
    PbLm d = {};
    d.order = 1;
    if (lm) {
        d.token_word = lm->token_word;
        d.unigram = reinterpret_cast<const float2*>(lm->unigram);
        for (int o = 0; o < 4; ++o) {
            const bool used = o + 2 <= lm->order;
            d.tab[o] = used ? reinterpret_cast<const ulonglong2*>(lm->table[o]) : nullptr;
            d.mask[o] = used ? lm->capacity[o] - 1 : 0;
        }
        d.order = lm->order; d.bos = lm->bos; d.eos = lm->eos;
        d.alpha = lm_weight; d.beta = token_bonus;
    }
    PbCtx c = {};
    if (cx) {
        c.token_sym = cx->token_sym;
        c.delta = cx->delta;
        c.node = reinterpret_cast<const double2*>(cx->node);
        c.alphabet = cx->alphabet;
    }
    const int rc = avctc_beam_topk_lists(log_probs, stride_n, stride_t, N, T, V, lengths, pl.k,
                                         reinterpret_cast<float*>(w + pl.off_tv),
                                         reinterpret_cast<int32_t*>(w + pl.off_ti), stream);
    if (rc) return rc;
    constexpr size_t fixed = kBias ? kPbBiasFixedBytes : kPbLmFixedBytes;
    const size_t per_warp = round_up(fixed + (pl.smem_nodes ? (size_t)pl.node_cap * 4 : 0), 16);
    const size_t smem = per_warp * kPbWarps;
    static bool configured = false;
    if (!configured && smem > 48 * 1024) {
        AVCTC_CUDA_RETURN(cudaFuncSetAttribute(ctc_prefix_beam_lm_kernel<kLm, kBias>,
                                               cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               (int)round_up(fixed + (size_t)kPbSmemNodes * 4, 16) * kPbWarps));
        configured = true;
    }
    ctc_prefix_beam_lm_kernel<kLm, kBias><<<(N + kPbWarps - 1) / kPbWarps, kPbWarps * 32, smem,
                                            reinterpret_cast<cudaStream_t>(stream)>>>(
        p, d, out_acoustic, out_lm, (int)per_warp, c, out_bias);
    return (int)cudaGetLastError();
}

}  // namespace

extern "C" int avctc_ctc_prefix_beam_lm(const float* log_probs, int64_t stride_n, int64_t stride_t, int N, int T, int V,
                                        const int64_t* lengths, int beam, int nbest, int blank, const avctc_ngram_lm* lm,
                                        double lm_weight, double token_bonus, int32_t* out_tokens, int32_t* out_len,
                                        double* out_scores, double* out_acoustic, double* out_lm, int32_t* status,
                                        void* workspace, size_t workspace_bytes, void* stream) {
    if (N < 0 || T < 0 || V < 1 || beam < 1 || nbest < 1 || nbest > beam || blank < 0 || blank >= V)
        return AVCTC_ERR_BAD_ARG;
    if (!lm_args_ok(lm, V, lm_weight, token_bonus)) return AVCTC_ERR_BAD_ARG;
    return launch_lm_search<true, false>(log_probs, stride_n, stride_t, N, T, V, lengths, beam, nbest, blank, lm,
                                         lm_weight, token_bonus, nullptr, out_tokens, out_len, out_scores,
                                         out_acoustic, out_lm, nullptr, status, workspace, workspace_bytes, stream);
}

extern "C" int avctc_ctc_prefix_beam_biased(const float* log_probs, int64_t stride_n, int64_t stride_t, int N, int T,
                                            int V, const int64_t* lengths, int beam, int nbest, int blank,
                                            const avctc_ngram_lm* lm, double lm_weight, double token_bonus,
                                            const avctc_context_graph* ctx, int32_t* out_tokens, int32_t* out_len,
                                            double* out_scores, double* out_acoustic, double* out_lm, double* out_bias,
                                            int32_t* status, void* workspace, size_t workspace_bytes, void* stream) {
    if (N < 0 || T < 0 || V < 1 || beam < 1 || nbest < 1 || nbest > beam || blank < 0 || blank >= V)
        return AVCTC_ERR_BAD_ARG;
    if (!ctx || ctx->num_nodes < 1 || ctx->map_len != V || ctx->alphabet < 1 || ctx->alphabet > V ||
        !ctx->token_sym || !ctx->delta || !ctx->node)
        return AVCTC_ERR_BAD_ARG;
    if (lm && !lm_args_ok(lm, V, lm_weight, token_bonus)) return AVCTC_ERR_BAD_ARG;
    if (lm)
        return launch_lm_search<true, true>(log_probs, stride_n, stride_t, N, T, V, lengths, beam, nbest, blank, lm,
                                            lm_weight, token_bonus, ctx, out_tokens, out_len, out_scores,
                                            out_acoustic, out_lm, out_bias, status, workspace, workspace_bytes, stream);
    return launch_lm_search<false, true>(log_probs, stride_n, stride_t, N, T, V, lengths, beam, nbest, blank, nullptr,
                                         0.0, 0.0, ctx, out_tokens, out_len, out_scores, out_acoustic, out_lm,
                                         out_bias, status, workspace, workspace_bytes, stream);
}
