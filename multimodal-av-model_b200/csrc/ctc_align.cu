// ctc_align.cu — batched CTC forced alignment (Viterbi over the CTC lattice) for sm_100a.
//
// Computes what torchaudio.functional.forced_align computes on the CPU, for a padded batch in one launch:
//
//  ctc_align_kernel  one WARP (= one CTA) per utterance.  The [2L+1]-state lattice lives in registers in the layout
//                    of the CTC scan (ctc_loss.cu): lane g owns states g*K .. g*K+K-1, K even, so a lane's states
//                    alternate blank / label.  Per frame: the neighbour lane's last state arrives by __shfl_up, each
//                    state picks its predecessor with torchaudio's comparison order and adds the emission with ONE
//                    fp32 add (natural log, no rescaling: the sums are the reference's, bit for bit), and each lane
//                    writes its K two-bit back-pointers as one 32-bit word into shared memory.  Emissions are gathered
//                    D frames ahead by cp.async into a shared-memory ring, as in ctc_scan_kernel.  After the last
//                    frame lane 0 walks the back-pointers, and the warp writes labels and scores coalesced.
//
// Back-pointers take T x 32 x 4 bytes of shared memory (19 KB at T = 150, 125 KB at T = 1000); shapes whose
// back-pointers do not fit return AVCTC_ERR_UNSUPPORTED (avctc_ctc_align_supported).  One warp per CTA: CTAs of one
// warp already co-reside on an SM up to its shared-memory and CTA limits, so packing several utterances into one CTA
// would only add barriers.
#include "common.cuh"

namespace avctc {

constexpr int kAlignMaxSmem = 226 * 1024;   // dynamic shared memory per CTA (sm_100 opt-in limit: 227 KB in all)

template <int K>
struct AlignCfg {
    static constexpr int KL = K / 2;                 // label states per lane
    static constexpr int D = (K >= 12) ? 8 : 16;     // emission prefetch depth (frames)
    static constexpr int EW = KL + 1;                // staged words per lane per frame: blank + KL labels
    static constexpr int ring_words = D * 32 * EW;
};

// dynamic shared memory: [emission ring][label-change flags: 256 + 32 bytes][back-pointers: T x 32 words]
static inline size_t align_smem_bytes(int K, int T) {
    const int KL = K / 2, D = (K >= 12) ? 8 : 16;
    return (size_t)D * 32 * (KL + 1) * 4 + 288 + (size_t)(T > 1 ? T : 1) * 32 * 4;
}

static inline int align_k(int max_target_len) {
    const int need = (2 * max_target_len + 1 + 31) / 32;
    static const int ks[6] = {2, 4, 6, 8, 12, 16};
    for (int i = 0; i < 6; ++i) if (ks[i] >= need) return ks[i];
    return 0;
}

struct AlignParams {
    const void* lp; int64_t stride_n, stride_t;
    int T, V;
    const int64_t* targets; int64_t target_stride;
    const int64_t* input_lengths; const int64_t* target_lengths;
    int Lmax, blank;
    int32_t* paths; void* scores; int32_t* status;
};

template <typename TIn>
__device__ __forceinline__ void store_score(void* scores, size_t i, TIn v) { reinterpret_cast<TIn*>(scores)[i] = v; }

template <int K, typename TIn>
__global__ void __launch_bounds__(32) ctc_align_kernel(const AlignParams p) {
    using Cfg = AlignCfg<K>;
    constexpr int KL = Cfg::KL, D = Cfg::D, EW = Cfg::EW;
    const int b = blockIdx.x;
    const int lane = threadIdx.x;
    extern __shared__ __align__(16) unsigned smem_raw[];
    unsigned* em_raw = smem_raw;                                                    // [D][32][EW]
    unsigned char* chg = reinterpret_cast<unsigned char*>(smem_raw + Cfg::ring_words);   // chg[j] = tg[j] != tg[j-1]
    unsigned* bp = smem_raw + Cfg::ring_words + 72;                                 // [T][32]
    __shared__ float fin[2];

    const TIn* lpb = reinterpret_cast<const TIn*>(p.lp) + (int64_t)b * p.stride_n;
    int32_t* prow = p.paths + (size_t)b * p.T;
    const size_t srow = (size_t)b * p.T;
    const TIn zero = TIn(0.f);

    // ---- validate the utterance (every lane computes the same verdict)
    const long long tbl = p.input_lengths[b], tll = p.target_lengths[b];
    int code = 0;
    if (tbl < 0 || tbl > p.T || tll < 0 || tll > p.Lmax) code = 3;
    const int Tb = code ? 0 : (int)tbl;
    const int L = code ? 0 : (int)tll;
    const int64_t* tg = p.targets + (int64_t)b * p.target_stride;
    int R = 0;
    for (int j0 = 0; j0 < L && !code; j0 += 32) {
        const int j = j0 + lane;
        long long c = 0, cp = -1;
        if (j < L) { c = tg[j]; if (j > 0) cp = tg[j - 1]; }
        const bool bad = j < L && (c < 0 || c >= p.V || c == p.blank);
        const bool rep = j < L && j > 0 && c == cp;
        if (j < L) chg[j] = (j > 0 && c != cp) ? 1 : 0;
        if (__any_sync(kFullMask, bad)) code = 1;
        R += __popc(__ballot_sync(kFullMask, rep));
    }
    if (!code && Tb < L + R) code = 2;
    if (code || Tb == 0) {            // rejected or empty: blank / 0 everywhere
        for (int t = lane; t < p.T; t += 32) { prow[t] = p.blank; store_score<TIn>(p.scores, srow + t, zero); }
        if (lane == 0) p.status[b] = code;
        return;
    }
    chg[L + lane] = 0;                // reads past the last label see "no change" (chg has 288 entries, L <= 255)
    __syncwarp();

    const int S = 2 * L + 1;
    const int LR = L + R;
    const int g = lane;
    const int nvalid = min(max(S - g * K, 0), K);
    int lab[KL];
#pragma unroll
    for (int i = 0; i < KL; ++i) {
        const int j = g * KL + i;
        lab[i] = (j < L) ? (int)tg[j] : p.blank;
    }
    bool skip[KL];
#pragma unroll
    for (int i = 0; i < KL; ++i) {
        const int j = g * KL + i;
        skip[i] = (j >= 1 && j < L) ? chg[j] != 0 : false;
    }

    // ---- frame 0: alpha[i] = lp[0][label(i)] for i in [start, end)
    int start = (Tb - LR > 0) ? 0 : 1;
    int end = (S == 1) ? 1 : 2;
    float a[K];
#pragma unroll
    for (int j = 0; j < K; ++j) a[j] = AVCTC_NEG_INF;
    if (g == 0) {
        if (start == 0) a[0] = to_float(lpb[p.blank]);
        if (end == 2) a[1] = to_float(lpb[lab[0]]);
    }

    // ---- emission staging (cp.async gathers, D frames ahead).  A register ring stalls: the scoreboard cannot track
    // D outstanding loads individually, so every frame would wait for the newest one (see ctc_scan_kernel).
    const long long fstep = p.stride_t;
    const TIn* gp_b = lpb + p.blank + fstep;
    const TIn* gp_l[KL];
#pragma unroll
    for (int i = 0; i < KL; ++i) gp_l[i] = lpb + lab[i] + fstep;
    constexpr int slot_words = 32 * EW;
    unsigned* em_mine = em_raw + lane * EW;
    int par_b = 0;                     // bf16: which half of the staged word holds the element (blank; labels as bits)
    unsigned par_l = 0;
    const int par_step = (int)(fstep & 1);
    const bool gathers = nvalid > 0;
    auto issue = [&](unsigned* dst, bool live) {
        if (live && gathers) {
            if constexpr (sizeof(TIn) == 4) {
                cp_async_4(dst, gp_b);
#pragma unroll
                for (int i = 0; i < KL; ++i) cp_async_4(dst + 1 + i, gp_l[i]);
            } else {   // 2-byte elements: copy the aligned 4-byte word holding the element
                cp_async_4(dst, reinterpret_cast<const void*>(reinterpret_cast<uintptr_t>(gp_b) & ~(uintptr_t)3));
#pragma unroll
                for (int i = 0; i < KL; ++i)
                    cp_async_4(dst + 1 + i,
                               reinterpret_cast<const void*>(reinterpret_cast<uintptr_t>(gp_l[i]) & ~(uintptr_t)3));
            }
        }
        cp_async_commit();
        gp_b += fstep;
#pragma unroll
        for (int i = 0; i < KL; ++i) gp_l[i] += fstep;
    };
    if constexpr (sizeof(TIn) == 2) {
        par_b = (int)((reinterpret_cast<uintptr_t>(gp_b) >> 1) & 1);
#pragma unroll
        for (int i = 0; i < KL; ++i) par_l |= (unsigned)((reinterpret_cast<uintptr_t>(gp_l[i]) >> 1) & 1) << i;
    }
    for (int d = 1; d <= D; ++d) issue(em_mine + (d & (D - 1)) * slot_words, d < Tb);

    int slot = 1 & (D - 1);
    int live_left = Tb - 1 - D;
    unsigned* bpw = bp + 32 + lane;    // this lane's word of frame 1
#pragma unroll 1
    for (int t = 1; t < Tb; ++t) {
        cp_async_wait<D - 1>();        // frames <= t have landed (own copies only)
        unsigned* sl_ptr = em_mine + slot * slot_words;
        float vb, vl[KL];
        if constexpr (sizeof(TIn) == 4) {
            vb = __uint_as_float(sl_ptr[0]);
#pragma unroll
            for (int i = 0; i < KL; ++i) vl[i] = __uint_as_float(sl_ptr[1 + i]);
        } else {
            auto pick = [](unsigned w, int par) { return __uint_as_float(par ? (w & 0xffff0000u) : (w << 16)); };
            vb = pick(sl_ptr[0], par_b);
            par_b ^= par_step;
#pragma unroll
            for (int i = 0; i < KL; ++i) vl[i] = pick(sl_ptr[1 + i], (par_l >> i) & 1u);
            if (par_step) par_l ^= (1u << KL) - 1u;
        }
        issue(sl_ptr, live_left > 0);  // refills the slot just read (frame t + D)
        --live_left;
        slot = (slot + 1) & (D - 1);

        // frame window (torchaudio): states that can no longer reach the end / not yet be reached are -inf
        if (Tb - t <= LR) start += ((start & 1) && chg[(start >> 1) + 1]) ? 2 : 1;
        if (t <= LR) end += (!(end & 1) && end < 2 * L && chg[end >> 1]) ? 2 : 1;
        const int lo = start - g * K, hi = end - g * K;   // this lane's states j with lo <= j < hi are live

        float up = __shfl_up_sync(kFullMask, a[K - 1], 1);
        if (lane == 0) up = AVCTC_NEG_INF;
        float nw[K];
        unsigned word = 0;
#pragma unroll
        for (int i = 0; i < KL; ++i) {
            const float below = (i == 0) ? up : a[2 * i - 1];
            // blank state 2i: x0 = itself, x1 = below, no skip
            {
                const float x0 = a[2 * i], x1 = below;
                const bool c1 = x1 > x0;
                const bool live = (2 * i >= lo) && (2 * i < hi);
                nw[2 * i] = live ? (c1 ? x1 : x0) + vb : AVCTC_NEG_INF;
                word |= (live ? (c1 ? 1u : 0u) : 3u) << (4 * i);   // field 3 = torchaudio's -1: outside the window
            }
            // label state 2i+1: x0 = itself, x1 = the blank below it, x2 = the label below that when it differs
            {
                const float x0 = a[2 * i + 1], x1 = a[2 * i];
                const float x2 = skip[i] ? below : AVCTC_NEG_INF;
                const bool c2 = x2 > x1 && x2 > x0;
                const bool c1 = !c2 && x1 > x0 && x1 > x2;
                const bool live = (2 * i + 1 >= lo) && (2 * i + 1 < hi);
                nw[2 * i + 1] = live ? (c2 ? x2 : (c1 ? x1 : x0)) + vl[i] : AVCTC_NEG_INF;
                word |= (live ? (c2 ? 2u : (c1 ? 1u : 0u)) : 3u) << (4 * i + 2);
            }
        }
#pragma unroll
        for (int j = 0; j < K; ++j) a[j] = nw[j];
        *bpw = word;
        bpw += 32;
    }
    cp_async_wait<0>();

    // ---- final state: S-1 if alpha[S-1] > alpha[S-2] else S-2 (L = 0: the single blank state)
#pragma unroll
    for (int j = 0; j < K; ++j) {
        const int s = g * K + j;
        if (s == S - 1) fin[0] = a[j];
        if (s == S - 2) fin[1] = a[j];
    }
    __syncwarp();
    // ---- backtrack (lane 0, serial): the state of frame t replaces word 0 of frame t, which nobody reads again
    if (lane == 0) {
        int s = (S == 1 || fin[0] > fin[1]) ? S - 1 : S - 2;
        for (int t = Tb - 1; t >= 1; --t) {
            const unsigned w = bp[t * 32 + s / K];
            const int f = (int)((w >> (2 * (s % K))) & 3u);
            bp[t * 32] = (unsigned)s;
            s = min(s - (f == 3 ? -1 : f), S - 1);
        }
        bp[0] = (unsigned)s;
    }
    __syncwarp();
    for (int t = lane; t < p.T; t += 32) {
        if (t < Tb) {
            const int s = (int)bp[t * 32];
            const int c = (s & 1) ? (int)tg[s >> 1] : p.blank;
            prow[t] = c;
            store_score<TIn>(p.scores, srow + t, lpb[(int64_t)t * p.stride_t + c]);
        } else {
            prow[t] = p.blank;
            store_score<TIn>(p.scores, srow + t, zero);
        }
    }
    if (lane == 0) p.status[b] = 0;
}

template <int K, typename TIn>
static int launch_align(const AlignParams& p, int N, cudaStream_t st) {
    const size_t smem = align_smem_bytes(K, p.T);
    auto kern = ctc_align_kernel<K, TIn>;
    AVCTC_CUDA_RETURN(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<N, 32, smem, st>>>(p);
    return (int)cudaGetLastError();
}

template <typename TIn>
static int dispatch_align(const AlignParams& p, int K, int N, cudaStream_t st) {
    switch (K) {
        case 2: return launch_align<2, TIn>(p, N, st);
        case 4: return launch_align<4, TIn>(p, N, st);
        case 6: return launch_align<6, TIn>(p, N, st);
        case 8: return launch_align<8, TIn>(p, N, st);
        case 12: return launch_align<12, TIn>(p, N, st);
        case 16: return launch_align<16, TIn>(p, N, st);
    }
    return AVCTC_ERR_UNSUPPORTED;
}

}  // namespace avctc

using namespace avctc;

extern "C" int avctc_ctc_align_supported(int T, int max_target_len) {
    if (T < 0 || max_target_len < 0) return 0;
    const int K = align_k(max_target_len);
    if (K == 0) return 0;
    return align_smem_bytes(K, T) <= (size_t)kAlignMaxSmem ? 1 : 0;
}

extern "C" int avctc_ctc_align(const void* log_probs, int dtype, int64_t stride_n, int64_t stride_t, int N, int T, int V,
                               const int64_t* targets, int64_t target_stride, const int64_t* input_lengths,
                               const int64_t* target_lengths, int max_target_len, int blank, int32_t* paths,
                               void* scores, int32_t* status, void* stream) {
    if (N < 0 || T < 0 || V <= 0 || max_target_len < 0 || blank < 0 || blank >= V) return AVCTC_ERR_BAD_ARG;
    if (dtype != AVCTC_F32 && dtype != AVCTC_BF16) return AVCTC_ERR_BAD_ARG;
    if (!avctc_ctc_align_supported(T, max_target_len)) return AVCTC_ERR_UNSUPPORTED;
    if (N == 0) return AVCTC_OK;
    if (!log_probs || !targets || !input_lengths || !target_lengths || !paths || !scores || !status)
        return AVCTC_ERR_BAD_ARG;
    AlignParams p;
    p.lp = log_probs; p.stride_n = stride_n; p.stride_t = stride_t;
    p.T = T; p.V = V;
    p.targets = targets; p.target_stride = target_stride;
    p.input_lengths = input_lengths; p.target_lengths = target_lengths;
    p.Lmax = max_target_len; p.blank = blank;
    p.paths = paths; p.scores = scores; p.status = status;
    const int K = align_k(max_target_len);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (dtype == AVCTC_F32) return dispatch_align<float>(p, K, N, st);
    return dispatch_align<__nv_bfloat16>(p, K, N, st);
}
