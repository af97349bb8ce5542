// lattice.cu -- alpha/beta recursion over the blank-extended label lattice (kernel 2).
//
// Replaces the two serial Python loops of the reference, _compute_transition_probability
// (asr/loss/gram_ctc.py:142-178): loop 1 (:153-156) = alpha, loop 2 (:171-175) = beta, each a dense
// (B,N,N) log-matmul per frame there.  Here the adjacency is walked as the banded structure it is
// (SURVEY.md section 8a "banded lattice spec"):
//   CTC      node q: self, q-1, and q-2 iff q is a label node whose label differs from the previous one
//   Gram-CTC forward  type 0 (blank): q, q-1, q-2        type 1 (unigram): q, q-1, q-2, q-3*
//                     type 2 (bigram): q, q-5, q-7, q-6* (dead when the bigram id is -1)
//            reversed type 0 (blank): q, q-1, q-5        type 1 (bigram): q, q-1, q-2, q-6*
//                     type 2 (unigram): q, q-2, q-3*, q-7          (* = only if the two ids differ)
//
// Arithmetic.  The reference works in log space (one logsumexp per node and frame: 3-4 exp + 1 log on the
// critical path).  Here every lattice value is a pair (m, e) = m * 2^e with a float32 mantissa and an
// integer-valued float32 exponent PER NODE (common.cuh, "scaled linear").  A step is then
//     E = max_i e_i;   pre = sum_i m_i * 2^(e_i - E);   m' = pre * em;   e' = E + ee
// where (em, ee) is the emission probability in the same format.  The exponent recursion is a (max,+) chain
// that does not depend on the mantissas, the mantissa chain is FMUL/FFMA only, the scale factors 2^(e_i - E)
// are exact powers of two built on the integer pipe, and the mantissas are pulled back into [1,2) once per
// chunk of frames (they drift by at most a factor 2^-1 .. 3 per frame).  Nothing can under/overflow whatever
// the dynamic range between nodes or along the utterance is; a microbenchmark of the step gives ~62 cycles
// against ~225 for the log-space step this replaces (tools/ubench_step_linear.cu, tools/ubench_step.cu).
//
// Mapping.  Two CTAs per utterance: one runs alpha forward in time, the other beta backward in time on the
// reversed lattice (the two are independent until the gradient kernel multiplies them; on separate SMs they
// do not share an issue port or the SM's store bandwidth, which is what bounds a step once the arithmetic is
// cheap: 2 x Np float2 per frame).  Within a CTA warp w owns nodes [w*32K, (w+1)*32K), K consecutive nodes per
// lane, all state in registers; K is kept small (2 for CTC, 3 for Gram-CTC) because the step is bound by the
// issue rate and the dependent chain of a single warp, so the lattice is spread over several warps, i.e. SM
// sub-partitions.
//   * inside a warp the 2 (CTC) / 7 (Gram) boundary values come from the lower lanes by warp shuffle;
//   * between warps they travel through shared memory, and the warps run as a systolic pipeline at
//     chunk granularity (16 frames): warp w works on chunk c while warp w+1 works on chunk c-1,
//     reading the per-frame boundary values warp w left behind.  Hand-over is one mbarrier wait and one
//     arrive per warp and chunk; the wait for chunk c+1 is issued before the last step of chunk c;
//   * the per-frame rows of gathered emission probabilities are staged in shared memory by 1-D bulk async
//     copies (TMA engine) issued by a dedicated I/O warp, as far ahead as the stage ring allows.
//
// Both directions run the full utterance: alpha writes av[t][j] = alpha_t[j], beta writes bv[t][j] = beta_t[j].
// P is read off alpha at the last frame.  The gradient kernel forms alpha * beta / P itself while it merges
// the per-symbol posteriors, so the recursion carries no "combine" work at all.
//
// beta convention as in the reference (:171-175): beta_t EXCLUDES the emission at t, so
// sum_j alpha_t[j] * beta_t[j] = P at every valid frame.
//
// The same launch carries B extra CTAs that build the gradient kernel's symbol tables (prep.cuh) while
// the recursion runs, and the last alpha CTA to finish reduces the batch loss in a fixed order.
#include "common.cuh"
#include "kernels.h"
#include "prep.cuh"

namespace b200ctc {

namespace {

// Frames per pipeline chunk (and per mantissa renormalisation) are a template parameter CH: 16 for the usual
// lattices, 8 or 4 for long label sequences, whose emission rows are wide -- the stage ring must hold the W chunks
// the warps are working on plus 3 in front of them (a bulk copy takes ~2 us from issue to landing, longer than a
// chunk), and a stage is CH rows.
constexpr int kMaxStages = 24;
constexpr int kMaxWarpsPerDir = 16;
constexpr int kGenericMaxWarps = 8;   // Gram-CTC lattices of up to 256 nodes run one node per lane (K = 1)

// Reversed direction: q <-> j = Nb - 1 - q, so the reversed CTC lattice has the same shape as the forward one
// (even q = blank, odd q = label) and a lane's two nodes are j-1 (label), j (blank) with j even.  The beta rows
// are STORED one element up (WsLayout::boff = 1 for CTC), which makes that pair a 16-byte aligned one and lets
// beta use the same single 128-bit store per lane as alpha.
template <int K, bool GRAM>
struct Geo {
    static constexpr int PAD = GRAM ? 7 : 2;                 // how far back a node's predecessors reach
    static constexpr int EXT = K + PAD;
};

template <int K, bool GRAM>
struct LaneState {
    float m[K], e[K];        // mantissa / exponent of the K nodes this lane owns (post-emission)
    int ci[K];               // column of each node's symbol in the emission row (0 = blank)
    float openoff[K];        // 0 when the "ids differ" edge into slot r is open, SENT when it is closed
    uint32_t valid;          // bit r: node index < Nb
    int dk[3];               // K == 1 only (one node per lane, its type known at run time): how many lanes back the
                             // three predecessors besides the node itself sit; 0 = no such edge
};

// shared-memory view of the pipeline (32-bit shared-space addresses: no generic-pointer conversion inside the
// recursion loop)
struct DirPipe {
    uint32_t lp;             // [S][CH][Wlp] float2   staged emission rows
    uint32_t bnd;            // [W-1][S][CH][PAD] float2 boundary values handed from warp w to warp w+1;
                             //   as deep as the stage ring, so a buffer is free by the time it comes round again
                             //   (a warp can only be at chunk c once the last warp has consumed chunk c-S)
    uint32_t bnd_none;       // [CH][PAD] float2 of (0, SENT): what warp 0 reads as "the warp before me"
    uint64_t *full;          // [S]     emission rows of a chunk have landed (tx count); warp 0 waits on it
    uint64_t *consumed;      // [S]     the last warp is done with the stage (hence every warp is)
    uint64_t *ready;         // [W-1][S] warp w finished the chunk: its boundary values can be read, and the
                             //          stage's emission rows are known to have landed
};

// Shared-memory loads as PURE asm (no volatile, no memory clobber): the compiler may hoist them to the top of a
// chunk, off the dependent chain.  They cannot cross a barrier wait because their address is derived from a
// token that the wait defines (after_wait()).
__device__ __forceinline__ float2 lds_f2(uint32_t addr) {
    float2 v;
    asm("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_f2(uint32_t addr, float x, float y) {
    asm volatile("st.shared.v2.f32 [%0], {%1,%2};" ::"r"(addr), "f"(x), "f"(y));
}
__device__ __forceinline__ uint32_t after_wait(uint32_t addr) {
    uint32_t r;
    asm volatile("mov.u32 %0, %1;" : "=r"(r) : "r"(addr) : "memory");
    return r;
}

struct UttCtx {
    const float2 *lp_g;      // this utterance's emission rows   [T][Wlp]
    float2 *out_g;           // this direction's output rows     [T][Np]
    int Wlp, Np, Nb, W, S, boff;
};

// ---- one lattice step: new (pre-emission) value of slot R from the extended old arrays ----
// xm/xe hold nodes [K*gl - PAD, K*gl + K) for this lane; index PAD + R is slot R itself.
template <int K, bool GRAM, bool REV, int R>
__device__ __forceinline__ void slot_update(const float (&xm)[Geo<K, GRAM>::EXT], const float (&xe)[Geo<K, GRAM>::EXT],
                                            float openoff, float &pre_m, float &pre_e) {
    constexpr int PAD = Geo<K, GRAM>::PAD;
    constexpr int I = PAD + R;
    if constexpr (!GRAM) {
        if constexpr ((R & 1) == 0) {                         // blank node: self, q-1
            const float E = fmaxf(xe[I], xe[I - 1]);
            pre_m = fmaf(xm[I - 1], pow2_nonpos(xe[I - 1] - E), xm[I] * pow2_nonpos(xe[I] - E));
            pre_e = E;
        } else {                                              // label node: self, q-1, q-2*
            const float e2 = xe[I - 2] + openoff;
            const float E = fmaxf(fmaxf(xe[I], xe[I - 1]), e2);
            float s = xm[I] * pow2_nonpos(xe[I] - E);
            s = fmaf(xm[I - 1], pow2_nonpos(xe[I - 1] - E), s);
            s = fmaf(xm[I - 2], pow2_nonpos(e2 - E), s);
            pre_m = s;
            pre_e = E;
        }
    } else {
        constexpr int TYPE = R % 3;
        // predecessor offsets per (direction, type); the starred one is gated by `openoff`
        constexpr int A = (TYPE == 0) ? 1 : (!REV ? (TYPE == 1 ? 1 : 5) : (TYPE == 1 ? 1 : 2));
        constexpr int Bk = (TYPE == 0) ? (!REV ? 2 : 5) : (!REV ? (TYPE == 1 ? 2 : 7) : (TYPE == 1 ? 2 : 7));
        constexpr int Cs = (TYPE == 0) ? 0 : (!REV ? (TYPE == 1 ? 3 : 6) : (TYPE == 1 ? 6 : 3));
        float E = fmaxf(fmaxf(xe[I], xe[I - A]), xe[I - Bk]);
        float ec = SENT;
        if constexpr (Cs != 0) {
            ec = xe[I - Cs] + openoff;
            E = fmaxf(E, ec);
        }
        float s = xm[I] * pow2_nonpos(xe[I] - E);
        s = fmaf(xm[I - A], pow2_nonpos(xe[I - A] - E), s);
        s = fmaf(xm[I - Bk], pow2_nonpos(xe[I - Bk] - E), s);
        if constexpr (Cs != 0) s = fmaf(xm[I - Cs], pow2_nonpos(ec - E), s);
        pre_m = s;
        pre_e = E;
        // a dead bigram node (id -1, gram_ctc.py:94-98) needs no special case: its emission column holds
        // probability zero (softmax_gather.cu), so its post-emission state is (0, SENT) at every frame
    }
}

// Old values of the PAD nodes below this lane's first node: from lower lanes by shuffle, or -- for the first
// lanes of a warp -- from the previous warp's boundary record (warp 0 reads a constant record of zeros).
// Branch-free: every lane reads a (clamped) boundary slot and the right source is picked by select.
template <int K, bool GRAM>
__device__ __forceinline__ void gather_ext(const LaneState<K, GRAM> &st, float (&xm)[Geo<K, GRAM>::EXT],
                                           float (&xe)[Geo<K, GRAM>::EXT], int lane, uint32_t bnd_in) {
    constexpr int PAD = Geo<K, GRAM>::PAD;
#pragma unroll
    for (int x = 0; x < PAD; ++x) {
        const int delta = (PAD - x + K - 1) / K;              // lanes back (compile-time after unrolling)
        const int slot = x - PAD + K * delta;
        const float2 bv = lds_f2(bnd_in + 8u * (uint32_t)min(K * lane + x, PAD - 1));
        const float nm = __shfl_up_sync(0xffffffffu, st.m[slot], delta);
        const float ne = __shfl_up_sync(0xffffffffu, st.e[slot], delta);
        const bool edge = lane < delta;
        xm[x] = edge ? bv.x : nm;
        xe[x] = edge ? bv.y : ne;
    }
#pragma unroll
    for (int r = 0; r < K; ++r) {
        xm[PAD + r] = st.m[r];
        xe[PAD + r] = st.e[r];
    }
}

template <int K, bool GRAM, bool REV, int R>
struct SlotLoop {
    __device__ __forceinline__ static void run(LaneState<K, GRAM> &st, const float (&xm)[Geo<K, GRAM>::EXT],
                                               const float (&xe)[Geo<K, GRAM>::EXT], uint32_t lprow, float2 (&outv)[K]) {
        float pm, pe;
        slot_update<K, GRAM, REV, R>(xm, xe, st.openoff[R], pm, pe);
        const float2 em = lds_f2(lprow + 8u * (uint32_t)st.ci[R]);       // emission (mantissa, exponent)
        const float nm = pm * em.x;
        const float ne = pe + em.y;
        st.m[R] = nm;
        st.e[R] = ne;
        // alpha keeps the emission at t, beta excludes it (gram_ctc.py:171-175)
        outv[R] = REV ? make_float2(pm, pe) : make_float2(nm, ne);
        if constexpr (R + 1 < K) SlotLoop<K, GRAM, REV, R + 1>::run(st, xm, xe, lprow, outv);
    }
};

// Write this lane's K results of one frame.  out points at the lane's first node (REV: walks downwards).
// Partial 32-byte sectors are poison here: the output lines are never resident in L2 when first written, so a
// half-written sector costs a DRAM fill.  For the CTC layout (K = 2) every lane therefore writes one aligned
// 16-byte pair (WsLayout::boff is what aligns the reversed direction's pairs).
template <int K, bool GRAM, bool REV>
__device__ __forceinline__ void store_results(const float2 (&outv)[K], float2 *out, uint32_t store_mask, int lane) {
    if constexpr (!GRAM && K == 2) {
        if constexpr (!REV) {
            // nodes (2gl, 2gl+1): aligned; the odd partner of the last valid node falls into the row padding
            if (store_mask & 1u) *reinterpret_cast<float4 *>(out) = make_float4(outv[0].x, outv[0].y, outv[1].x, outv[1].y);
        } else {
            // slot 0 = node j (blank), slot 1 = node j-1; out points at slot 0's (shifted, odd) storage element
            if (store_mask & 1u) *reinterpret_cast<float4 *>(out - 1) = make_float4(outv[1].x, outv[1].y, outv[0].x, outv[0].y);
        }
    } else if constexpr (!GRAM && K == 4) {
        // four nodes = one 32-byte sector, written whole by ONE 256-bit store (STG.E.256): four predicated 8-byte stores
        // made four partial-sector writes per lane and frame, and the long lattices this mapping is for ran four times
        // slower per frame than the two-node mapping.  The reversed direction's groups are sector-aligned because its
        // lanes are shifted by `rev_shift` phantom nodes (init_lane); slots of a group that hold no node land in the
        // row padding.
        if (store_mask != 0u) {
            float2 *dst = REV ? out - 3 : out;
            const float2 a = outv[REV ? 3 : 0], b = outv[REV ? 2 : 1], c = outv[REV ? 1 : 2], d = outv[REV ? 0 : 3];
            asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dst), "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y),
                         "f"(c.x), "f"(c.y), "f"(d.x), "f"(d.y)
                         : "memory");
        }
    } else {
#pragma unroll
        for (int r = 0; r < K; ++r)
            if ((store_mask >> r) & 1u) out[REV ? -r : r] = outv[r];
    }
}

// Reversed direction of the four-node CTC mapping: number of phantom nodes in front of the lattice's first node, chosen
// so that every lane's group of four storage elements (node j is stored at j + boff whatever the mapping) starts on a
// 32-byte boundary: (Nb + shift + boff) % 4 == 0.  Even for CTC (Nb odd, boff 1), so blank/label parity is kept.
template <int K, bool GRAM>
__host__ __device__ inline int rev_shift(int Nb, int boff) {
    return (!GRAM && K == 4) ? ((4 - ((Nb + boff) & 3)) & 3) : 0;
}

// one frame of the recursion for this lane
template <int K, bool GRAM, bool REV>
__device__ __forceinline__ void lattice_step(LaneState<K, GRAM> &st, int lane, bool has_next,
                                             uint32_t bin, uint32_t bout, uint32_t lprow, float2 *out) {
    constexpr int PAD = Geo<K, GRAM>::PAD;
    if constexpr (K == 1) {
        // One node per lane: the Gram-CTC lattice of a usual utterance (181 nodes at L = 60) then spreads over six
        // warps instead of two, and a step is ~50 instructions instead of ~120.  The node types alternate along the
        // lanes, so the predecessors are fetched with per-lane source lanes (SHFL.IDX); the first lanes of a warp
        // take them from the previous warp's boundary record.
        const float m0 = st.m[0], e0 = st.e[0];
        float vm[3], ve[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int src = lane - st.dk[k];
            const float sm_ = __shfl_sync(0xffffffffu, m0, src & 31);
            const float se_ = __shfl_sync(0xffffffffu, e0, src & 31);
            const float2 bv = lds_f2(bin + 8u * (uint32_t)max(0, min(PAD - 1, PAD + src)));
            const bool edge = src < 0;
            vm[k] = edge ? bv.x : sm_;
            ve[k] = st.dk[k] == 0 ? SENT : (edge ? bv.y : se_);
        }
        if (has_next && lane >= 32 - PAD) sts_f2(bout + 8u * (uint32_t)(lane - (32 - PAD)), m0, e0);
        const float E = fmaxf(fmaxf(e0, ve[0]), fmaxf(ve[1], ve[2]));
        float sum = m0 * pow2_nonpos(e0 - E);
        sum = fmaf(vm[0], pow2_nonpos(ve[0] - E), sum);
        sum = fmaf(vm[1], pow2_nonpos(ve[1] - E), sum);
        sum = fmaf(vm[2], pow2_nonpos(ve[2] - E), sum);
        const float2 em = lds_f2(lprow + 8u * (uint32_t)st.ci[0]);
        const float nm = sum * em.x, ne = E + em.y;
        st.m[0] = nm;
        st.e[0] = ne;
        if (st.valid & 1u) *out = REV ? make_float2(sum, E) : make_float2(nm, ne);
        return;
    }
    float xm[Geo<K, GRAM>::EXT], xe[Geo<K, GRAM>::EXT];
    gather_ext<K, GRAM>(st, xm, xe, lane, bin);
    // leave my last PAD nodes' old values for warp w+1 (predicated stores, no branch)
#pragma unroll
    for (int r = 0; r < K; ++r) {
        const int idx = K * lane + r - (32 * K - PAD);
        if (has_next && idx >= 0) sts_f2(bout + 8u * (uint32_t)idx, st.m[r], st.e[r]);
    }
    float2 outv[K];
    SlotLoop<K, GRAM, REV, 0>::run(st, xm, xe, lprow, outv);
    store_results<K, GRAM, REV>(outv, out, st.valid, lane);
}

// The I/O warp: stages the emission rows of every chunk, as far ahead as the stage ring allows.
// Keeping this off the compute warps matters: the recursion is a single dependent chain per warp.
// The softmax/gather kernel may still be running (api.cu launches the two kernels concurrently): before a chunk's
// rows are copied, the warp makes sure the 16-frame blocks the chunk touches are complete.  It keeps a watermark of
// blocks known complete in its direction of travel and, when it has to look, checks 32 blocks with one round trip.
// A wait that lasts seconds means the softmax/gather kernel is not running next to this one at all (something else
// holds the SMs): give up, flag it (WsHeader::stalled; the call's losses become NaN) and run on with whatever is there --
// a wrong result that the caller's NaN guard catches, not a hung GPU.
constexpr unsigned kPollLimit = 1u << 24;         // x (128 ns nap + one L2 round trip): several seconds
template <bool REV, int CH>
__device__ __forceinline__ void io_direction(const DirPipe &pp, const UttCtx &c, int f0, int n, int lane,
                                             const unsigned char *ws, const WsLayout &wl, int b, bool poll,
                                             volatile unsigned *stalled) {
    if (n <= 0) return;
    unsigned idle = 0;
    const int S = c.S;
    const int nchunks = (n + CH - 1) / CH;
    const uint32_t row_bytes = (uint32_t)c.Wlp * 8u;
    const uint32_t stage_bytes = row_bytes * CH;
    int stage = 0;
    uint32_t wrap = 0;
    // blocks [0, known) (forward) / (known, last] (reversed) are complete
    int known = REV ? (n + kProgBlock - 1) / kProgBlock : 0;
    for (int ch = 0; ch < nchunks; ++ch) {
        const int i0 = ch * CH;
        const int cnt = min(CH, n - i0);
        const int flo = REV ? (f0 - i0 - cnt + 1) : (f0 + i0);
        if (wrap > 0 && lane == 0) mbar_wait(&pp.consumed[stage], (wrap - 1) & 1u);
        if (!poll) {
        } else if (!REV) {
            const int need = (flo + cnt - 1) / kProgBlock + 1;           // blocks [0, need) must be complete
            while (known < need) {
                const int got = count_blocks_done(ws, wl, b, n, known, 1, lane);
                known += got;
                if (got == 0) { __nanosleep(128); if (++idle > kPollLimit) { *stalled = 1u; break; } }
            }
        } else {
            const int need = flo / kProgBlock;                           // blocks [need, last] must be complete
            while (known > need) {
                const int got = count_blocks_done(ws, wl, b, n, known - 1, -1, lane);
                known -= got;
                if (got == 0) { __nanosleep(128); if (++idle > kPollLimit) { *stalled = 1u; break; } }
            }
        }
        if (lane == 0) {
            fence_proxy_async_global();                       // rows written through the generic proxy, read by the copy engine
            mbar_arrive_expect_tx(&pp.full[stage], row_bytes * cnt);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             pp.lp + (uint32_t)stage * stage_bytes),
                         "l"(c.lp_g + (size_t)flo * c.Wlp), "r"(row_bytes * cnt), "r"(smem_u32(&pp.full[stage]))
                         : "memory");
        }
        __syncwarp();
        if (++stage == S) { stage = 0; ++wrap; }
    }
}

// Visit n frames starting at f0 (ascending for alpha, descending for beta) with warp w of W.
template <int K, bool GRAM, bool REV, int CH>
__device__ __forceinline__ void run_direction(LaneState<K, GRAM> &st, const DirPipe &pp, const UttCtx &c, int f0, int n,
                                              int w, int lane) {
    constexpr int PAD = Geo<K, GRAM>::PAD;
    if (n <= 0) return;
    const int W = c.W, S = c.S;
    const int nchunks = (n + CH - 1) / CH;
    const bool has_prev = (w > 0), has_next = (w + 1 < W);
    const uint32_t row_bytes = (uint32_t)c.Wlp * 8u;
    const uint32_t stage_bytes = row_bytes * CH;
    const uint32_t bnd_chunk_bytes = CH * PAD * 8u;
    const int gl = 32 * w + lane;                             // lane index within the direction
    const int jbase = REV ? (c.Nb - 1 + rev_shift<K, GRAM>(c.Nb, c.boff) - K * gl + c.boff) : (K * gl);
    const int64_t frame_step = REV ? -(int64_t)c.Np : (int64_t)c.Np;
    float2 *out_ptr = c.out_g + (size_t)f0 * c.Np + jbase;    // this lane's first node in frame f0
    // what this warp waits for before a chunk: warp 0 the emission rows, the others the warp before them (which
    // has seen the emission rows land by then); what it signals after: the next warp, or -- the last warp -- the
    // I/O warp that the stage is free
    uint64_t *const wait_bar = has_prev ? pp.ready + (w - 1) * S : pp.full;
    uint64_t *const done_bar = has_next ? pp.ready + w * S : pp.consumed;

    int stage = 0;
    uint32_t wrap = 0;
    bool early = false;                                       // the wait for the coming chunk already succeeded
    for (int ch = 0; ch < nchunks; ++ch) {
        const int cnt = min(CH, n - ch * CH);
        if (!early) {
            if (ch == 0) mbar_wait_backoff(&wait_bar[stage], wrap & 1u);
            else mbar_wait(&wait_bar[stage], wrap & 1u);
        }

        const uint32_t lp_s = after_wait(pp.lp + (uint32_t)stage * stage_bytes);
        const uint32_t bin = after_wait(has_prev ? pp.bnd + (uint32_t)((w - 1) * S + stage) * bnd_chunk_bytes : pp.bnd_none);
        const uint32_t bout = pp.bnd + (uint32_t)((has_next ? w : 0) * S + stage) * bnd_chunk_bytes;
        const int nstage = (stage + 1 == S) ? 0 : stage + 1;
        const uint32_t nwrap = (stage + 1 == S) ? wrap + 1 : wrap;
        early = false;
        if (cnt == CH) {                                  // full chunk: straight-line code, no per-step branch
#pragma unroll
            for (int i = 0; i < CH; ++i) {
                const int row = REV ? (CH - 1 - i) : i;
                if (i == CH - 1 && ch + 1 < nchunks) early = mbar_test_wait(&wait_bar[nstage], nwrap & 1u);
                lattice_step<K, GRAM, REV>(st, lane, has_next, bin + i * PAD * 8u, bout + i * PAD * 8u,
                                           lp_s + (uint32_t)row * row_bytes, out_ptr + i * frame_step);
            }
        } else {                                              // last, partial chunk
#pragma unroll 1
            for (int i = 0; i < cnt; ++i) {
                const int row = REV ? (cnt - 1 - i) : i;
                lattice_step<K, GRAM, REV>(st, lane, has_next, bin + i * PAD * 8u, bout + i * PAD * 8u,
                                           lp_s + (uint32_t)row * row_bytes, out_ptr + i * frame_step);
            }
        }
        out_ptr += CH * frame_step;
        // pull the mantissas back into [1,2): they moved by at most 2^-CH .. 3^CH since the last time
#pragma unroll
        for (int r = 0; r < K; ++r) renorm_pair(st.m[r], st.e[r]);
        __syncwarp();
        if (lane == 0) mbar_arrive(&done_bar[stage]);
        stage = nstage; wrap = nwrap;
    }
}

template <int K, bool GRAM>
__device__ __forceinline__ void init_lane(LaneState<K, GRAM> &st, const ProblemDesc &d, int b, int Lb, int Nb,
                                          bool rev, int gl) {
    const int32_t *lab = d.labels + (size_t)b * d.Lmax;
    const int32_t *big = GRAM ? d.bigrams + (size_t)b * d.Lmax : nullptr;
    st.valid = 0u;
    const int shift = rev ? rev_shift<K, GRAM>(Nb, GRAM ? 0 : 1) : 0;     // phantom nodes in front (reversed 4-node CTC mapping)
#pragma unroll
    for (int r = 0; r < K; ++r) {
        const int q = K * gl + r - shift;                // node index in this direction's coordinates
        const int j = rev ? Nb - 1 - q : q;              // forward node index
        const bool ok = q >= 0 && q < Nb;
        st.m[r] = (q == 0) ? 1.f : 0.f;                  // virtual state: all mass on the first node (gram_ctc.py:144)
        st.e[r] = (q == 0) ? 0.f : SENT;
        if (ok) st.valid |= (1u << r);
        int ci = 0;
        bool open = false;
        if (ok) {
            if constexpr (!GRAM) {
                if (j & 1) {
                    const int i = j >> 1;
                    ci = 1 + i;
                    if (!rev) open = (i >= 1) && (lab[i] != lab[i - 1]);
                    else open = (i + 1 < Lb) && (lab[i + 1] != lab[i]);
                }
            } else {
                const int i = j / 3, type = j % 3;
                if (type == 1) {
                    ci = 1 + i;
                    if (!rev) open = (i >= 1) && (lab[i] != lab[i - 1]);
                    else open = (i + 1 < Lb) && (lab[i + 1] != lab[i]);
                } else if (type == 2) {
                    ci = 1 + d.Lmax + i;                 // a dead bigram (id -1) has emission probability 0 there
                    if (!rev) open = (i >= 2) && (big[i] != big[i - 2]);
                    else open = (i + 2 < Lb) && (big[i + 2] != big[i]);
                }
            }
        }
        st.ci[r] = ci;
        st.openoff[r] = open ? 0.f : SENT;
        if constexpr (K == 1 && GRAM) {
            // predecessor table of the header comment, as lanes back; the starred edge only when `open`
            const int t3 = (K * gl + r) % 3;             // position type in this direction's coordinates
            if (!rev) {
                st.dk[0] = t3 == 2 ? 5 : 1;
                st.dk[1] = t3 == 2 ? 7 : 2;
                st.dk[2] = t3 == 0 ? 0 : (open ? (t3 == 1 ? 3 : 6) : 0);
            } else {
                st.dk[0] = t3 == 2 ? 2 : 1;
                st.dk[1] = t3 == 0 ? 5 : (t3 == 1 ? 2 : 7);
                st.dk[2] = t3 == 0 ? 0 : (open ? (t3 == 1 ? 6 : 3) : 0);
            }
        }
    }
}

struct SmemPlan {
    size_t lp_elems, bnd_elems, none_elems;      // float2 elements
    size_t off_bars, off_red, total;
    int nbars;
};

__host__ __device__ inline SmemPlan plan_smem(int Wlp, int W, int S, int PAD, int CH) {
    SmemPlan p;
    p.lp_elems = (size_t)S * CH * Wlp;
    p.bnd_elems = (size_t)(W > 1 ? W - 1 : 1) * S * CH * PAD;
    p.bnd_elems = (p.bnd_elems + 1) & ~(size_t)1;                      // keep 16-byte alignment of what follows
    p.none_elems = ((size_t)CH * PAD + 1) & ~(size_t)1;
    p.nbars = 2 * S + S * (W > 1 ? W - 1 : 0);
    size_t o = (p.lp_elems + p.bnd_elems + p.none_elems) * sizeof(float2);
    p.off_bars = align_up(o, 16);
    o = p.off_bars + (size_t)p.nbars * sizeof(uint64_t);
    p.off_red = o;
    o += 4 * sizeof(float);
    p.total = o;
    return p;
}

// MAXW bounds the compute warps of an instantiation, so that small lattices (the common case) are not
// compiled under the register cap a large CTA implies.
template <int K, bool GRAM, int MAXW, int CH>
__global__ void __launch_bounds__(32 * (MAXW + 1)) lattice_kernel(LatticeParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int PAD = Geo<K, GRAM>::PAD;
    const ProblemDesc &d = p.d;
    if ((int)blockIdx.x >= 2 * d.B) {                      // ---- symbol-table CTAs (prep.cuh); none in a `second` launch ----
        prep_utterance(d, p.w, p.ws, (int)blockIdx.x - 2 * d.B, reinterpret_cast<int *>(smem_raw));
        return;
    }
    const int b = blockIdx.x >> 1;
    const int dir = blockIdx.x & 1;                        // 0: alpha, 1: beta
    const int W = p.W, S = p.S;
    // warps [0,W): recursion, warp W: I/O.  Read through a shuffle so that the compiler knows the value is
    // warp-uniform: every branch below is then a uniform branch, and the recursion's shuffles need no divergence
    // check (a BRA.DIV per shuffle otherwise, each one a scheduling barrier inside the unrolled chunk).
    const int w = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31;
    const bool io = (w == W);
    UttInfo *ui = reinterpret_cast<UttInfo *>(p.ws + p.w.off_utt) + b;
    WsHeader *hdr = reinterpret_cast<WsHeader *>(p.ws + p.w.off_hdr);

    const int Tb = __shfl_sync(0xffffffffu, utt_input_length(d, b), 0);
    const int Lb = __shfl_sync(0xffffffffu, utt_label_length(d, b), 0);
    const int Nb = (GRAM ? 3 : 2) * Lb + 1;

    const SmemPlan sp = plan_smem(p.w.W, W, S, PAD, CH);
    float2 *f2base = reinterpret_cast<float2 *>(smem_raw);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + sp.off_bars);
    float *red = reinterpret_cast<float *>(smem_raw + sp.off_red);
    DirPipe pp;
    pp.lp = smem_u32(f2base);
    pp.bnd = pp.lp + (uint32_t)(sp.lp_elems * sizeof(float2));
    pp.bnd_none = pp.bnd + (uint32_t)(sp.bnd_elems * sizeof(float2));
    pp.full = bars;
    pp.consumed = pp.full + S;
    pp.ready = pp.consumed + S;

    if (threadIdx.x == 0) {
        for (int i = 0; i < sp.nbars; ++i) mbar_init(&bars[i], 1u);      // every barrier has exactly one arriver
        mbar_init_fence();
    }
    for (int i = threadIdx.x; i < CH * PAD; i += blockDim.x)
        f2base[sp.lp_elems + sp.bnd_elems + i] = make_float2(0.f, SENT);
    __syncthreads();

    float2 *av = reinterpret_cast<float2 *>(p.ws + p.w.off_av) + (size_t)b * d.T * p.w.Np;
    float2 *bv = reinterpret_cast<float2 *>(p.ws + p.w.off_bv) + (size_t)b * d.T * p.w.Np;
    if (Tb > 0) {
        UttCtx c;
        c.lp_g = reinterpret_cast<const float2 *>(p.ws + p.w.off_lp) + (size_t)b * d.T * p.w.W;
        c.out_g = dir == 0 ? av : bv;
        c.Wlp = p.w.W; c.Np = p.w.Np; c.Nb = Nb; c.W = W; c.S = S; c.boff = p.w.boff;
        if (io) {
            if (dir == 0) io_direction<false, CH>(pp, c, 0, Tb, lane, p.ws, p.w, b, d.concurrent != 0, &hdr->stalled);
            else          io_direction<true, CH>(pp, c, Tb - 1, Tb, lane, p.ws, p.w, b, d.concurrent != 0, &hdr->stalled);
        } else {
            LaneState<K, GRAM> st;
            init_lane<K, GRAM>(st, d, b, Lb, Nb, dir == 1, 32 * w + lane);
            if (dir == 0) run_direction<K, GRAM, false, CH>(st, pp, c, 0, Tb, w, lane);         // alpha: frames 0 .. Tb-1
            else          run_direction<K, GRAM, true, CH>(st, pp, c, Tb - 1, Tb, w, lane);     // beta:  frames Tb-1 .. 0
        }
    }
    if (dir == 1) {                                        // the beta CTA is done
        __syncthreads();
        return;
    }
    __threadfence_block();
    __syncthreads();

    // ---- P = sum of alpha over the final nodes at the last frame (gram_ctc.py:279; SURVEY 8a "end") ----
    if (threadIdx.x == 0) {
        float loss;
        bool feas;
        float Ph = -SENT, Pl = 0.f;                       // exponent +1e30: every posterior becomes 0
        if (Tb <= 0) {                                   // no frames: P = 1 iff there is nothing to emit
            feas = (Lb == 0);
            if (feas) { Ph = 0.f; Pl = 1.f; }
            loss = feas ? 0.f : 1e10f;
        } else {
            const float2 *last = av + (size_t)(Tb - 1) * p.w.Np;
            const int nfin = GRAM ? 3 : 2;
            float fm[3], fe[3];
            float pe = SENT;
            for (int i = 0; i < 3; ++i) { fm[i] = 0.f; fe[i] = SENT; }
            for (int i = 0; i < nfin; ++i) {
                const int j = Nb - 1 - i;
                if (j >= 0) { const float2 v = last[j]; fm[i] = v.x; fe[i] = v.y; }
                pe = fmaxf(pe, fe[i]);
            }
            double sum = 0.0;
            for (int i = 0; i < nfin; ++i)
                if (fe[i] > SENT_TEST || fm[i] != fm[i]) sum += (double)fm[i] * exp2((double)(fe[i] - pe));
            feas = !(sum <= 0.0) && (pe > SENT_TEST || sum != sum);      // a NaN stays a NaN loss (train.py NaN guard)
            if (feas) {
                const double total = (double)pe + log2(sum);             // log2 P
                int ex = 0;
                const double mant = 2.0 * frexp(sum, &ex);               // sum = mant * 2^(ex-1), mant in [1,2)
                Ph = pe + (float)(ex - 1);
                Pl = (float)(1.0 / mant);                                // P = 2^Ph / Pl
                loss = (float)(-total * LN2_D);
            } else {
                loss = 1e10f;                            // what the reference returns (SURVEY.md 8a quirks)
            }
        }
        if (*reinterpret_cast<volatile unsigned *>(&hdr->stalled) != 0u) loss = __int_as_float(0x7fc00000);      // see kPollLimit
        ui->Ph = Ph; ui->Pl = Pl; ui->loss = loss; ui->infeasible = feas ? 0 : 1;
        p.loss_per_utt[b] = p.second ? __ldcg(p.loss_per_utt + b) + loss : loss;     // joint: Gram-CTC loss + CTC loss
        // ---- the last CTA reduces the batch in a fixed order (gram_ctc.py:280-281) ----
        __threadfence();
        const unsigned done = atomicAdd(p.second ? &hdr->k2b_done : &hdr->k2_done, 1u) + 1u;
        red[0] = (done == (unsigned)d.B) ? 1.f : 0.f;
    }
    __syncthreads();
    if (red[0] != 0.f && w == 0) {
        __threadfence();
        double acc = 0.0;
        for (int i = lane; i < d.B; i += 32) acc += (double)__ldcg(p.loss_per_utt + i);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (*reinterpret_cast<volatile unsigned *>(&hdr->stalled) != 0u) acc = (double)__int_as_float(0x7fc00000);
        if (lane == 0) *p.loss_reduced = (float)(acc * (double)p.loss_scale);
    }
}

using LatticeKernel = void (*)(LatticeParams);

// the instantiation with MAXW compute warps and the chunk length CH out of CHS, or nullptr
template <int K, bool GRAM, int MAXW, int... CHS>
LatticeKernel with_chunk(int CH) {
    LatticeKernel kern = nullptr;
    ((kern = CH == CHS ? lattice_kernel<K, GRAM, MAXW, CHS> : kern), ...);
    return kern;
}
template <int K, bool GRAM>
LatticeKernel any_tier(int W, int CH) {
    if (W <= 3) return with_chunk<K, GRAM, 3, 16>(CH);
    if (W <= 7) return with_chunk<K, GRAM, 7, 16, 8, 4>(CH);
    return with_chunk<K, GRAM, kMaxWarpsPerDir, 8, 4>(CH);
}
// The instantiated kernels: exactly the (K, W, CH) that launch_lattice's plan can reach.  Up to 3 warps the chunk is
// always 16 frames (CHmin); a chunk starts at 8 frames beyond 7 warps or 3 nodes per lane; CTC K = 4 means more than
// 512 nodes, so W >= 5; Gram-CTC K = 6 means more than 1536 nodes, so W >= 9.  nullptr: no kernel for the plan.
LatticeKernel lattice_kernel_for(int kind, int K, int W, int CH) {
    if (kind == 0) {
        if (K == 2) return any_tier<2, false>(W, CH);
        if (K == 4 && W > 3)
            return W <= 7 ? with_chunk<4, false, 7, 8, 4>(CH) : with_chunk<4, false, kMaxWarpsPerDir, 8, 4>(CH);
        return nullptr;
    }
    if (K == 1) return any_tier<1, true>(W, CH);
    if (K == 3) return any_tier<3, true>(W, CH);
    if (K == 6 && W > 7) return with_chunk<6, true, kMaxWarpsPerDir, 8, 4>(CH);
    return nullptr;
}

constexpr size_t kLatticeSmemBudget = 224 * 1024;

}  // namespace

WsLayout ctc_view_of_joint(const WsLayout &w) {
    WsLayout v = w;                 // same emission rows (v.W), header, progress counters
    v.kind = 0; v.joint = 0;
    v.Nmax = w.Nmax2; v.Np = w.Np2; v.boff = 1;
    v.off_av = w.off_av2; v.off_bv = w.off_bv2; v.off_utt = w.off_utt2;
    return v;
}

int lattice_max_nodes(int kind) { return kind == 0 ? 32 * 4 * kMaxWarpsPerDir - 3 : 32 * 6 * kMaxWarpsPerDir; }      // - 3: phantom nodes of the 4-node mapping

cudaError_t launch_lattice(LatticeParams p, cudaStream_t stream, int *status, bool concurrent, size_t *smem_out,
                           bool launch) {
    *status = 0;
    const int kind = p.d.kind;
    const int Nmax = p.w.Nmax;
    // nodes per lane: two for the usual lattices (one recursion warp per SM sub-partition is the measured optimum at
    // L = 80); four once the lattice would need more than eight warps (measured at L = 320, 11 warps: 1.51 -> 1.09 ms
    // for the forward pass at T = 3200 with K = 4 and 4-frame chunks; K = 8 is slower again, profiles/r2_lattice_sweep.txt)
    int K;
    if (kind == 0) K = (Nmax <= 32 * 2 * 8) ? 2 : 4;
    else K = (Nmax <= 32 * kGenericMaxWarps) ? 1 : ((Nmax <= 32 * 3 * kMaxWarpsPerDir) ? 3 : 6);
    const int W = (Nmax + (kind == 0 && K == 4 ? 3 : 0) + 32 * K - 1) / (32 * K);      // + the reversed direction's phantom nodes
    if (W > kMaxWarpsPerDir) { *status = 2; return cudaSuccess; }
    const int PAD = kind == 0 ? 2 : 7;
    // chunk length: the longest one instantiated for this W whose ring of W + 3 stages fits
    // (next to the softmax/gather kernel a small lattice gets one stage less: shared memory taken here is taken
    // from that kernel's ring, and measured on the bench workload the shallower ring is the better trade)
    const int ahead = (concurrent && W <= 3) ? 2 : 3;
    const int want = W + ahead < kMaxStages ? W + ahead : kMaxStages;
    // (a fully unrolled 16-frame chunk of a four-node step is ~48 KB of code: measured 309 cycles per frame against 154
    // with 8-frame chunks -- instruction fetch, not arithmetic)
    int CH = (W <= 7 && K <= 3) ? 16 : 8;
    const int CHmin = W <= 3 ? 16 : 4;
    // next to the softmax/gather kernel every byte here is taken from that kernel's ring: stay below 64 KB if a
    // shorter chunk allows it
    const size_t budget = concurrent ? (size_t)64 * 1024 : kLatticeSmemBudget;
    while (CH > CHmin && plan_smem(p.w.W, W, want, PAD, CH).total > budget) CH >>= 1;
    int S = want;
    while (S > 2 && plan_smem(p.w.W, W, S, PAD, CH).total > kLatticeSmemBudget) --S;
    const SmemPlan sp = plan_smem(p.w.W, W, S, PAD, CH);
    if (sp.total > kLatticeSmemBudget) { *status = 2; return cudaSuccess; }
    size_t smem = sp.total;
    const size_t prep = p.second ? 0 : prep_smem_bytes(kind, p.d.Lmax, p.w.nwords);
    if (prep > smem) smem = prep;
    if (smem > 227 * 1024) { *status = 2; return cudaSuccess; }
    const LatticeKernel kern = lattice_kernel_for(kind, K, W, CH);
    if (!kern) { *status = 2; return cudaSuccess; }
    p.W = W; p.S = S;
    if (smem_out) *smem_out = smem;
    if (!launch) return cudaSuccess;
    // the SM's L1/shared split is chosen per kernel: ask for the maximum so that a lattice CTA and a ring CTA of the
    // softmax/gather kernel (which asks for the same) can share an SM
    cudaError_t e = ensure_dynamic_smem(reinterpret_cast<const void *>(kern), smem);
    if (e != cudaSuccess) return e;
    kern<<<(p.second ? 2 : 3) * p.d.B, 32 * (p.W + 1), smem, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace b200ctc
