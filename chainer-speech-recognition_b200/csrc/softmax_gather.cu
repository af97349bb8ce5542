// softmax_gather.cu -- kernel 1: fused log-softmax statistics + label gather + optional greedy argmax.
//
// Replaces, in the reference (asr/loss/gram_ctc.py):
//   _softmax :18-21 and _log_matrix :48-57 over the whole (T,B,V) tensor (two extra 717 MB arrays at
//   B=64,T=800,V=3500) and the per-frame `xp.take(y, index)` of loop 1/2 (:155,:175).
// Kernel 1 reads each activation row exactly once and writes, per frame, ONE float (the log2
// normaliser) plus the gathered probabilities, as (mantissa, exponent) pairs, of the <= 1+2*Lmax symbols the lattice can emit.
// No (T,B,V) log-probability tensor is ever materialised.
//
// One warp per frame, 128-bit loads, online (max, sum) per lane, warp-shuffle reduction.
#include "common.cuh"
#include "kernels.h"
#include "row_ring.cuh"

namespace b200ctc {

namespace {

constexpr int kWarpsPerCta = 8;
constexpr int kUnroll = 4;

// ---------------------------------------------------------------------------------------------
// kernel 1
// ---------------------------------------------------------------------------------------------
// Ticket -> frame.  Tickets walk the utterances' frames from BOTH ends towards the middle (slice 0 = frame 0 of
// every utterance, slice 1 = frame T-1, slice 2 = frame 1, ...): the lattice kernel may run concurrently with this
// one, its alpha CTAs consume frames in ascending and its beta CTAs in descending order, so each direction finds
// the rows it needs next already written (common.cuh, signal_frame_done).  Independent of the memory layout: a
// row is one contiguous 4*V-byte read either way.
// (Tried and dropped: walking every utterance from ITS two ends, in groups ordered by decreasing length so that the
// rows produced last belong to the shortest utterances.  The exposed lattice tail shrank from 33 to 27 us, but this
// kernel lost 8 us to the scattered row order -- no net gain, measured on per-kernel timelines.)
__device__ __forceinline__ void frame_of_ticket(unsigned f, int B, int T, bool two_ended, int &b, int &t) {
    const int slice = (int)(f / (unsigned)B);
    b = (int)(f % (unsigned)B);
    t = !two_ended ? slice : (slice & 1) ? (T - 1 - (slice >> 1)) : (slice >> 1);
}

struct RowStat {
    float m;      // running max (raw activation units)
    float s;      // running sum of 2^((x - m) * log2 e)
    float bv;     // best value for argmax (NaN-aware)
    int bi;       // its index
};

template <bool ARGMAX>
__device__ __forceinline__ void fold(RowStat &st, float x, int idx) {
    if (ARGMAX) {
        // numpy.argmax: first maximum wins, NaN is maximal
        const bool better = (x > st.bv) || ((x != x) && (st.bv == st.bv)) || (st.bi == 0x7fffffff);
        if (better) { st.bv = x; st.bi = idx; }
    }
}

template <bool ARGMAX>
__device__ __forceinline__ void fold4(RowStat &st, const float4 &v, int idx) {
    const float cm = fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w));
    if (cm > st.m) {
        st.s *= ex2_approx((st.m - cm) * LOG2E_HI);
        st.m = cm;
    }
    const float c = st.m == -INFINITY ? 0.f : -st.m * LOG2E_HI;        // nothing finite seen yet: every term is 2^-inf = 0
    st.s += (ex2_approx(fmaf(v.x, LOG2E_HI, c)) + ex2_approx(fmaf(v.y, LOG2E_HI, c))) +
            (ex2_approx(fmaf(v.z, LOG2E_HI, c)) + ex2_approx(fmaf(v.w, LOG2E_HI, c)));
    fold<ARGMAX>(st, v.x, idx);
    fold<ARGMAX>(st, v.y, idx + 1);
    fold<ARGMAX>(st, v.z, idx + 2);
    fold<ARGMAX>(st, v.w, idx + 3);
}

template <bool ARGMAX>
__device__ __forceinline__ void fold1(RowStat &st, float x, int idx) {
    if (x > st.m) {
        st.s *= ex2_approx((st.m - x) * LOG2E_HI);
        st.m = x;
    }
    st.s += ex2_approx((x - st.m) * LOG2E_HI);
    fold<ARGMAX>(st, x, idx);
}

// numpy.argmax over the warp from each lane's (best value, its index): lane order is not index order, so reduce on
// (value, index) with "NaN beats all, then larger value, then smaller index".  Returns the index, warp-uniform.
__device__ __forceinline__ int warp_argmax(float bv, int bi) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        const bool onan = (ov != ov), mnan = (bv != bv);
        bool take;
        if (onan || mnan) take = onan && (!mnan || oi < bi);
        else take = (ov > bv) || (ov == bv && oi < bi);
        if (take) { bv = ov; bi = oi; }
    }
    return bi;
}

// Scan one row with the whole warp.  Returns warp-uniform (max, log2 normaliser, argmax).
template <bool ARGMAX, bool SOFTMAX>
__device__ __forceinline__ void scan_row(const float *__restrict__ row, int V, int lane, float &row_max,
                                         float &lse2, int &amax) {
    RowStat st;
    st.m = -INFINITY; st.s = 0.f; st.bv = -INFINITY; st.bi = 0x7fffffff;
    // a row that is not 16-byte aligned starts with up to 3 scalar elements
    const int mis = (int)((reinterpret_cast<uintptr_t>(row) >> 2) & 3);
    const int head = mis ? min(V, 4 - mis) : 0;
    if (lane < head) {
        if (SOFTMAX) fold1<ARGMAX>(st, row[lane], lane);
        else fold<ARGMAX>(st, row[lane], lane);
    }
    const float4 *row4 = reinterpret_cast<const float4 *>(row + head);
    const int n4 = (V - head) >> 2;
    int i = lane;
    for (; i + 32 * (kUnroll - 1) < n4; i += 32 * kUnroll) {
        float4 v[kUnroll];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) v[u] = __ldg(row4 + i + 32 * u);
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            if (SOFTMAX) fold4<ARGMAX>(st, v[u], head + 4 * (i + 32 * u));
            else {
                fold<ARGMAX>(st, v[u].x, head + 4 * (i + 32 * u));
                fold<ARGMAX>(st, v[u].y, head + 4 * (i + 32 * u) + 1);
                fold<ARGMAX>(st, v[u].z, head + 4 * (i + 32 * u) + 2);
                fold<ARGMAX>(st, v[u].w, head + 4 * (i + 32 * u) + 3);
            }
        }
    }
    for (; i < n4; i += 32) {
        const float4 v = __ldg(row4 + i);
        if (SOFTMAX) fold4<ARGMAX>(st, v, head + 4 * i);
        else {
            fold<ARGMAX>(st, v.x, head + 4 * i);
            fold<ARGMAX>(st, v.y, head + 4 * i + 1);
            fold<ARGMAX>(st, v.z, head + 4 * i + 2);
            fold<ARGMAX>(st, v.w, head + 4 * i + 3);
        }
    }
    const int tail0 = head + 4 * n4;
    if (tail0 + lane < V) {
        if (SOFTMAX) fold1<ARGMAX>(st, row[tail0 + lane], tail0 + lane);
        else fold<ARGMAX>(st, row[tail0 + lane], tail0 + lane);
    }
    if (SOFTMAX) {
        const float m = warp_max(st.m);
        float s = st.s * ex2_approx((st.m - m) * LOG2E_HI);     // lanes that saw nothing: 0 * 2^-inf = 0
        if (st.m == -INFINITY) s = 0.f;
        s = warp_sum(s);
        row_max = m;
        lse2 = s;                                                // caller finishes with split_lse2(row_max, lse2)
    }
    if (ARGMAX) amax = warp_argmax(st.bv, st.bi);
}

template <bool ARGMAX>
__global__ void __launch_bounds__(kWarpsPerCta * 32) softmax_gather_kernel(ProblemDesc d, WsLayout w,
                                                                          unsigned char *ws, int64_t *argmax_out) {
    const int lane = threadIdx.x & 31;
    WsHeader *hdr = reinterpret_cast<WsHeader *>(ws + w.off_hdr);
    float2 *lse_out = reinterpret_cast<float2 *>(ws + w.off_lse);
    float2 *lp_out = reinterpret_cast<float2 *>(ws + w.off_lp);
    const unsigned frames = (unsigned)d.B * (unsigned)d.T;
    // The "row written" signal of a frame is a release at GPU scope, i.e. it waits for the warp's outstanding stores.
    // It is therefore sent one frame late, just before the NEXT frame's stores: by then the previous frame's stores
    // have long been acknowledged and the release costs next to nothing.
    int pend_b = -1, pend_t = 0;
    for (;;) {
        // work queue: one ticket per frame, handed out in memory order of the activations, so that the
        // (variable-length) valid frames spread evenly over the warps whatever the batch layout is
        unsigned f = 0;
        if (lane == 0) f = atomicAdd(&hdr->k1_ticket, 1u);
        f = __shfl_sync(0xffffffffu, f, 0);
        if (f >= frames) break;
        int b, t;
        frame_of_ticket(f, d.B, d.T, d.concurrent != 0, b, t);
        // Lengths and label ids are read with plain (coherent) loads here, not through the read-only path of
        // utt_input_length() / EmissionColumns: with those ptxas issues only two of the four row loads of scan_row's
        // unrolled step up front, and this kernel took 8 % longer (V = 20000, B200).
        const bool valid = t < clamp_length(d.input_lengths ? d.input_lengths[b] : d.T, d.T);
        if (!valid && !ARGMAX) continue;
        const float *row = d.acts + (int64_t)t * d.stride_t + (int64_t)b * d.stride_b;
        float row_max = 0.f, lse2 = 0.f;
        int amax = 0;
        if (valid) scan_row<ARGMAX, true>(row, d.V, lane, row_max, lse2, amax);
        else scan_row<ARGMAX, false>(row, d.V, lane, row_max, lse2, amax);
        if (ARGMAX && lane == 0) argmax_out[(size_t)b * d.T + t] = amax;
        if (!valid) continue;
        float la, lb;
        split_lse2(row_max, lse2, la, lb);
        if (lane == 0 && pend_b >= 0 && d.concurrent) signal_frame_done(ws, w, pend_b, pend_t);
        if (lane == 0) lse_out[(size_t)b * d.T + t] = grad_normaliser(row_max, la, lb);
        // gather the emission row (WsLayout::W, as EmissionColumns maps it)
        const int Lb = clamp_length(d.label_lengths ? d.label_lengths[b] : d.Lmax, d.Lmax);
        float2 *lprow = lp_out + ((size_t)b * d.T + t) * w.W;
        const int32_t *lab = d.labels + (size_t)b * d.Lmax;
        const int32_t *big = d.kind == 1 ? d.bigrams + (size_t)b * d.Lmax : nullptr;
        const int ncol = 1 + (d.kind == 1 ? d.Lmax + Lb : Lb);
        for (int c = lane; c < ncol; c += 32) {
            int sym;
            if (c == 0) sym = d.blank;
            else if (c <= d.Lmax) sym = (c - 1 < Lb) ? lab[c - 1] : -1;
            else sym = big[c - 1 - d.Lmax];
            float2 v = make_float2(0.f, SENT);
            if (sym >= 0 && sym < d.V) v = emission_pair(__ldg(row + sym), la, lb);
            lprow[c] = v;
        }
        __syncwarp();
        pend_b = b; pend_t = t;
    }
    if (lane == 0 && pend_b >= 0 && d.concurrent) signal_frame_done(ws, w, pend_b, pend_t);
}

// ---------------------------------------------------------------------------------------------
// kernel 1, TMA row-ring variant (see row_ring.cuh): the row sits in shared memory, so the statistics
// take two cheap passes (max/argmax, then sum of exponentials) and the label gather reads shared
// memory instead of going back to L2.
// ---------------------------------------------------------------------------------------------
// "Row written" signals for a concurrently running lattice kernel (common.cuh, signal_frame_done).  A signal must
// be a release at GPU scope, and such a fence costs ~1.5 us on this part whatever is outstanding -- per row and
// consumer warp that was 28 us of a 105 us kernel.  So the consumers only note finished rows in a small
// shared-memory FIFO (CTA-scope ordering, cheap) and one extra warp drains all FIFOs with ONE GPU-scope fence per
// sweep, then bumps the progress counters (the __syncthreads / thread 0 fences / atomic pattern of a grid barrier).
constexpr int kK1Consumers = 10;
constexpr int kK1Threads = 32 * (1 + kK1Consumers + 1);   // producer + consumers + signal warp
constexpr int kGatherRegs = 4;                         // emitted ids per lane on the early-release path (<= 128 columns)
constexpr int kFifoDepth = 4;
constexpr int kLenCache = 2048;                        // utterances whose lengths the ring kernel keeps in shared memory
struct SignalFifo {
    int2 entry[kK1Consumers][kFifoDepth];            // (b, t); b < 0 = this consumer is done
    unsigned head[kK1Consumers];                     // rows pushed by consumer c
    unsigned tail[kK1Consumers];                     // rows taken by the signal warp
};
constexpr size_t kFifoBytes = (sizeof(SignalFifo) + 127) / 128 * 128;

// consumer warp c, after a __syncwarp() that follows the row's global stores (lane 0 only)
__device__ __forceinline__ void fifo_push(SignalFifo *f, int c, unsigned &pushed, int b, int t) {
    volatile unsigned *tail = &f->tail[c];
    while (pushed - *tail >= (unsigned)kFifoDepth) __nanosleep(64);
    f->entry[c][pushed % kFifoDepth] = make_int2(b, t);
    __threadfence_block();                             // row stores and entry before the head update
    *reinterpret_cast<volatile unsigned *>(&f->head[c]) = ++pushed;
}

__device__ __forceinline__ void signal_warp(SignalFifo *f, int nc, int lane, unsigned char *ws, const WsLayout &w) {
    unsigned taken = 0;
    bool done = lane >= nc;
    for (;;) {
        bool have = false;
        int2 e = make_int2(-1, 0);
        if (!done && *reinterpret_cast<volatile unsigned *>(&f->head[lane]) != taken) {
            __threadfence_block();
            const volatile int *ep = reinterpret_cast<volatile int *>(&f->entry[lane][taken % kFifoDepth]);
            e.x = ep[0];
            e.y = ep[1];
            have = true;
        }
        if (__any_sync(0xffffffffu, have)) {
            // release at GPU scope: one MEMBAR.ALL.GPU for the warp, then the REDs.  Not __threadfence(): that is a
            // sequentially consistent fence plus an L1 invalidation (CCTL.IVALL), which would throw the consumers'
            // cached label tables away every time.
            if (have) {
                if (e.x < 0) done = true;
                else signal_frame_done(ws, w, e.x, e.y);
                *reinterpret_cast<volatile unsigned *>(&f->tail[lane]) = ++taken;
            }
        } else {
            if (__all_sync(0xffffffffu, done)) break;
            __nanosleep(256);
        }
    }
}

// Sum of exponentials of a staged row WITHOUT a running maximum: every lane takes the largest of its first four
// elements as its own reference (an integer in log2 units), so the loop body is load / FFMA / MUFU.EX2 / FADD with
// four independent accumulators -- no loop-carried maximum, no rescaling branch.  The references are aligned at the
// end with exact powers of two.  A reference that is not the maximum only moves the intermediate sums along the
// float32 exponent range (no precision is lost); what it cannot absorb is an element more than ~2^100 above a
// lane's reference -- the sum then overflows to +inf (or a NaN / all -inf row shows up), fast_row_scan reports it
// (warp-uniform) and the caller redoes the row with the running-maximum scan below.  Split in two so that the ring
// slot can be handed back between the scan (which needs the row) and the warp reductions (which do not).
__device__ __forceinline__ bool fast_row_scan(const float4 *__restrict__ row4, int n4, int lane, float &ref, float &sl) {
    float nr = 0.f;
    ref = -INFINITY;
    if (lane < n4) {
        const float4 v = row4[lane];
        const float cm = fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w));       // NaNs are dropped here and caught by the sum
        if (cm > -INFINITY) { ref = rintf(cm * LOG2E_HI); nr = -ref; } else ref = 0.f;
    }
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll 4
    for (int i = lane; i < n4; i += 32) {
        const float4 v = row4[i];
        s0 += ex2_approx(fmaf(v.x, LOG2E_HI, nr));
        s1 += ex2_approx(fmaf(v.y, LOG2E_HI, nr));
        s2 += ex2_approx(fmaf(v.z, LOG2E_HI, nr));
        s3 += ex2_approx(fmaf(v.w, LOG2E_HI, nr));
    }
    sl = (s0 + s1) + (s2 + s3);
    // every lane's partial sum must be an ordinary number (NaN fails both comparisons) with room for 32 of them to
    // be added, its reference an exactly representable integer; and the row must have some probability mass
    const bool lane_ok = sl >= 0.f && sl < 1e30f && (ref == -INFINITY || fabsf(ref) < 4194304.f);
    return __all_sync(0xffffffffu, lane_ok) && __any_sync(0xffffffffu, sl > 0.f);
}
// The sums above are of 2^(x*LOG2E_HI); emission_pair adds x*LOG2E_LO to every symbol, so the normaliser gets the
// row maximum's share of it, m*LOG2E_LO with m ~ R/LOG2E_HI, as split_lse2 gives it (2e-5 in log2 p at |logits| ~ 1000).
// m is returned for grad_normaliser.
__device__ __forceinline__ void fast_row_finish(float ref, float sl, float &la, float &lb, float &m) {
    const float R = warp_max(ref);
    const float S = warp_sum(sl * ex2_approx(ref - R));                  // ref - R: integer <= 0 (or -inf for an empty lane)
    const float lg = log2f(S);
    const float a = R + lg;                                              // TwoSum(R, lg)
    const float bb = a - R;
    m = R * (1.f / LOG2E_HI);
    la = a;
    lb = fmaf(m, LOG2E_LO, (R - (a - bb)) + (lg - bb));
}

template <bool ARGMAX>
__global__ void __launch_bounds__(kK1Threads, 1) softmax_gather_ring_kernel(ProblemDesc d, WsLayout w,
                                                                              unsigned char *ws,
                                                                              int64_t *argmax_out, RingLayout rl) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Ring ring = ring_setup(smem_raw, rl);
    const uint64_t l2pol = l2_policy_evict_first();
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    WsHeader *hdr = reinterpret_cast<WsHeader *>(ws + w.off_hdr);
    const unsigned frames = (unsigned)d.B * (unsigned)d.T;
    SignalFifo *fifo = reinterpret_cast<SignalFifo *>(smem_raw + rl.off_extra);
    const bool signalling = d.concurrent != 0;
    if (threadIdx.x < kK1Consumers) { fifo->head[threadIdx.x] = 0u; fifo->tail[threadIdx.x] = 0u; }
    // clamped lengths of every utterance, once per CTA: the producer then turns a ticket into copies without a round
    // trip to L2 in between (that round trip, per batch of 8 rows, was 15 % of its time)
    int *len_sm = reinterpret_cast<int *>(smem_raw + rl.off_extra + kFifoBytes);
    const bool len_cached = d.B <= kLenCache;
    if (len_cached) {
        for (int i = threadIdx.x; i < d.B; i += blockDim.x) {
            len_sm[i] = utt_input_length(d, i);
            len_sm[d.B + i] = utt_label_length(d, i);
        }
    }
    __syncthreads();
    if (warp == kK1Consumers + 1) {                     // ===== signal warp =====
        if (signalling) signal_warp(fifo, ring.nc, lane, ws, w);
        return;
    }

    if (warp == 0) {
        // ===== producer (lane i owns frame i of the current batch) =====
        unsigned q = 0;
        // one batch of tickets -> rows into the ring; returns false when the queue is exhausted
        auto issue_batch = [&](unsigned base) -> bool {
            if (base >= frames) return false;
            const unsigned f = base + (unsigned)lane;
            int b = 0, t = 0, Lb = 0;
            bool valid = false, need = false;
            if (lane < ring.batch && f < frames) {
                frame_of_ticket(f, d.B, d.T, d.concurrent != 0, b, t);
                int Tb;
                if (len_cached) { Tb = len_sm[b]; Lb = len_sm[d.B + b]; }
                else { Tb = utt_input_length(d, b); Lb = utt_label_length(d, b); }
                valid = t < Tb;
                need = valid || ARGMAX;
            }
            const unsigned mask = __ballot_sync(0xffffffffu, need);
            const unsigned myq = q + (unsigned)__popc(mask & ((1u << lane) - 1u));
            // every lane issues its row as soon as ITS slot is free, in whatever order the consumers hand slots back
            bool pending = need;
            while (__any_sync(0xffffffffu, pending)) {
                bool issued = false;
                if (pending && ring_slot_free(ring, myq)) {
                    const int s = (int)(myq % (unsigned)ring.slots);
                    // the 16-byte aligned span that covers the row (rows themselves only need 4-byte alignment)
                    const float *src = d.acts + (int64_t)t * d.stride_t + (int64_t)b * d.stride_b;
                    const int off = row_misalignment(src);
                    const uint32_t span = row_span_bytes(off, d.V);
                    ring.meta[s].b = b; ring.meta[s].t = t; ring.meta[s].kind = valid ? 0 : 1; ring.meta[s].off = off;
                    ring.meta[s].Lb = Lb;
                    ring_publish(ring, s, myq);
                    mbar_arrive_expect_tx(&ring.full[s], span);
                    // evict-first in L2 (common.cuh): measured 4 us off the forward pass
                    bulk_g2s_hint(ring.slot(s), src - off, span, &ring.full[s], l2pol);
                    pending = false;
                    issued = true;
                }
                if (!__any_sync(0xffffffffu, issued)) __nanosleep(40);
            }
            q += (unsigned)__popc(mask);
            return true;
        };
        // Batches of rows are drawn from a global ticket counter (variable-length utterances balance themselves; dealing
        // the batches round-robin instead was measured: the slowest CTA then finishes 8 % later).  Under a full-rate stream
        // one atomic on that hot address takes ~5 us to come back, so two tickets are kept in flight: the one a batch
        // needs was requested two batches ago.
        unsigned pa = 0, pb = 0;
        if (lane == 0) { pa = atomicAdd(&hdr->k1_ticket, (unsigned)ring.batch); pb = atomicAdd(&hdr->k1_ticket, (unsigned)ring.batch); }
        for (;;) {
            unsigned base = __shfl_sync(0xffffffffu, pa, 0);
            if (lane == 0 && base < frames) pa = atomicAdd(&hdr->k1_ticket, (unsigned)ring.batch);
            if (!issue_batch(base)) break;
            base = __shfl_sync(0xffffffffu, pb, 0);
            if (lane == 0 && base < frames) pb = atomicAdd(&hdr->k1_ticket, (unsigned)ring.batch);
            if (!issue_batch(base)) break;
        }
        ring_stop(ring, q, lane);
        return;
    }

    // ===== consumers =====
    float2 *lse_out = reinterpret_cast<float2 *>(ws + w.off_lse);
    float2 *lp_out = reinterpret_cast<float2 *>(ws + w.off_lp);
    if (warp - 1 >= ring.nc) return;                      // short ring: fewer active consumers (row_ring.cuh)
    unsigned pushed = 0;
    for (;;) {
        const unsigned q = ring_next_row(ring, lane);
        const int s = ring_acquire(ring, q);
        const RowMeta m = ring.meta[s];
        if (m.kind < 0) {                       // stop record: hand the slot back (the ring may be shorter than
            __syncwarp();                       // the number of consumers) and leave
            if (lane == 0) mbar_arrive(&ring.empty[s]);
            break;
        }
        float *slotf = reinterpret_cast<float *>(ring.slot(s));
        const float *row = slotf + m.off;                              // element v of the frame
        const float4 *row4 = reinterpret_cast<const float4 *>(slotf);  // the aligned span, float4 by float4
        const int n4 = (m.off + d.V + 3) >> 2;
        if (m.off != 0 || (d.V & 3) != 0) {
            // elements of the span outside the row: -inf, i.e. probability 0 and never a maximum
            if (lane < m.off) slotf[lane] = -INFINITY;
            if (m.off + d.V + lane < 4 * n4) slotf[m.off + d.V + lane] = -INFINITY;
            __syncwarp();
        }
        bool released = false;                  // the slot has already been handed back (early, see the gather)
        // Emitted ids of this lane's columns of the emission row (WsLayout::W), requested now so that their latency
        // hides behind the row scan
        int Lb = 0, ncol = 0;
        const EmissionColumns cols(d, m.b);
        int syms[kGatherRegs];
        bool early = false;
        if (m.kind == 0) {
            Lb = m.Lb;
            ncol = cols.count(Lb);
            early = ncol <= 32 * kGatherRegs;
            if (early) {
#pragma unroll
                for (int k = 0; k < kGatherRegs; ++k) syms[k] = (lane + 32 * k < ncol) ? cols.symbol(lane + 32 * k, Lb) : -1;
            }
        }
        float la = 0.f, lb = 0.f, mx = 0.f;
        float ref = 0.f, sl = 0.f;
        bool fast = false;
        if (!ARGMAX && m.kind == 0) fast = fast_row_scan(row4, n4, lane, ref, sl);
        if (!fast) {
            // one pass with a per-lane running (max, sum of 2^((x - max) * log2 e)) and the greedy index; a padded
            // frame (argmax only) skips the exponentials
            RowStat st;
            st.m = -INFINITY; st.s = 0.f; st.bv = -INFINITY; st.bi = 0x7fffffff;
            if (m.kind == 0) {
#pragma unroll 4
                for (int i = lane; i < n4; i += 32) fold4<ARGMAX>(st, row4[i], 4 * i - m.off);
            } else {
#pragma unroll 4
                for (int i = lane; i < n4; i += 32) {
                    const float4 v = row4[i];
                    fold<ARGMAX>(st, v.x, 4 * i - m.off);
                    fold<ARGMAX>(st, v.y, 4 * i - m.off + 1);
                    fold<ARGMAX>(st, v.z, 4 * i - m.off + 2);
                    fold<ARGMAX>(st, v.w, 4 * i - m.off + 3);
                }
            }
            if (ARGMAX) {
                const int bi = warp_argmax(st.bv, st.bi);
                // an element of the span in front of the row (index < 0, value -inf) can only "win" when every
                // element of the row is -inf, and numpy.argmax of such a row is 0
                if (lane == 0) argmax_out[(size_t)m.b * d.T + m.t] = bi < 0 ? 0 : bi;
            }
            if (m.kind == 0) {
                mx = warp_max(st.m);
                float sum = st.m == -INFINITY ? 0.f : st.s * ex2_approx((st.m - mx) * LOG2E_HI);
                sum = warp_sum(sum);
                split_lse2(mx, sum, la, lb);
            }
        }
        if (m.kind == 0) {
            float2 *lprow = lp_out + ((size_t)m.b * d.T + m.t) * w.W;
            if (early) {
                // The usual case.  Only the activations at the emitted ids are still needed from the row: fetch them,
                // hand the slot back to the producer, and only then do the arithmetic and the global stores.  A slot
                // held by a consumer is a row NOT in flight from HBM, and the ring is what covers the memory latency.
                float xv[kGatherRegs];
                bool ok[kGatherRegs];
#pragma unroll
                for (int k = 0; k < kGatherRegs; ++k) {
                    ok[k] = syms[k] >= 0 && syms[k] < d.V;
                    xv[k] = ok[k] ? row[syms[k]] : 0.f;
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&ring.empty[s]);
                released = true;
                if (fast) fast_row_finish(ref, sl, la, lb, mx);
                if (lane == 0) lse_out[(size_t)m.b * d.T + m.t] = grad_normaliser(mx, la, lb);
#pragma unroll
                for (int k = 0; k < kGatherRegs; ++k) {
                    const int cidx = lane + 32 * k;
                    if (cidx < ncol) lprow[cidx] = ok[k] ? emission_pair(xv[k], la, lb) : make_float2(0.f, SENT);
                }
            } else {
                if (fast) fast_row_finish(ref, sl, la, lb, mx);
                if (lane == 0) lse_out[(size_t)m.b * d.T + m.t] = grad_normaliser(mx, la, lb);
                for (int cidx = lane; cidx < ncol; cidx += 32) {
                    const int sym = cols.symbol(cidx, Lb);
                    float2 v = make_float2(0.f, SENT);
                    if (sym >= 0 && sym < d.V) v = emission_pair(row[sym], la, lb);
                    lprow[cidx] = v;
                }
            }
            __syncwarp();
            if (signalling && lane == 0) fifo_push(fifo, warp - 1, pushed, m.b, m.t);
        }
        __syncwarp();
        if (lane == 0 && !released) mbar_arrive(&ring.empty[s]);
    }
    if (signalling && lane == 0) fifo_push(fifo, warp - 1, pushed, -1, 0);
}

__global__ void __launch_bounds__(kWarpsPerCta * 32) argmax_kernel(const float *acts, int64_t stride_t,
                                                                  int64_t stride_b, int B, int T, int V,
                                                                  int64_t *argmax_out, int b_major) {
    const int lane = threadIdx.x & 31;
    const int warp_global = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
    const int warps_total = gridDim.x * kWarpsPerCta;
    const long long frames = (long long)B * T;
    for (long long f = warp_global; f < frames; f += warps_total) {
        int b, t;
        if (b_major) { b = (int)(f / T); t = (int)(f % T); }
        else { t = (int)(f / B); b = (int)(f % B); }
        const float *row = acts + (int64_t)t * stride_t + (int64_t)b * stride_b;
        float row_max, lse2;
        int amax = 0;
        scan_row<true, false>(row, V, lane, row_max, lse2, amax);
        if (lane == 0) argmax_out[(size_t)b * T + t] = amax;
    }
}

int grid_for_frames(long long frames) {
    long long ctas = (frames + kWarpsPerCta - 1) / kWarpsPerCta;
    const long long cap = (long long)sm_count() * 8;       // 8 CTAs x 8 warps = 64 resident warps per SM
    if (ctas > cap) ctas = cap;
    if (ctas < 1) ctas = 1;
    return (int)ctas;
}

}  // namespace

// Rows qualify for the TMA ring when at least kMinSlots of them (each with room for the 16-byte aligned span around a
// row that is only 4-byte aligned) fit in shared memory; base pointer and strides are in floats, so any of them do.
bool ring_usable(const void *base, const RingLayout &rl) {
    return (reinterpret_cast<uintptr_t>(base) & 3) == 0 && rl.slots >= kMinSlots;
}

cudaError_t launch_softmax_gather(const ProblemDesc &d, const WsLayout &w, void *ws, int64_t *argmax_out,
                                  size_t smem_reserve, cudaStream_t stream) {
    const long long frames = (long long)d.B * d.T;
    if (frames == 0) return cudaSuccess;
    unsigned char *wsb = static_cast<unsigned char *>(ws);
    const RingLayout rl = make_ring(ring_row_bytes(d.V), kFifoBytes + (d.B <= kLenCache ? 8 * (size_t)d.B : 0), smem_reserve, kK1Consumers);
    if (ring_usable(d.acts, rl)) {
        long long ctas = (frames + kTicketBatch - 1) / kTicketBatch;
        if (ctas > sm_count()) ctas = sm_count();
        if (ctas < 1) ctas = 1;
        cudaError_t e;
        if (argmax_out) {
            e = ensure_dynamic_smem(reinterpret_cast<const void *>(softmax_gather_ring_kernel<true>), rl.total);
            if (e != cudaSuccess) return e;
            softmax_gather_ring_kernel<true><<<(int)ctas, kK1Threads, rl.total, stream>>>(d, w, wsb, argmax_out, rl);
        } else {
            e = ensure_dynamic_smem(reinterpret_cast<const void *>(softmax_gather_ring_kernel<false>), rl.total);
            if (e != cudaSuccess) return e;
            softmax_gather_ring_kernel<false><<<(int)ctas, kK1Threads, rl.total, stream>>>(d, w, wsb, nullptr, rl);
        }
        return cudaGetLastError();
    }
    const int grid = grid_for_frames(frames);
    if (argmax_out)
        softmax_gather_kernel<true><<<grid, kWarpsPerCta * 32, 0, stream>>>(d, w, wsb, argmax_out);
    else
        softmax_gather_kernel<false><<<grid, kWarpsPerCta * 32, 0, stream>>>(d, w, wsb, nullptr);
    return cudaGetLastError();
}

cudaError_t launch_argmax(const float *acts, int64_t stride_t, int64_t stride_b, int B, int T, int V,
                          int64_t *argmax_out, cudaStream_t stream) {
    const long long frames = (long long)B * T;
    if (frames == 0) return cudaSuccess;
    const int grid = grid_for_frames(frames);
    const int b_major = stride_b > stride_t ? 1 : 0;
    argmax_kernel<<<grid, kWarpsPerCta * 32, 0, stream>>>(acts, stride_t, stride_b, B, T, V, argmax_out, b_major);
    return cudaGetLastError();
}

}  // namespace b200ctc
