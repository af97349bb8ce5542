// gradient.cu -- kernel 3: fused gradient.
//
// Replaces GramCTC.backward (asr/loss/gram_ctc.py:284-297) and _compute_label_probability (:180-217):
//   grad[t,b,k] = ( softmax[t,b,k] - exp( LSE_{j: symbol_j = k} (alpha_t[j]+beta_t[j]) - log P_b ) ) * gy * scale
//   and exactly 0 for t >= input_length[b] (:296).
// The reference keeps the softmax tensor alive from forward (717 MB) and materialises a second
// (T,B,V) array of per-unit posteriors; here the activations are re-read once, the softmax is
// recomputed from the saved per-frame normaliser, and the <= L+1 non-zero posteriors of a frame are
// merged from gamma on the fly.  One read + one write of (T,B,V), nothing else of that size.
//
// One warp per frame, frames handed out by a ticket counter; 128-bit streaming loads/stores.  Which
// columns carry a posterior is looked up in a per-utterance V-bit bitmap (1 word per 32 columns, L1
// resident), so the correction happens in registers and every gradient element is written once.
#include "common.cuh"
#include "kernels.h"
#include "row_ring.cuh"

namespace b200ctc {

namespace {

constexpr int kWarpsPerCta = 8;
constexpr int kUnroll = 4;
constexpr int kUttCache = 160;        // utterance records the ring kernel keeps in shared memory (40 bytes each)

__device__ __forceinline__ void zero_row(float *__restrict__ g, int V, int lane) {
    const int mis = (int)((reinterpret_cast<uintptr_t>(g) >> 2) & 3);
    const int head = mis ? min(V, 4 - mis) : 0;
    if (lane < head) g[lane] = 0.f;
    float4 *g4 = reinterpret_cast<float4 *>(g + head);
    const int n4 = (V - head) >> 2;
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = lane; i < n4; i += 32) stg_stream4(g4 + i, z);
    const int tail0 = head + 4 * n4;
    if (tail0 + lane < V) g[tail0 + lane] = 0.f;
}

// joint Gram-CTC + CTC: the plain-CTC node that carries the same symbol occurrence as Gram-CTC node j -- unigram
// node 3i+1 <-> CTC label node 2i+1 (blank nodes are summed separately, bigram nodes have no partner)
__device__ __forceinline__ float joint_partner(const float *e2_sm, int j, int Nb2) {
    if (Nb2 == 0 || j % 3 != 1) return 0.f;
    const int jc = 2 * (j / 3) + 1;
    return jc < Nb2 ? e2_sm[jc] : 0.f;
}

// softmax * sc for 4 consecutive columns, minus the (pre-scaled) posterior of the columns the lattice emits
__device__ __forceinline__ float4 grad4(const float4 &v, float c, float sc, unsigned word, int bit0, int pc,
                                        const float *__restrict__ post_sm) {
    float4 o;
    o.x = ex2_approx(fmaf(v.x, LOG2E_HI, c)) * sc;
    o.y = ex2_approx(fmaf(v.y, LOG2E_HI, c)) * sc;
    o.z = ex2_approx(fmaf(v.z, LOG2E_HI, c)) * sc;
    o.w = ex2_approx(fmaf(v.w, LOG2E_HI, c)) * sc;
    const unsigned nib = (word >> bit0) & 0xfu;
    if (nib) {                                              // ~2% of the columns: label/blank ids of this utterance
        int slot = pc + __popc(word & ((1u << bit0) - 1u));
        if (nib & 1u) o.x -= post_sm[slot++];
        if (nib & 2u) o.y -= post_sm[slot++];
        if (nib & 4u) o.z -= post_sm[slot++];
        if (nib & 8u) o.w -= post_sm[slot];
    }
    return o;
}

__global__ void __launch_bounds__(kWarpsPerCta * 32) gradient_kernel(GradParams gp, WsLayout w,
                                                                     unsigned char *ws, int b_major,
                                                                     int sm_floats_per_warp) {
    extern __shared__ float sm_all[];
    const ProblemDesc &d = gp.d;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    float *e_sm = sm_all + (size_t)warp * sm_floats_per_warp;        // [Np]   alpha*beta/P of this frame
    float *post_sm = e_sm + w.Np;                                    // [Umax] merged posterior * sc, by sorted id
    float *e2_sm = post_sm + ((w.Umax + 3) & ~3);                    // [Np2]  joint: the same for the plain-CTC lattice
    const UttInfo *utt2 = reinterpret_cast<const UttInfo *>(ws + w.off_utt2);
    const float2 *av2_all = reinterpret_cast<const float2 *>(ws + w.off_av2);
    const float2 *bv2_all = reinterpret_cast<const float2 *>(ws + w.off_bv2);
    WsHeader *hdr = reinterpret_cast<WsHeader *>(ws + w.off_hdr);
    const UttInfo *utt = reinterpret_cast<const UttInfo *>(ws + w.off_utt);
    const float2 *lse_all = reinterpret_cast<const float2 *>(ws + w.off_lse);
    const float2 *av_all = reinterpret_cast<const float2 *>(ws + w.off_av);
    const float2 *bv_all = reinterpret_cast<const float2 *>(ws + w.off_bv);
    const int *uoff_all = reinterpret_cast<const int *>(ws + w.off_uoff);
    const int *unode_all = reinterpret_cast<const int *>(ws + w.off_unode);
    const unsigned *bm_all = reinterpret_cast<const unsigned *>(ws + w.off_bm);
    const int *pc_all = reinterpret_cast<const int *>(ws + w.off_pc);
    const int per = d.kind == 0 ? 2 : 3;
    const unsigned frames = (unsigned)d.B * (unsigned)d.T;

    for (;;) {
        unsigned f = 0;
        if (lane == 0) f = atomicAdd(&hdr->k3_ticket, 1u);
        f = __shfl_sync(0xffffffffu, f, 0);
        if (f >= frames) break;
        int b, t;
        if (b_major) { b = (int)(f / d.T); t = (int)(f % d.T); }
        else { t = (int)(f / d.B); b = (int)(f % d.B); }
        float *grow = gp.grad_out + (int64_t)t * gp.gstride_t + (int64_t)b * gp.gstride_b;
        const UttInfo ui = utt[b];
        if (t >= ui.Tb) { zero_row(grow, d.V, lane); continue; }             // :296

        const float *row = d.acts + (int64_t)t * d.stride_t + (int64_t)b * d.stride_b;
        const float2 nrm = lse_all[(size_t)b * d.T + t];                     // grad_normaliser (common.cuh)
        const float gy = gp.per_utterance ? gp.grad_loss[b] : gp.grad_loss[0];
        const float sc = gy * gp.scale;                                      // :291-294
        const float c = -nrm.x;

        // ---- posteriors of this frame: e[j] = alpha*beta/P[t][j], merged per emitted id (:180-217) ----
        const float2 *arow = av_all + ((size_t)b * d.T + t) * w.Np;
        const float2 *brow = bv_all + ((size_t)b * d.T + t) * w.Np;
        float blank_part = 0.f;
        for (int j = lane; j < ui.Nb; j += 32) {
            const float2 a = __ldg(arow + j), bb = __ldg(brow + j + w.boff);
            const float e = node_posterior(a, bb, ui.Ph, ui.Pl);
            e_sm[j] = e;
            if (j % per == 0) blank_part += e;
        }
        const int Nb2 = w.joint ? 2 * ui.Lb + 1 : 0;
        if (w.joint) {                                                       // posteriors of the plain-CTC lattice
            const UttInfo u2 = utt2[b];
            const float2 *a2row = av2_all + ((size_t)b * d.T + t) * w.Np2;
            const float2 *b2row = bv2_all + ((size_t)b * d.T + t) * w.Np2;
            for (int j = lane; j < Nb2; j += 32) {
                const float e = node_posterior(__ldg(a2row + j), __ldg(b2row + j + 1), u2.Ph, u2.Pl);
                e2_sm[j] = e;
                if ((j & 1) == 0) blank_part += e;
            }
        }
        blank_part = warp_sum(blank_part);
        __syncwarp();
        const int *uoff = uoff_all + (size_t)b * (w.Nmax + 1);
        const int *unode = unode_all + (size_t)b * w.Nmax;
        for (int u = lane; u < ui.Ub; u += 32) {
            const int n0 = __ldg(uoff + u), n1 = __ldg(uoff + u + 1);
            float post = (u == ui.ublank) ? blank_part : 0.f;
            for (int n = n0; n < n1; ++n) {
                const int j = __ldg(unode + n);
                if (j < ui.Nb) post += e_sm[j];
                post += joint_partner(e2_sm, j, Nb2);
            }
            post_sm[u] = post * sc;
        }
        __syncwarp();
        const float sc_soft = (w.joint ? 2.f * sc : sc) * nrm.y;             // two losses, two softmax terms

        // ---- stream the row: grad = (softmax - posterior) * sc, one read and one write ----
        const unsigned *bm = bm_all + (size_t)b * w.nwords;
        const int *pc = pc_all + (size_t)b * w.nwords;
        const bool aligned = ((reinterpret_cast<uintptr_t>(row) | reinterpret_cast<uintptr_t>(grow)) & 15) == 0;
        if (aligned) {
            const float4 *row4 = reinterpret_cast<const float4 *>(row);
            float4 *g4 = reinterpret_cast<float4 *>(grow);
            const int n4 = d.V >> 2;
            int i = lane;
            for (; i + 32 * (kUnroll - 1) < n4; i += 32 * kUnroll) {
                float4 v[kUnroll];
                unsigned wd[kUnroll];
                int pcw[kUnroll];
#pragma unroll
                for (int u = 0; u < kUnroll; ++u) v[u] = ldg_stream4(row4 + i + 32 * u);
#pragma unroll
                for (int u = 0; u < kUnroll; ++u) {
                    const int wi = (i + 32 * u) >> 3;                        // column 4*(i+32u) lives in word col/32
                    wd[u] = __ldg(bm + wi);
                    pcw[u] = __ldg(pc + wi);
                }
#pragma unroll
                for (int u = 0; u < kUnroll; ++u)
                    stg_stream4(g4 + i + 32 * u, grad4(v[u], c, sc_soft, wd[u], ((i + 32 * u) & 7) << 2, pcw[u], post_sm));
            }
            for (; i < n4; i += 32) {
                const float4 v = ldg_stream4(row4 + i);
                const int wi = i >> 3;
                stg_stream4(g4 + i, grad4(v, c, sc_soft, __ldg(bm + wi), (i & 7) << 2, __ldg(pc + wi), post_sm));
            }
            for (int k = 4 * n4 + lane; k < d.V; k += 32) {
                float o = ex2_approx(fmaf(row[k], LOG2E_HI, c)) * sc_soft;
                const unsigned word = __ldg(bm + (k >> 5));
                if ((word >> (k & 31)) & 1u) o -= post_sm[__ldg(pc + (k >> 5)) + __popc(word & ((1u << (k & 31)) - 1u))];
                grow[k] = o;
            }
        } else {                                                             // unaligned rows (V % 4 != 0 ...)
            for (int k = lane; k < d.V; k += 32) {
                float o = ex2_approx(fmaf(row[k], LOG2E_HI, c)) * sc_soft;
                const unsigned word = __ldg(bm + (k >> 5));
                if ((word >> (k & 31)) & 1u) o -= post_sm[__ldg(pc + (k >> 5)) + __popc(word & ((1u << (k & 31)) - 1u))];
                grow[k] = o;
            }
        }
        __syncwarp();
    }
    // re-arm the queue for a possible second backward over the same workspace
    if (lane == 0) {
        __threadfence();
        const unsigned done = atomicAdd(&hdr->k3_done, 1u) + 1u;
        if (done == gridDim.x * kWarpsPerCta) { hdr->k3_ticket = 0u; hdr->k3_done = 0u; }
    }
}

// ---------------------------------------------------------------------------------------------
// kernel 3, TMA row-ring variant (see row_ring.cuh).  The producer bulk-copies the activation row AND
// the frame's alpha and beta rows into a ring slot; a consumer warp turns the row into the gradient in place
// (softmax * sc, then subtracts the merged posteriors at the <= L+1 label columns -- a plain scatter in
// shared memory, no bitmap needed) and hands it back to the TMA engine as one bulk store.  Padded frames
// never touch a consumer: the producer bulk-stores a zero row for them.
// Slot layout: [16-byte aligned span around the V-float row][Np float2 alpha row][Np float2 beta row].
// ---------------------------------------------------------------------------------------------
// Store a row image that sits in shared memory at the same 16-byte phase as its destination: the aligned body as
// one bulk copy, the <= 3 floats in front of and behind it with ordinary stores.  Called by one lane.
__device__ __forceinline__ void store_row_image(float *dst, const float *src_sm, int V) {
    const int head = min(V, (4 - row_misalignment(dst)) & 3);
    const int body = (V - head) & ~3;
    for (int i = 0; i < head; ++i) dst[i] = src_sm[i];
    for (int i = head + body; i < V; ++i) dst[i] = src_sm[i];
    if (body > 0) bulk_s2g(dst + head, src_sm + head, (uint32_t)body * 4u);
    bulk_commit();
}

__global__ void __launch_bounds__(kRingThreads, 1) gradient_ring_kernel(GradParams gp, WsLayout w, unsigned char *ws,
                                                                       int b_major, RingLayout rl) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Ring ring = ring_setup(smem_raw, rl);
    const ProblemDesc &d = gp.d;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    WsHeader *hdr = reinterpret_cast<WsHeader *>(ws + w.off_hdr);
    const UttInfo *utt = reinterpret_cast<const UttInfo *>(ws + w.off_utt);
    const unsigned frames = (unsigned)d.B * (unsigned)d.T;
    const uint32_t span_max = (uint32_t)ring_row_bytes(d.V);             // where the alpha row starts in a slot
    const uint32_t ab_bytes = (uint32_t)w.Np * 8u;
    const uint32_t ab2_bytes = w.joint ? (uint32_t)w.Np2 * 8u : 0u;      // joint: + the plain-CTC lattice's alpha/beta rows
    // extra region: [V + 4 floats of zeros][utterance records]
    float *zero_row = reinterpret_cast<float *>(smem_raw + rl.off_extra);
    // the utterance records, once per CTA: a consumer's row then starts without a round trip to L2
    UttInfo *utt_sm = reinterpret_cast<UttInfo *>(zero_row + ((d.V + 4 + 3) & ~3));
    const bool utt_cached = d.B <= kUttCache;
    for (int i = threadIdx.x; i < d.V + 4; i += blockDim.x) zero_row[i] = 0.f;
    if (utt_cached) {
        const int nwords = d.B * (int)(sizeof(UttInfo) / 4);
        for (int i = threadIdx.x; i < nwords; i += blockDim.x)
            reinterpret_cast<int *>(utt_sm)[i] = reinterpret_cast<const int *>(utt)[i];
    }
    fence_proxy_async_smem();
    __syncthreads();

    if (warp == 0) {
        // ===== producer (lane i owns frame i of the current batch) =====
        const float2 *av_all = reinterpret_cast<const float2 *>(ws + w.off_av);
        const float2 *bv_all = reinterpret_cast<const float2 *>(ws + w.off_bv);
        unsigned q = 0;
        auto issue_batch = [&](unsigned base) -> bool {
            if (base >= frames) return false;
            const unsigned f = base + (unsigned)lane;
            int b = 0, t = 0;
            bool need = false;
            if (lane < ring.batch && f < frames) {
                if (b_major) { b = (int)(f / d.T); t = (int)(f % d.T); }
                else { t = (int)(f / d.B); b = (int)(f % d.B); }
                if (t >= (utt_cached ? utt_sm[b].Tb : utt[b].Tb)) {                  // :296 -- zeros, straight from smem
                    float *dst = gp.grad_out + (int64_t)t * gp.gstride_t + (int64_t)b * gp.gstride_b;
                    store_row_image(dst, zero_row + row_misalignment(dst), d.V);
                } else {
                    need = true;
                }
            }
            const unsigned mask = __ballot_sync(0xffffffffu, need);
            const unsigned myq = q + (unsigned)__popc(mask & ((1u << lane) - 1u));
            // every lane issues its row as soon as ITS slot is free, in whatever order the consumers hand slots back
            bool pending = need;
            while (__any_sync(0xffffffffu, pending)) {
                bool issued = false;
                if (pending && ring_slot_free(ring, myq)) {
                    const int s = (int)(myq % (unsigned)ring.slots);
                    const float *src = d.acts + (int64_t)t * d.stride_t + (int64_t)b * d.stride_b;
                    const int off = row_misalignment(src);
                    const uint32_t span = row_span_bytes(off, d.V);
                    ring.meta[s].b = b; ring.meta[s].t = t; ring.meta[s].kind = 0; ring.meta[s].off = off;
                    ring_publish(ring, s, myq);
                    mbar_arrive_expect_tx(&ring.full[s], span + 2 * ab_bytes + 2 * ab2_bytes);
                    // no L2 hint: evict-first on these loads measured 2 us slower here (unlike kernel 1)
                    bulk_g2s(ring.slot(s), src - off, span, &ring.full[s]);
                    bulk_g2s(ring.slot(s) + span_max, av_all + ((size_t)b * d.T + t) * w.Np, ab_bytes, &ring.full[s]);
                    bulk_g2s(ring.slot(s) + span_max + ab_bytes, bv_all + ((size_t)b * d.T + t) * w.Np, ab_bytes, &ring.full[s]);
                    if (w.joint) {
                        const float2 *av2 = reinterpret_cast<const float2 *>(ws + w.off_av2) + ((size_t)b * d.T + t) * w.Np2;
                        const float2 *bv2 = reinterpret_cast<const float2 *>(ws + w.off_bv2) + ((size_t)b * d.T + t) * w.Np2;
                        bulk_g2s(ring.slot(s) + span_max + 2 * ab_bytes, av2, ab2_bytes, &ring.full[s]);
                        bulk_g2s(ring.slot(s) + span_max + 2 * ab_bytes + ab2_bytes, bv2, ab2_bytes, &ring.full[s]);
                    }
                    pending = false;
                    issued = true;
                }
                if (!__any_sync(0xffffffffu, issued)) __nanosleep(40);
            }
            q += (unsigned)__popc(mask);
            return true;
        };
        // two tickets in flight: the one a batch needs was requested two batches ago (see softmax_gather.cu)
        unsigned pa = 0, pb = 0;
        if (lane == 0) { pa = atomicAdd(&hdr->k3_ticket, (unsigned)ring.batch); pb = atomicAdd(&hdr->k3_ticket, (unsigned)ring.batch); }
        for (;;) {
            unsigned base = __shfl_sync(0xffffffffu, pa, 0);
            if (lane == 0 && base < frames) pa = atomicAdd(&hdr->k3_ticket, (unsigned)ring.batch);
            if (!issue_batch(base)) break;
            base = __shfl_sync(0xffffffffu, pb, 0);
            if (lane == 0 && base < frames) pb = atomicAdd(&hdr->k3_ticket, (unsigned)ring.batch);
            if (!issue_batch(base)) break;
        }
        ring_stop(ring, q, lane);
        bulk_wait_all<0>();
        // re-arm the queue for a possible second backward over the same workspace
        if (lane == 0) {
            __threadfence();
            const unsigned done = atomicAdd(&hdr->k3_done, 1u) + 1u;
            if (done == gridDim.x) { hdr->k3_ticket = 0u; hdr->k3_done = 0u; }
        }
        return;
    }

    // ===== consumers =====
    const float2 *lse_all = reinterpret_cast<const float2 *>(ws + w.off_lse);
    const int *unode_all = reinterpret_cast<const int *>(ws + w.off_unode);
    const int4 *urec_all = reinterpret_cast<const int4 *>(ws + w.off_urec);
    constexpr int kRecBatch = 4;                          // id records per lane requested in one go
    const int per = d.kind == 0 ? 2 : 3;
    if (warp - 1 >= ring.nc) return;                      // short ring: fewer active consumers (row_ring.cuh)
    for (;;) {
        const unsigned q = ring_next_row(ring, lane);
        const int s = ring_acquire(ring, q);
        const RowMeta m = ring.meta[s];
        if (m.kind < 0) {                       // stop record: hand the slot back (the ring may be shorter than
            __syncwarp();                       // the number of consumers) and leave
            if (lane == 0) mbar_arrive(&ring.empty[s]);
            break;
        }
        const int b = m.b, t = m.t;
        float *slotf = reinterpret_cast<float *>(ring.slot(s));
        float *row = slotf + m.off;                                          // element v of the frame
        const int n4 = (m.off + d.V + 3) >> 2;                               // float4s of the aligned span
        const float2 *a_sm = reinterpret_cast<const float2 *>(ring.slot(s) + span_max);   // alpha row
        const float2 *b_sm = a_sm + w.Np;                                    // beta row
        float *e_sm = reinterpret_cast<float *>(const_cast<float2 *>(a_sm)); // alpha*beta/P, written over the alpha row
        const float2 *a2_sm = b_sm + w.Np;                                   // joint: plain-CTC alpha row, beta row
        const float2 *b2_sm = a2_sm + w.Np2;
        float *e2_sm = reinterpret_cast<float *>(const_cast<float2 *>(a2_sm));
        const UttInfo ui = utt_cached ? utt_sm[b] : utt[b];
        // requested now, needed after the posteriors: their round trip hides behind the node loop
        const float2 nrm = __ldg(lse_all + (size_t)b * d.T + t);             // grad_normaliser (common.cuh)
        const float sc = (gp.per_utterance ? __ldg(gp.grad_loss + b) : __ldg(gp.grad_loss)) * gp.scale;      // :291-294
        const int4 *urec = urec_all + (size_t)b * w.Nmax;
        int4 rec[kRecBatch];
#pragma unroll
        for (int k = 0; k < kRecBatch; ++k)
            rec[k] = 32 * k + lane < ui.Ub ? __ldg(urec + 32 * k + lane) : make_int4(0, 0, 0, -1);

        float blank_part = 0.f;
        for (int j0 = 0; j0 < ui.Nb; j0 += 32) {
            const int j = j0 + lane;
            float e = 0.f;
            if (j < ui.Nb) {
                const float2 a = a_sm[j], bb = b_sm[j + w.boff];
                e = node_posterior(a, bb, ui.Ph, ui.Pl);
            }
            __syncwarp();                                                    // e_sm aliases the alpha row: reads first
            if (j < ui.Nb) e_sm[j] = e;
            if (j < ui.Nb && j % per == 0) blank_part += e;
        }
        const int Nb2 = w.joint ? 2 * ui.Lb + 1 : 0;
        if (w.joint) {
            const UttInfo *utt2 = reinterpret_cast<const UttInfo *>(ws + w.off_utt2);
            const float Ph2 = utt2[b].Ph, Pl2 = utt2[b].Pl;
            for (int j0 = 0; j0 < Nb2; j0 += 32) {
                const int j = j0 + lane;
                float e = 0.f;
                if (j < Nb2) e = node_posterior(a2_sm[j], b2_sm[j + 1], Ph2, Pl2);
                __syncwarp();                                                // e2_sm aliases the alpha row: reads first
                if (j < Nb2) e2_sm[j] = e;
                if (j < Nb2 && (j & 1) == 0) blank_part += e;
            }
        }
        blank_part = warp_sum(blank_part);
        const float sc_soft = (w.joint ? 2.f * sc : sc) * nrm.y;             // two losses, two softmax terms
        const float c = -nrm.x;
        // softmax * sc in place, over the whole aligned span (what lies outside the row is never stored)
        float4 *row4 = reinterpret_cast<float4 *>(slotf);
#pragma unroll 4
        for (int i = lane; i < n4; i += 32) {
            float4 v = row4[i];
            v.x = ex2_approx(fmaf(v.x, LOG2E_HI, c)) * sc_soft;
            v.y = ex2_approx(fmaf(v.y, LOG2E_HI, c)) * sc_soft;
            v.z = ex2_approx(fmaf(v.z, LOG2E_HI, c)) * sc_soft;
            v.w = ex2_approx(fmaf(v.w, LOG2E_HI, c)) * sc_soft;
            row4[i] = v;
        }
        __syncwarp();
        // merge per emitted id (:180-217) and subtract at the id's column (distinct columns, :290): blank nodes from
        // the strided sum above, the others in node order (fixed order => deterministic).  The records of the first
        // 128 ids were requested at the start of the row; an id carried by one node needs nothing else.
        const int *unode = unode_all + (size_t)b * w.Nmax;
        for (int u0 = 0; u0 < ui.Ub; u0 += 32 * kRecBatch) {
            if (u0 > 0) {
#pragma unroll
                for (int k = 0; k < kRecBatch; ++k) {
                    const int u = u0 + 32 * k + lane;
                    rec[k] = u < ui.Ub ? __ldg(urec + u) : make_int4(0, 0, 0, -1);
                }
            }
#pragma unroll
            for (int k = 0; k < kRecBatch; ++k) {
                const int u = u0 + 32 * k + lane;
                if (u >= ui.Ub) continue;
                float post = (u == ui.ublank) ? blank_part : 0.f;
                int j = rec[k].w;
                for (int n = 0; n < rec[k].z; ++n) {
                    if (n > 0) j = __ldg(unode + rec[k].y + n);
                    if (j < ui.Nb) post += e_sm[j];
                    post += joint_partner(e2_sm, j, Nb2);
                }
                row[rec[k].x] -= post * sc;
            }
        }
        float *dst = gp.grad_out + (int64_t)t * gp.gstride_t + (int64_t)b * gp.gstride_b;
        if (row_misalignment(dst) == m.off) {                                // warp-uniform
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
                store_row_image(dst, row, d.V);
                bulk_wait_read<0>();             // the TMA engine has read the slot: hand it back to the producer
                mbar_arrive(&ring.empty[s]);
            }
        } else {
            // activation row and gradient row sit at different 16-byte phases (different pitches): the image in the
            // slot cannot be bulk-stored, the warp writes it with ordinary coalesced stores
            __syncwarp();
            for (int i = lane; i < d.V; i += 32) dst[i] = row[i];
            __syncwarp();
            if (lane == 0) mbar_arrive(&ring.empty[s]);
        }
    }
    if (lane == 0) bulk_wait_all<0>();
}

}  // namespace

cudaError_t launch_gradient(const GradParams &g, const WsLayout &w, const void *ws, cudaStream_t stream) {
    const long long frames = (long long)g.d.B * g.d.T;
    if (frames == 0) return cudaSuccess;
    unsigned char *wsb = const_cast<unsigned char *>(static_cast<const unsigned char *>(ws));
    const int b_major = g.gstride_b > g.gstride_t ? 1 : 0;
    const size_t extra = sizeof(float) * (size_t)((g.d.V + 4 + 3) & ~3) + (g.d.B <= kUttCache ? sizeof(UttInfo) * (size_t)g.d.B : 0);
    const RingLayout rl = make_ring(ring_row_bytes(g.d.V) + sizeof(float) * (4 * (size_t)w.Np + (w.joint ? 4 * (size_t)w.Np2 : 0)), extra);
    if (ring_usable(g.d.acts, rl) && ring_usable(g.grad_out, rl)) {
        long long ctas = (frames + kTicketBatch - 1) / kTicketBatch;
        if (ctas > sm_count()) ctas = sm_count();
        if (ctas < 1) ctas = 1;
        cudaError_t e = ensure_dynamic_smem(reinterpret_cast<const void *>(gradient_ring_kernel), rl.total);
        if (e != cudaSuccess) return e;
        gradient_ring_kernel<<<(int)ctas, kRingThreads, rl.total, stream>>>(g, w, wsb, b_major, rl);
        return cudaGetLastError();
    }
    const int per_warp = w.Np + ((w.Umax + 3) & ~3) + (w.joint ? w.Np2 : 0);
    const size_t smem = sizeof(float) * (size_t)per_warp * kWarpsPerCta;
    cudaError_t e = ensure_dynamic_smem(reinterpret_cast<const void *>(gradient_kernel), smem);
    if (e != cudaSuccess) return e;
    long long ctas = (frames + kWarpsPerCta - 1) / kWarpsPerCta;
    const long long cap = (long long)sm_count() * 8;
    if (ctas > cap) ctas = cap;
    gradient_kernel<<<(int)ctas, kWarpsPerCta * 32, smem, stream>>>(g, w, wsb, b_major, per_warp);
    return cudaGetLastError();
}

}  // namespace b200ctc
