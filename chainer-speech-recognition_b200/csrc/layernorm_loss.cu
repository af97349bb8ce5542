// layernorm_loss.cu -- LayerNormalization fused into the loss (SURVEY.md 8f rank 3).
//
// In the reference every CTC / Gram-CTC model ends in Convolution2D(.., vocab_size, ksize=1) -> LayerNormalization
// (run/ctc/cnn/model.py:85-88): the convolution output z is (B, V, 1, T), NormalizeLayer normalises every frame over
// the vocabulary axis (asr/nn/layernorm.py:33-46: mean and std over axes (1,2), no epsilon), gamma/beta scale and
// shift along axis 1 (asr/nn/nn.py:265), and AcousticModel.__call__ then makes a TRANSPOSED COPY of the whole tensor --
// swapaxes(1,3), reshape, split_axis into T arrays of (B,V) (asr/model/cnn.py:41-44) -- before the loss reads it.
// Backward undoes all of it.  Per activation element that is ~48 bytes of HBM traffic around a 12-byte loss.
//
// Here the loss kernels read z where it lies, T-contiguous, as 2-D tiles moved by the TMA engine
// (cp.async.bulk.tensor, SASS UTMALDG): a tile is all V vocabulary rows x 8 consecutive frames of one utterance,
// split into boxes of 240 rows (7.5 KB; a TMA box dimension is at most 256) that land in a shared-memory ring.  A frame's vocabulary
// is then spread over the CTA -- thread (warp w of 15, lane) owns rows 240k + 16w + lane/2 (k = 0..K-1) and four of the
// eight frames -- so per-frame statistics are reductions over threads (shuffles inside a warp, shared memory
// between warps) and everything per element happens in registers:
//   forward  (ln_softmax_gather_kernel): one read of z.  Mean / centred second moment of every frame (Chan's
//            pairwise update, so one reduction round), the softmax statistics of a = gamma*(z-mean)*rstd + beta
//            (per-thread max and sum, merged as (max, sum) pairs: the second round), the emission probabilities of
//            the lattice's symbols.  Writes mean, rstd, log2-normaliser and the emission rows; the alpha/beta
//            recursion (lattice.cu) runs unchanged, next to this kernel.
//   backward (ln_gradient_kernel): one read of z, one write of dz, in z's own layout.  Sweep 1 re-forms the softmax,
//            subtracts the merged posteriors (gram_ctc.py:284-297), multiplies by gamma and accumulates the two
//            per-frame sums LayerNormalization's backward needs (asr/nn/layernorm.py:48-60) while dgamma/dbeta
//            accumulate per thread over all tiles (a thread's rows never change); sweep 2 re-reads z from the ring
//            (it is still there) and stores dz = rstd * (dn - mean_v(dn) - n * mean_v(dn*n)).
// 12 bytes per element again -- for the loss AND the normalisation AND both transposes.
//   argmax   (ln_argmax_kernel): the development loop's greedy ids (run/ctc/cnn/train.py:224-234) from one read of z.
//            Round 1 as in forward, then the best (value, row) of every frame, merged numpy.argmax-style; every frame
//            of the padded batch is decoded (asr/error.py:40).  No workspace, one launch.
//
// Joint Gram-CTC + CTC objective (run/gram_ctc/cnn/train.py:196-198): the forward pass is Gram-CTC's plus the second,
// plain-CTC lattice on the same emission rows (api.cu); the backward kernel adds the plain-CTC posteriors to the Gram-CTC
// ones node by node in phase (a) and doubles the softmax term (two losses).
//
// Limits of this version: V <= 4080 (a tile must stay resident in shared memory in the backward kernel: 17 boxes),
// rows of z 16-byte aligned (T_pitch % 4 == 0 -- a TMA requirement), at most 480 emission columns, and a backward ring
// of at least K + 2 boxes next to the lattice's per-tile tables (plan_ln_backward: long labels at a large V do not fit).
// Outside them the entry points return B200CTC_UNSUPPORTED and the caller uses the unfused path.  The argmax has only
// the first two limits.
#include <cuda.h>
#include <stdio.h>
#include <mutex>

#include "common.cuh"
#include "kernels.h"
#include "prep.cuh"

namespace b200ctc {

namespace {

constexpr int kLnWarps = 15;                               // compute warps: with the producer warp 512 threads, i.e. 128 registers each
constexpr int kLnThreads = 32 * (kLnWarps + 1);            // + the producer warp
constexpr int kLnTT = 8;                                   // frames per tile
constexpr int kLnBoxRows = 16 * kLnWarps;                  // 240 rows: one step of every compute warp
constexpr uint32_t kLnBoxBytes = kLnBoxRows * kLnTT * 4;   // 7.5 KB
constexpr int kLnMetaRing = 64;                            // >= ring slots: a padded tile takes one slot and one record
constexpr int kLnMaxCols = 32 * kLnWarps;                  // emission columns one tile pass can gather: one per compute thread
constexpr int kLnJointPre = 4;                             // joint backward: plain-CTC alpha/beta items a thread requests ahead

// Everything a tile's consumers need to know about it, fetched by the producer lane (a dependent global load at the
// start of a tile would stall all fifteen compute warps for its round trip)
struct LnTileMeta {
    int b, t0, kind;                 // kind 0: work, -1: stop
    int Tb, Lb;                      // clamped input / label length of the utterance
    int Nb, Ub, ublank;              // backward: lattice nodes, distinct symbols, position of the blank among them
    float Ph, Pl, sc;                // backward: P as in UttInfo, upstream gradient * scale
    int pad;
};

constexpr int kLnFifo = 8;
constexpr int kLnGroup = 4;              // 8-frame blocks with consecutive tickets: one 128-byte line of every row in flight together
constexpr int kLnBlankChunks = 64;                         // 32-node chunks of the largest lattice (Nmax <= 2048)
struct LnSignalFifo {                // forward: finished tiles on their way to the progress counters
    int4 entry[kLnFifo];             // (b, 16-frame block, valid frames, 0); b < 0: done
    unsigned head, tail;
};

struct LnSmem {
    size_t off_ring, off_full, off_empty, off_meta, off_red, off_tot, off_fc, off_fifo, off_ab, off_abbar, off_post, off_ebuf,
        off_csr, off_gb, off_bm, off_zero, total;
    int R;
};

// ring of R boxes + everything else a kernel needs (the backward-only parts are 0 in the forward kernel)
LnSmem plan_ln_smem(size_t ab_bytes, size_t post_floats, size_t ebuf_floats, size_t csr_ints, size_t gb_floats,
                    size_t bm_words, size_t zero_bytes, size_t smem_reserve = 0) {
    LnSmem s;
    size_t o = 0;
    s.off_full = o;  o += 8 * 64;
    s.off_empty = o; o += 8 * 64;
    s.off_abbar = o; o += 32;                               // alpha/beta full, empty; output full; spare
    s.off_meta = o;  o += sizeof(LnTileMeta) * kLnMetaRing;
    s.off_red = o;   o += sizeof(float) * 16 * kLnTT * 4;
    s.off_tot = o;   o += sizeof(float) * kLnTT * 8;
    s.off_fc = o;    o += sizeof(float) * 3 * kLnTT;        // per-frame mean, 1/std, log2 normaliser (16-byte aligned)
    s.off_fifo = o;  o += sizeof(LnSignalFifo);
    s.off_post = o;  o += sizeof(float) * post_floats;
    s.off_ebuf = o;  o += sizeof(float) * ebuf_floats;
    s.off_csr = o;   o += sizeof(int) * csr_ints;
    s.off_gb = o;    o += sizeof(float) * gb_floats;
    s.off_bm = o;    o += sizeof(unsigned) * bm_words;
    o = align_up(o, 128);
    s.off_zero = o;  o += align_up(zero_bytes, 128);
    s.off_ab = o;    o += align_up(ab_bytes, 128);
    s.off_ring = o;
    const long long room = (smem_reserve ? 228 * 1024 - 2 * 1024 - (long long)smem_reserve : 227 * 1024) - (long long)o;
    int R = (int)(room / (long long)kLnBoxBytes);
    if (R > 64) R = 64;
    s.R = R;
    s.total = o + (size_t)(R > 0 ? R : 0) * kLnBoxBytes;
    return s;
}

__device__ __forceinline__ void tma_load_box(void *dst, const CUtensorMap *map, int t0, int v0, int b, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
            smem_u32(dst)),
        "l"(map), "r"(t0), "r"(v0), "r"(b), "r"(smem_u32(bar))
        : "memory");
}
// shared -> global tile store (bulk-group completion); elements outside the tensor are not written
__device__ __forceinline__ void tma_store_box(const CUtensorMap *map, const void *src, int t0, int v0, int b) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%1, %2, %3}], [%4];" ::"l"(map), "r"(t0), "r"(v0),
                 "r"(b), "r"(smem_u32(src))
                 : "memory");
}
__device__ __forceinline__ void sts128(uint32_t addr, const float4 &v) {
    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
// For the lanes of the producer warp, which share ONE warp while running different loops: a suspending wait in one
// lane would put the others to sleep with it, so these lanes only probe (test_wait returns at once) and nap.
__device__ __forceinline__ void mbar_poll(uint64_t *bar, uint32_t parity) {
    while (!mbar_test_wait(bar, parity)) __nanosleep(40);
}
__device__ __forceinline__ void bar_compute() { asm volatile("bar.sync 1, %0;" ::"n"(32 * kLnWarps) : "memory"); }

// ---- tile order ----
// A tile takes 32 bytes out of every row of z, rows 4*T bytes apart: what DRAM sees depends on which tiles are in flight
// TOGETHER.  Groups of G consecutive 8-frame blocks of one utterance get consecutive tickets, so the SMs working on them
// touch 32*G contiguous bytes of every row at about the same time.  G = 4 (one 128-byte line) is the measured best:
// 8 and 16 change nothing, 32 and whole rows are slower (measured with a tuning switch that is in git history) -- longer groups
// serve the lattice kernel in coarser lumps and balance the variable-length utterances worse.  Groups walk the time axis from
// both ends (the alpha CTAs of the lattice kernel consume frames in ascending, the beta CTAs in descending order).
__device__ __forceinline__ bool ln_tile_of_ticket(unsigned f, int B, int nTB, bool two_ended, int &b, int &tb) {
    constexpr int G = kLnGroup;
    const int sub = (int)(f % (unsigned)G);
    const unsigned q = f / (unsigned)G;
    b = (int)(q % (unsigned)B);
    const int gs = (int)(q / (unsigned)B);
    const int ngroups = (nTB + G - 1) / G;
    const int g = !two_ended ? gs : (gs & 1) ? (ngroups - 1 - (gs >> 1)) : (gs >> 1);
    tb = G * g + sub;
    return tb < nTB;
}

// ---- reductions of four per-frame values over the 16 lanes that share this lane's half (lane bits 1..4) ----
// Transposed: after the first two exchanges every lane carries ONE frame (index 2*bit1 + bit2 of its half), so the
// whole thing takes 5 merges instead of 16.  `merge(a, b)` combines two partial results.
template <typename T, typename F>
__device__ __forceinline__ T reduce_frames16(T x0, T x1, T x2, T x3, int lane, F merge, int &frame_in_half) {
    const bool b1 = (lane >> 1) & 1, b2 = (lane >> 2) & 1;
    T k0 = b1 ? x2 : x0, k1 = b1 ? x3 : x1;           // kept
    T s0 = b1 ? x0 : x2, s1 = b1 ? x1 : x3;           // sent to lane ^ 2
    k0 = merge(k0, T::shfl_xor(s0, 2));
    k1 = merge(k1, T::shfl_xor(s1, 2));
    T k = b2 ? k1 : k0, s = b2 ? k0 : k1;
    k = merge(k, T::shfl_xor(s, 4));
    k = merge(k, T::shfl_xor(k, 8));
    k = merge(k, T::shfl_xor(k, 16));
    frame_in_half = 2 * (int)b1 + (int)b2;
    return k;
}

struct Moments {                      // count, mean, centred second moment (Chan et al.)
    float n, mean, m2;
    static __device__ __forceinline__ Moments shfl_xor(const Moments &a, int o) {
        Moments r;
        r.n = __shfl_xor_sync(0xffffffffu, a.n, o);
        r.mean = __shfl_xor_sync(0xffffffffu, a.mean, o);
        r.m2 = __shfl_xor_sync(0xffffffffu, a.m2, o);
        return r;
    }
};
__device__ __forceinline__ Moments merge_moments(const Moments &a, const Moments &b) {
    Moments r;
    r.n = a.n + b.n;
    const float inv = r.n > 0.f ? __fdividef(1.f, r.n) : 0.f;
    const float d = b.mean - a.mean;
    r.mean = fmaf(d, b.n * inv, a.mean);
    r.m2 = a.m2 + b.m2 + d * d * (a.n * b.n * inv);
    return r;
}
struct MaxSum {                       // running maximum (natural units) and sum of 2^((x - max) * log2 e)
    float m, s;
    static __device__ __forceinline__ MaxSum shfl_xor(const MaxSum &a, int o) {
        MaxSum r;
        r.m = __shfl_xor_sync(0xffffffffu, a.m, o);
        r.s = __shfl_xor_sync(0xffffffffu, a.s, o);
        return r;
    }
};
__device__ __forceinline__ MaxSum merge_maxsum(const MaxSum &a, const MaxSum &b) {
    MaxSum r;
    r.m = fmaxf(a.m, b.m);
    const float fa = a.m == -INFINITY ? 0.f : ex2_approx((a.m - r.m) * LOG2E_HI);
    const float fb = b.m == -INFINITY ? 0.f : ex2_approx((b.m - r.m) * LOG2E_HI);
    r.s = a.s * fa + b.s * fb;
    return r;
}
struct Pair2 {                        // two plain sums
    float a, b;
    static __device__ __forceinline__ Pair2 shfl_xor(const Pair2 &x, int o) {
        Pair2 r;
        r.a = __shfl_xor_sync(0xffffffffu, x.a, o);
        r.b = __shfl_xor_sync(0xffffffffu, x.b, o);
        return r;
    }
};
__device__ __forceinline__ Pair2 merge_pair2(const Pair2 &x, const Pair2 &y) { return Pair2{x.a + y.a, x.b + y.b}; }

struct LnParams {
    ProblemDesc d;                  // d.acts unused; kind/B/T/V/Lmax/blank/labels/bigrams/lengths/concurrent as usual
    WsLayout w;
    unsigned char *ws;
    const float *z;                 // (B, V, T): element (b, v, t) at z[b*zs_b + v*zs_v + t]
    int64_t zs_b, zs_v;
    const float *gamma, *beta;
    size_t off_mu, off_rstd, off_lse, off_part;
    int Tq;                         // row pitch of the per-frame arrays: T rounded up to a multiple of 4 (16-byte rows)
    int K;                          // boxes per tile = ceil(V / 240)
    int nTB;                        // 8-frame blocks = ceil(T / 8)
    int R;                          // ring slots
    // backward only
    const float *grad_loss;
    int per_utterance;
    float scale;
    float *dz;
    int64_t dzs_b, dzs_v;
    float *dgamma, *dbeta;
};

// ---- producer lane: tickets -> tile records -> TMA box loads, as far ahead as the ring allows ----
// kLnBackward: tile i of the kernel goes to CTA i % gridDim.x (a fixed assignment makes the dgamma/dbeta sums
// deterministic); kLnForward: tiles are drawn from the global ticket counter (variable-length utterances balance
// themselves, and the order serves the lattice kernel running next to it).
// Tiles whose frames are all padding never reach the compute warps: the forward pass skips them, the backward pass
// stores their zeros (gram_ctc.py:296; LayerNormalization's backward of zero is zero) straight from a box of zeros.
// kLnArgmax: every frame is decoded (all T of them, asr/error.py:40), so every tile is work of the same size: the fixed
// assignment of the backward pass, with no counter to reset and nothing but z to load.
enum LnPass { kLnForward, kLnBackward, kLnArgmax };
template <int PASS>
__device__ __forceinline__ void ln_producer(const CUtensorMap *tmap, const CUtensorMap *tmap_out, const LnParams &p,
                                            unsigned char *smem, const LnSmem &sm) {
    constexpr bool BACKWARD = PASS == kLnBackward;
    constexpr bool FIXED = PASS != kLnForward;
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + sm.off_full);
    uint64_t *empty = reinterpret_cast<uint64_t *>(smem + sm.off_empty);
    uint64_t *abbar = reinterpret_cast<uint64_t *>(smem + sm.off_abbar);          // [0] full, [1] empty
    LnTileMeta *metas = reinterpret_cast<LnTileMeta *>(smem + sm.off_meta);
    WsHeader *hdr = reinterpret_cast<WsHeader *>(p.ws + p.w.off_hdr);
    const UttInfo *utt = reinterpret_cast<const UttInfo *>(p.ws + p.w.off_utt);
    constexpr int G = kLnGroup;
    const unsigned tiles = (unsigned)p.d.B * (unsigned)(((p.nTB + G - 1) / G) * G);
    const unsigned R = (unsigned)p.R;
    const int K = p.K;
    unsigned box = 0, seq = 0, n_ab = 0;             // boxes / tile records / alpha-beta loads issued by this CTA
    auto claim = [&](unsigned bx) {                  // wait until the box slot's previous occupant was released
        if (bx >= R) mbar_poll(&empty[bx % R], ((bx / R) - 1u) & 1u);
        return (int)(bx % R);
    };
    unsigned f = FIXED ? blockIdx.x : atomicAdd(&hdr->k1_ticket, 1u);
    while (f < tiles) {
        const unsigned fnext = FIXED ? f + gridDim.x : atomicAdd(&hdr->k1_ticket, 1u);     // in flight while we issue
        int b, tb;
        const bool real = ln_tile_of_ticket(f, p.d.B, p.nTB, !FIXED && p.d.concurrent != 0, b, tb);
        f = fnext;
        if (!real) continue;
        const int t0 = tb * kLnTT;
        LnTileMeta mm;
        mm.b = b; mm.t0 = t0; mm.kind = 0; mm.pad = 0;
        mm.Nb = 0; mm.Ub = 0; mm.ublank = 0; mm.Ph = 0.f; mm.Pl = 0.f; mm.sc = 0.f;
        if (BACKWARD) {
            const UttInfo ui = utt[b];
            mm.Tb = ui.Tb; mm.Lb = ui.Lb; mm.Nb = ui.Nb; mm.Ub = ui.Ub; mm.ublank = ui.ublank; mm.Ph = ui.Ph; mm.Pl = ui.Pl;
            mm.sc = (p.per_utterance ? __ldg(p.grad_loss + b) : __ldg(p.grad_loss)) * p.scale;      // gram_ctc.py:291-294
        } else if (PASS == kLnArgmax) {
            mm.Tb = p.d.T; mm.Lb = 0;
        } else {
            mm.Tb = utt_input_length(p.d, b);
            mm.Lb = utt_label_length(p.d, b);
        }
        if (t0 >= mm.Tb) {                            // nothing but padding
            if (BACKWARD) {
                for (int k = 0; k < K; ++k) tma_store_box(tmap_out, smem + sm.off_zero, t0, k * kLnBoxRows, b);
                bulk_commit();
            }
            continue;
        }
        // the tile record travels with the tile's first box
        const int slot0 = claim(box);
        metas[seq % kLnMetaRing] = mm;
        ++seq;
        if (BACKWARD) {
            // alpha and beta rows of the tile's frames (contiguous in the workspace: [b][t][Np]) and the per-frame
            // mean, 1/std and log2 normaliser the forward pass left
            const int nfr = min(kLnTT, p.d.T - t0);
            const uint32_t bytes = (uint32_t)nfr * (uint32_t)p.w.Np * 8u;
            const uint32_t fbytes = (uint32_t)min(kLnTT, p.Tq - t0) * 4u;          // 16 or 32 bytes
            if (n_ab > 0) mbar_poll(&abbar[1], (n_ab - 1u) & 1u);
            ++n_ab;
            const size_t fo = (size_t)b * p.Tq + t0;                                // 16-byte aligned rows of the per-frame arrays
            const float2 *av = reinterpret_cast<const float2 *>(p.ws + p.w.off_av) + ((size_t)b * p.d.T + t0) * p.w.Np;
            const float2 *bv = reinterpret_cast<const float2 *>(p.ws + p.w.off_bv) + ((size_t)b * p.d.T + t0) * p.w.Np;
            float *fc = reinterpret_cast<float *>(smem + sm.off_fc);
            mbar_arrive_expect_tx(&abbar[0], 2 * bytes + 3 * fbytes);
            bulk_g2s(smem + sm.off_ab, av, bytes, &abbar[0]);
            bulk_g2s(smem + sm.off_ab + (size_t)kLnTT * p.w.Np * 8, bv, bytes, &abbar[0]);
            bulk_g2s(fc, reinterpret_cast<const float *>(p.ws + p.off_mu) + fo, fbytes, &abbar[0]);
            bulk_g2s(fc + kLnTT, reinterpret_cast<const float *>(p.ws + p.off_rstd) + fo, fbytes, &abbar[0]);
            bulk_g2s(fc + 2 * kLnTT, reinterpret_cast<const float *>(p.ws + p.off_lse) + fo, fbytes, &abbar[0]);
        }
        for (int k = 0; k < K; ++k, ++box) {
            const int slot = k == 0 ? slot0 : claim(box);
            mbar_arrive_expect_tx(&full[slot], kLnBoxBytes);
            tma_load_box(smem + sm.off_ring + (size_t)slot * kLnBoxBytes, tmap, t0, k * kLnBoxRows, b, &full[slot]);
        }
    }
    const int slot0 = claim(box);                    // stop record
    metas[seq % kLnMetaRing].kind = -1;
    mbar_arrive(&full[slot0]);
    if (BACKWARD) bulk_wait_all<0>();                // the zero box must outlive the stores that read it
}

// ---- forward, lane 1 of the producer warp: finished tiles -> progress counters of the lattice kernel ----
// The "rows written" signal is a release at GPU scope and costs ~1.5 us (common.cuh): it must not sit on a compute warp.
__device__ __forceinline__ void ln_signaller(const LnParams &p, unsigned char *smem, const LnSmem &sm) {
    LnSignalFifo *ff = reinterpret_cast<LnSignalFifo *>(smem + sm.off_fifo);
    unsigned taken = 0;
    for (;;) {
        while (*reinterpret_cast<volatile unsigned *>(&ff->head) == taken) __nanosleep(100);
        __threadfence_block();
        const volatile int *e = reinterpret_cast<volatile int *>(&ff->entry[taken % kLnFifo]);
        const int b = e[0], blk = e[1], n = e[2];
        *reinterpret_cast<volatile unsigned *>(&ff->tail) = ++taken;
        if (b < 0) break;
        unsigned *pc = reinterpret_cast<unsigned *>(p.ws + p.w.off_prog) + (size_t)b * p.w.nblk + blk;
        asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(pc), "r"((unsigned)n) : "memory");
    }
}
__device__ __forceinline__ void ln_signal_push(LnSignalFifo *ff, unsigned &pushed, int b, int blk, int n) {
    while (pushed - *reinterpret_cast<volatile unsigned *>(&ff->tail) >= (unsigned)kLnFifo) __nanosleep(64);
    ff->entry[pushed % kLnFifo] = make_int4(b, blk, n, 0);
    __threadfence_block();                           // the tile's stores (ordered by the CTA barrier) and the entry, then the head
    *reinterpret_cast<volatile unsigned *>(&ff->head) = ++pushed;
}

// ---- backward, lane 1 of the producer warp: finished tiles (dz images in their boxes) -> TMA tile stores ----
__device__ __forceinline__ void ln_storer(const CUtensorMap *tmap_out, const LnParams &p, unsigned char *smem, const LnSmem &sm) {
    uint64_t *empty = reinterpret_cast<uint64_t *>(smem + sm.off_empty);
    uint64_t *outbar = reinterpret_cast<uint64_t *>(smem + sm.off_abbar) + 2;
    const LnTileMeta *metas = reinterpret_cast<const LnTileMeta *>(smem + sm.off_meta);
    const unsigned R = (unsigned)p.R;
    // How many tiles there will be is announced through a plain word, NOT as one more arrival on the barrier: the
    // compute warps meet the stop record nanoseconds after their last tile, and two completions in a row would move the
    // barrier's parity bit back to where this lane is still waiting for it.  (Two TILE arrivals can never run ahead of
    // this lane: a tile's boxes only become free when this lane has stored the tile before it.)
    const volatile unsigned *total = &reinterpret_cast<const LnSignalFifo *>(smem + sm.off_fifo)->head;      // tiles + 1, 0 = not known yet
    unsigned slot = 0;
    for (unsigned n = 0;; ++n) {
        bool stop = false;
        while (!mbar_test_wait(outbar, n & 1u)) {
            if (*total == n + 1u) { stop = true; break; }
            __nanosleep(40);
        }
        if (stop) break;
        const LnTileMeta m = metas[n % kLnMetaRing];
        unsigned s = slot;
        for (int k = 0; k < p.K; ++k) {
            tma_store_box(tmap_out, smem + sm.off_ring + (size_t)s * kLnBoxBytes, m.t0, k * kLnBoxRows, m.b);
            if (++s == R) s = 0;
        }
        bulk_commit();
        bulk_wait_read<0>();                         // the engine has read the boxes: hand them back to the loader
        for (int k = 0; k < p.K; ++k) {
            mbar_arrive(&empty[slot]);
            if (++slot == R) slot = 0;
        }
    }
    bulk_wait_all<0>();
}

// cross-warp stage of a per-frame reduction: the lanes that carry a warp's result for frame f write it to
// red[f][w][0..NV), everybody meets, warp f (< 8) merges the 16 partials of frame f and lane 0 of it finalises.
template <int NV>
__device__ __forceinline__ void red_store(float *red, int f, int w, const float (&v)[NV]) {
#pragma unroll
    for (int i = 0; i < NV; ++i) red[(f * 16 + w) * 4 + i] = v[i];
}

// A box slot and its barrier phase, advanced without a division.
struct SlotIter {
    unsigned slot, phase;
    __device__ __forceinline__ void next(unsigned R) { if (++slot == R) { slot = 0; phase ^= 1u; } }
};
__device__ __forceinline__ void mbar_spin(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) { }                              // try_wait suspends the thread in hardware while it waits
}

// ---- round 1 of the tile kernels: mean and centred second moment of every frame (asr/nn/layernorm.py:41-44) ----
// z: this thread's rows 240k + 16w + lane/2 of frames 4h .. 4h+3, zeros where a row does not exist (fn of them do; fmissing
// = KMAX - fn).  Per thread, then over the 16 lanes of a half, then over the warps through `red`: after one meeting of
// the compute warps, lane 0 of warp f < 8 hands frame f's (count, mean, centred second moment) over all V rows to
// `finish`.  Returns the frame this lane's half-warp result belongs to (4h + the returned value).
template <int KMAX, typename F>
__device__ __forceinline__ int ln_frame_moments(const float4 (&z)[KMAX], float fn, float inv_n, float fmissing, int lane, int h,
                                                int w, float *red, F finish) {
    Moments mo[4];
    {
        float sx = 0.f, sy = 0.f, sz = 0.f, sw = 0.f;
#pragma unroll
        for (int k = 0; k < KMAX; ++k) { sx += z[k].x; sy += z[k].y; sz += z[k].z; sw += z[k].w; }      // missing rows are zeros
        const float mx_ = sx * inv_n, my_ = sy * inv_n, mz_ = sz * inv_n, mw_ = sw * inv_n;
        float qx = 0.f, qy = 0.f, qz = 0.f, qw = 0.f;
#pragma unroll
        for (int k = 0; k < KMAX; ++k) {
            const float dx = z[k].x - mx_, dy = z[k].y - my_, dz = z[k].z - mz_, dw = z[k].w - mw_;
            qx = fmaf(dx, dx, qx); qy = fmaf(dy, dy, qy); qz = fmaf(dz, dz, qz); qw = fmaf(dw, dw, qw);
        }
        // a missing row read as 0 and contributed mean^2: take that back
        mo[0].mean = mx_; mo[0].m2 = fmaf(-fmissing * mx_, mx_, qx);
        mo[1].mean = my_; mo[1].m2 = fmaf(-fmissing * my_, my_, qy);
        mo[2].mean = mz_; mo[2].m2 = fmaf(-fmissing * mz_, mz_, qz);
        mo[3].mean = mw_; mo[3].m2 = fmaf(-fmissing * mw_, mw_, qw);
        mo[0].n = mo[1].n = mo[2].n = mo[3].n = fn;
    }
    int fih;
    const Moments mr = reduce_frames16(mo[0], mo[1], mo[2], mo[3], lane, merge_moments, fih);
    if (lane < 8) { const float v3[3] = {mr.n, mr.mean, mr.m2}; red_store<3>(red, 4 * h + fih, w, v3); }
    bar_compute();
    if (w < kLnTT) {
        Moments a;
        const float *src = red + (w * 16 + (lane & 15)) * 4;
        a.n = src[0]; a.mean = src[1]; a.m2 = src[2];
        if ((lane & 15) >= kLnWarps) { a.n = 0.f; a.mean = 0.f; a.m2 = 0.f; }
#pragma unroll
        for (int o = 1; o < 16; o <<= 1) a = merge_moments(a, Moments::shfl_xor(a, o));
        if (lane == 0) finish(a);
    }
    return fih;
}


// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
// 104 registers per thread: 512 threads then leave 12K of the SM's 64K registers to a lattice CTA, which runs next
// to this kernel exactly as it runs next to the row kernel (api.cu).
// Rows that do not exist (v >= V: the tail of the last box, read as zeros, and register slots k >= K) are made
// neutral by DATA, not by predicates: their gamma is 0 and their beta -inf in the shared-memory table, so their
// activation is -inf -- never a maximum, probability 0 -- and the one place where a zero row is not neutral, the centred
// second moment, is corrected in closed form.
template <int KMAX>
__global__ void __maxnreg__(104) ln_softmax_gather_kernel(const __grid_constant__ CUtensorMap tmap, LnParams p, LnSmem sm) {
    extern __shared__ __align__(128) unsigned char smem[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + sm.off_full);
    uint64_t *empty = reinterpret_cast<uint64_t *>(smem + sm.off_empty);
    LnTileMeta *metas = reinterpret_cast<LnTileMeta *>(smem + sm.off_meta);
    float *red = reinterpret_cast<float *>(smem + sm.off_red);
    float *tot = reinterpret_cast<float *>(smem + sm.off_tot);
    float *gb = reinterpret_cast<float *>(smem + sm.off_gb);
    const uint32_t ring = smem_u32(smem + sm.off_ring);
    const ProblemDesc &d = p.d;
    const unsigned R = (unsigned)p.R;
    const int K = p.K;
    constexpr int Vt = KMAX * kLnBoxRows;                 // rows of the gamma/beta table
    if (threadIdx.x == 0) {
        for (unsigned i = 0; i < R; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], kLnWarps); }
        mbar_init_fence();
        reinterpret_cast<LnSignalFifo *>(smem + sm.off_fifo)->head = 0u;
        reinterpret_cast<LnSignalFifo *>(smem + sm.off_fifo)->tail = 0u;
    }
    for (int i = threadIdx.x; i < Vt; i += blockDim.x) {
        gb[i] = i < d.V ? __ldg(p.gamma + i) : 0.f;
        gb[Vt + i] = i < d.V ? __ldg(p.beta + i) : -INFINITY;
    }
    __syncthreads();
    const int w = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31;
    LnSignalFifo *fifo = reinterpret_cast<LnSignalFifo *>(smem + sm.off_fifo);
    if (w == kLnWarps) {
        if (lane == 0) ln_producer<kLnForward>(&tmap, nullptr, p, smem, sm);
        else if (lane == 1 && d.concurrent) ln_signaller(p, smem, sm);
        return;
    }
    const int r = lane >> 1, h = lane & 1;
    const int vrow = 16 * w + r;                          // this thread's row inside every box
    int nrows = 0;
#pragma unroll
    for (int k = 0; k < KMAX; ++k) nrows += (k < K && kLnBoxRows * k + vrow < d.V) ? 1 : 0;
    const float fn = (float)nrows, inv_n = nrows > 0 ? 1.f / (float)nrows : 0.f, fmissing = (float)(KMAX - nrows);
    const uint32_t lane_off = (uint32_t)(w * 512 + lane * 16);
    float *mu_out = reinterpret_cast<float *>(p.ws + p.off_mu);
    float *rstd_out = reinterpret_cast<float *>(p.ws + p.off_rstd);
    float *lse_out = reinterpret_cast<float *>(p.ws + p.off_lse);
    float2 *lp_out = reinterpret_cast<float2 *>(p.ws + p.w.off_lp);
    const int tid = threadIdx.x;

    SlotIter it = {0u, 0u};
    unsigned seq = 0, pushed = 0;
    for (;;) {
        mbar_spin(&full[it.slot], it.phase);
        const LnTileMeta m = metas[seq % kLnMetaRing];
        ++seq;
        if (m.kind < 0) break;
        const int Tb = m.Tb, Lb = m.Lb;
        const EmissionColumns cols(d, m.b);
        const int ncol = cols.count(Lb);
        // the id of this thread's emission column (thread c takes column c of WsLayout::W), requested now: its round trip
        // hides behind the tile load and the moments
        int sym = -1;
        if (tid < ncol) sym = cols.symbol(tid, Lb);
        // ---- the tile into registers: rows 240k + 16w + r, frames 4h .. 4h+3; the threads that own an emission column
        //      pick up their symbol's row on the way.  Every box goes back to the loader as soon as this warp has read it:
        //      the ring is a sliding window of boxes in flight ----
        float4 z[KMAX];
        float4 zs0 = make_float4(0.f, 0.f, 0.f, 0.f), zs1 = zs0;
        if (!(sym >= 0 && sym < d.V)) sym = -1;
        const int sym_box = sym >= 0 ? sym / kLnBoxRows : -1;
        const uint32_t sym_off = sym >= 0 ? (uint32_t)((sym % kLnBoxRows) * 32) : 0u;
        {
            SlotIter s = it;
#pragma unroll
            for (int k = 0; k < KMAX; ++k) {
                z[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (k < K) {
                    if (k > 0) mbar_spin(&full[s.slot], s.phase);
                    const uint32_t box = ring + s.slot * kLnBoxBytes;
                    z[k] = lds128(box + lane_off);
                    if (sym_box == k) { zs0 = lds128(box + sym_off); zs1 = lds128(box + sym_off + 16); }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&empty[s.slot]);
                    s.next(R);
                }
            }
            it = s;
        }

        // ---- round 1: mean and centred second moment of every frame (asr/nn/layernorm.py:41-44) ----
        int fih = ln_frame_moments<KMAX>(z, fn, inv_n, fmissing, lane, h, w, red, [&](const Moments &a) {
            const float var = fmaxf(a.m2, 0.f) / a.n;                      // sum(diff^2) / size, no epsilon (:44)
            const float rstd = 1.f / sqrtf(var);
            tot[w * 8 + 0] = a.mean;
            tot[w * 8 + 1] = rstd;
            const int t = m.t0 + w;
            if (t < Tb) { mu_out[(size_t)m.b * p.Tq + t] = a.mean; rstd_out[(size_t)m.b * p.Tq + t] = rstd; }
        });
        bar_compute();

        // ---- round 2: a = gamma * (z - mean) * rstd + beta (asr/nn/nn.py:265), in place; softmax statistics ----
        MaxSum ms[4];
        {
            float rs[4], mur[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) { rs[j] = tot[(4 * h + j) * 8 + 1]; mur[j] = -tot[(4 * h + j) * 8 + 0] * rs[j]; }
            float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
#pragma unroll
            for (int k = 0; k < KMAX; ++k) {
                const float gk = gb[kLnBoxRows * k + vrow], bk = gb[Vt + kLnBoxRows * k + vrow];      // (0, -inf) for a missing row
                z[k].x = fmaf(fmaf(z[k].x, rs[0], mur[0]), gk, bk); m0 = fmaxf(m0, z[k].x);
                z[k].y = fmaf(fmaf(z[k].y, rs[1], mur[1]), gk, bk); m1 = fmaxf(m1, z[k].y);
                z[k].z = fmaf(fmaf(z[k].z, rs[2], mur[2]), gk, bk); m2 = fmaxf(m2, z[k].z);
                z[k].w = fmaf(fmaf(z[k].w, rs[3], mur[3]), gk, bk); m3 = fmaxf(m3, z[k].w);
            }
            const float c0 = m0 == -INFINITY ? 0.f : -m0 * LOG2E_HI, c1 = m1 == -INFINITY ? 0.f : -m1 * LOG2E_HI;
            const float c2 = m2 == -INFINITY ? 0.f : -m2 * LOG2E_HI, c3 = m3 == -INFINITY ? 0.f : -m3 * LOG2E_HI;
            float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
            for (int k = 0; k < KMAX; ++k) {
                s0 += ex2_approx(fmaf(z[k].x, LOG2E_HI, c0));
                s1 += ex2_approx(fmaf(z[k].y, LOG2E_HI, c1));
                s2 += ex2_approx(fmaf(z[k].z, LOG2E_HI, c2));
                s3 += ex2_approx(fmaf(z[k].w, LOG2E_HI, c3));
            }
            ms[0].m = m0; ms[0].s = s0; ms[1].m = m1; ms[1].s = s1; ms[2].m = m2; ms[2].s = s2; ms[3].m = m3; ms[3].s = s3;
        }
        const MaxSum sr = reduce_frames16(ms[0], ms[1], ms[2], ms[3], lane, merge_maxsum, fih);
        if (lane < 8) { const float v2[2] = {sr.m, sr.s}; red_store<2>(red, 4 * h + fih, w, v2); }
        bar_compute();
        if (w < kLnTT) {
            MaxSum a;
            const float *src = red + (w * 16 + (lane & 15)) * 4;
            a.m = src[0]; a.s = src[1];
            if ((lane & 15) >= kLnWarps) { a.m = -INFINITY; a.s = 0.f; }
#pragma unroll
            for (int o = 1; o < 16; o <<= 1) a = merge_maxsum(a, MaxSum::shfl_xor(a, o));
            if (lane == 0) {
                float la, lb;
                split_lse2(a.m, a.s, la, lb);
                tot[w * 8 + 2] = la;
                tot[w * 8 + 3] = lb;
                const int t = m.t0 + w;
                if (t < Tb) lse_out[(size_t)m.b * p.Tq + t] = la + lb;
            }
        }
        bar_compute();

        // ---- emission probabilities of the lattice's symbols ----
        if (tid < ncol) {
            const float zz[8] = {zs0.x, zs0.y, zs0.z, zs0.w, zs1.x, zs1.y, zs1.z, zs1.w};
            const float gs = sym >= 0 ? gb[sym] : 0.f, bs = sym >= 0 ? gb[Vt + sym] : 0.f;
#pragma unroll
            for (int f = 0; f < kLnTT; ++f) {
                const int t = m.t0 + f;
                if (t < Tb) {
                    float2 v = make_float2(0.f, SENT);
                    if (sym >= 0) {
                        const float a = fmaf((zz[f] - tot[f * 8 + 0]) * tot[f * 8 + 1], gs, bs);
                        v = emission_pair(a, tot[f * 8 + 2], tot[f * 8 + 3]);
                    }
                    lp_out[((size_t)m.b * d.T + t) * p.w.W + tid] = v;
                }
            }
        }
        bar_compute();            // rows stored; also protects red/tot against the next tile
        if (tid == 0 && d.concurrent) ln_signal_push(fifo, pushed, m.b, m.t0 / kProgBlock, min(kLnTT, Tb - m.t0));
    }
    if (tid == 0 && d.concurrent) ln_signal_push(fifo, pushed, -1, 0, 0);
}

// ---------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------
// Rows that do not exist get gamma = beta = 0 in the shared-memory table: their dn is 0 (nothing enters the per-frame
// sums) and what they add to this thread's dgamma/dbeta slots is never stored.  Frames that do not exist (padding) get
// rstd = 0 and a log2 normaliser of -inf (softmax 0), which makes every quantity of theirs exactly zero.  No predicates in
// the sweeps.
// dz leaves as it came in: sweep 2 writes each box's image over the z it was computed from, and lane 1 of the producer
// warp hands the boxes to the TMA engine as tile stores (an SM storing 32-byte pieces itself spends 16 L1 wavefronts
// per instruction: the LSU, not HBM, bounded the first version of this kernel).
template <int KMAX>
__global__ void __launch_bounds__(kLnThreads, 1) ln_gradient_kernel(const __grid_constant__ CUtensorMap tmap,
                                                                     const __grid_constant__ CUtensorMap tmap_dz, LnParams p,
                                                                     LnSmem sm) {
    extern __shared__ __align__(128) unsigned char smem[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + sm.off_full);
    uint64_t *empty = reinterpret_cast<uint64_t *>(smem + sm.off_empty);
    uint64_t *abbar = reinterpret_cast<uint64_t *>(smem + sm.off_abbar);
    LnTileMeta *metas = reinterpret_cast<LnTileMeta *>(smem + sm.off_meta);
    float *red = reinterpret_cast<float *>(smem + sm.off_red);
    float *tot = reinterpret_cast<float *>(smem + sm.off_tot);
    const float *fc = reinterpret_cast<const float *>(smem + sm.off_fc);
    float *post = reinterpret_cast<float *>(smem + sm.off_post);
    float *ebuf = reinterpret_cast<float *>(smem + sm.off_ebuf);
    int *csr = reinterpret_cast<int *>(smem + sm.off_csr);
    float *gb = reinterpret_cast<float *>(smem + sm.off_gb);
    unsigned *bm_sm = reinterpret_cast<unsigned *>(smem + sm.off_bm);
    const uint32_t ring = smem_u32(smem + sm.off_ring);
    const ProblemDesc &d = p.d;
    const WsLayout &wl = p.w;
    const unsigned R = (unsigned)p.R;
    const int K = p.K;
    constexpr int Vt = KMAX * kLnBoxRows;
    const int Upad = (wl.Umax + 3) & ~3;
    const int Nst = wl.Np;                                // row pitch of ebuf
    float *bpart = ebuf + (size_t)kLnTT * wl.Np;          // [frame][32-node chunk] partial sums over the blank nodes
    if (threadIdx.x == 0) {
        for (unsigned i = 0; i < R; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        mbar_init(&abbar[0], 1);
        mbar_init(&abbar[1], 1);
        mbar_init(&abbar[2], 1);
        mbar_init_fence();
        reinterpret_cast<LnSignalFifo *>(smem + sm.off_fifo)->head = 0u;
    }
    for (int i = threadIdx.x; i < Vt; i += blockDim.x) {
        gb[i] = i < d.V ? __ldg(p.gamma + i) : 0.f;
        gb[Vt + i] = i < d.V ? __ldg(p.beta + i) : 0.f;
    }
    for (int i = threadIdx.x; i < 2 * (Vt / 32 + 1); i += blockDim.x) bm_sm[i] = 0u;
    for (int i = threadIdx.x; i < (int)(kLnBoxBytes / 4); i += blockDim.x) reinterpret_cast<float *>(smem + sm.off_zero)[i] = 0.f;
    fence_proxy_async_smem();                             // the zero box is read by the TMA engine
    __syncthreads();
    const int w = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31;
    if (w == kLnWarps) {
        if (lane == 0) ln_producer<kLnBackward>(&tmap, &tmap_dz, p, smem, sm);
        else if (lane == 1) ln_storer(&tmap_dz, p, smem, sm);
        return;
    }
    const int r = lane >> 1, h = lane & 1;
    const int vrow = 16 * w + r;
    const int tid = threadIdx.x;
    const uint32_t lane_off = (uint32_t)(w * 512 + lane * 16);
    const int per = d.kind == 0 ? 2 : 3;
    const float inv_v = 1.f / (float)d.V;
    const int nwt = Vt / 32 + 1;                          // words of the bitmap / prefix tables in shared memory
    // dgamma (h = 0) or dbeta (h = 1) of this thread's rows: the two threads of a row add up their halves of every tile
    // with one shuffle and keep one sum each (one register per box instead of two: sweep 1 is the register peak)
    float dgb[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) dgb[k] = 0.f;

    SlotIter it = {0u, 0u};
    unsigned seq = 0, n_ab = 0;
    for (;;) {
        mbar_spin(&full[it.slot], it.phase);
        const LnTileMeta m = metas[seq % kLnMetaRing];
        ++seq;
        if (m.kind < 0) {
            // tell the store lane how many tiles there were (see ln_storer for why this is not a barrier arrival)
            if (tid == 0) *reinterpret_cast<volatile unsigned *>(&reinterpret_cast<LnSignalFifo *>(smem + sm.off_fifo)->head) = seq;
            break;
        }
        // ---- phase (a): merged posteriors of the tile's frames (gram_ctc.py:180-217, :290), all warps ----
        // requested first, used last: this utterance's symbol tables (prep.cuh)
        {
            const int *uoff = reinterpret_cast<const int *>(p.ws + wl.off_uoff) + (size_t)m.b * (wl.Nmax + 1);
            const int *unode = reinterpret_cast<const int *>(p.ws + wl.off_unode) + (size_t)m.b * wl.Nmax;
            const unsigned *bm_g = reinterpret_cast<const unsigned *>(p.ws + wl.off_bm) + (size_t)m.b * wl.nwords;
            const int *pc_g = reinterpret_cast<const int *>(p.ws + wl.off_pc) + (size_t)m.b * wl.nwords;
            for (int i = tid; i <= m.Ub; i += 32 * kLnWarps) csr[i] = __ldg(uoff + i);
            for (int i = tid; i < m.Nb; i += 32 * kLnWarps) csr[wl.Nmax + 1 + i] = __ldg(unode + i);
            for (int i = tid; i < wl.nwords; i += 32 * kLnWarps) { bm_sm[i] = __ldg(bm_g + i); bm_sm[nwt + i] = (unsigned)__ldg(pc_g + i); }
        }
        // Joint objective: each blank / unigram node of the Gram-CTC lattice shares its symbol occurrence with one node of
        // the plain-CTC lattice (3i <-> 2i, 3i+1 <-> 2i+1; bigram nodes have no partner, gradient.cu joint_partner).
        // Adding the partner's posterior to e[j] leaves the per-id merge, the blank sums and sweep 2 as they are.  The
        // partner's alpha/beta come from global memory straight into registers, requested here so that their round trip
        // hides behind the wait for the Gram-CTC rows: no shared memory is taken from the ring.  The plain-CTC lattice's P
        // comes the same way (not in the tile record: a larger record would take shared memory from the ring too).
        const int nfv = min(kLnTT, m.Tb - m.t0);
        const int Nbp = (m.Nb + 31) & ~31;
        const int nitems = nfv * Nbp;
        const float2 *a2g = reinterpret_cast<const float2 *>(p.ws + wl.off_av2) + ((size_t)m.b * d.T + m.t0) * wl.Np2;
        const float2 *b2g = reinterpret_cast<const float2 *>(p.ws + wl.off_bv2) + ((size_t)m.b * d.T + m.t0) * wl.Np2 + 1;
        auto ctc_partner_ab = [&](int i) {                // (alpha.m, alpha.e, beta.m, beta.e); probability 0 if none
            float4 v = make_float4(0.f, SENT, 0.f, SENT);
            const int f = i / Nbp, j = i - f * Nbp;
            if (wl.joint && j < m.Nb && j % 3 != 2) {
                const int jc = 2 * (j / 3) + j % 3;
                const float2 a = __ldg(a2g + (size_t)f * wl.Np2 + jc), bb = __ldg(b2g + (size_t)f * wl.Np2 + jc);
                v = make_float4(a.x, a.y, bb.x, bb.y);
            }
            return v;
        };
        float Ph2 = 0.f, Pl2 = 0.f;
        if (wl.joint) {
            const UttInfo *u2 = reinterpret_cast<const UttInfo *>(p.ws + wl.off_utt2) + m.b;
            Ph2 = __ldg(&u2->Ph);
            Pl2 = __ldg(&u2->Pl);
        }
        float4 ab2[kLnJointPre];
#pragma unroll
        for (int q = 0; q < kLnJointPre; ++q) {
            const int i = tid + q * 32 * kLnWarps;
            ab2[q] = (wl.joint && i < nitems) ? ctc_partner_ab(i) : make_float4(0.f, SENT, 0.f, SENT);
        }
        mbar_spin(&abbar[0], n_ab & 1u);
        ++n_ab;
        // per-frame constants of this thread's four frames (staged by the producer)
        float rs[4], mur[4], nl[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const bool valid = m.t0 + 4 * h + j < m.Tb;
            const float rr = valid ? fc[kLnTT + 4 * h + j] : 0.f;
            rs[j] = rr; mur[j] = valid ? -fc[4 * h + j] * rr : 0.f;
            nl[j] = valid ? -fc[2 * kLnTT + 4 * h + j] : -INFINITY;
        }
        const float scs = wl.joint ? 2.f * m.sc : m.sc;                     // joint: two losses, two softmax terms
        {
            // alpha * beta / P of every node of every valid frame
            const float2 *a_sm = reinterpret_cast<const float2 *>(smem + sm.off_ab);
            const float2 *b_sm = a_sm + (size_t)kLnTT * wl.Np;
            // a warp's 32 items are 32 consecutive nodes of ONE frame (Nbp and the stride are multiples of 32): the blank
            // nodes among them are summed by shuffle and left as one partial per 32-node chunk, summed in order below
            auto node_item = [&](int i, const float4 &c2) {
                const int f = i / Nbp, j = i - f * Nbp;
                float e = 0.f;
                if (j < m.Nb) {
                    e = node_posterior(a_sm[f * wl.Np + j], b_sm[f * wl.Np + j + wl.boff], m.Ph, m.Pl);
                    if (wl.joint && j % 3 != 2) e += node_posterior(make_float2(c2.x, c2.y), make_float2(c2.z, c2.w), Ph2, Pl2);
                    ebuf[f * Nst + j] = e;
                }
                const float bp = warp_sum((j < m.Nb && j % per == 0) ? e : 0.f);
                if (lane == 0) bpart[f * kLnBlankChunks + (j >> 5)] = bp;
            };
#pragma unroll
            for (int q = 0; q < kLnJointPre; ++q) {
                const int i = tid + q * 32 * kLnWarps;
                if (i < nitems) node_item(i, ab2[q]);
            }
            // long lattices (joint: more than kLnJointPre items per thread): the rest loads as it goes
            for (int i = tid + kLnJointPre * 32 * kLnWarps; i < nitems; i += 32 * kLnWarps) node_item(i, ctc_partner_ab(i));
        }
        bar_compute();
        if (tid == 0) mbar_arrive(&abbar[1]);                                 // alpha/beta and the frame constants can be refilled
        {
            // merged per emitted id, in node order (deterministic); the blank collects every per-th node
            for (int i = tid; i < kLnTT * m.Ub; i += 32 * kLnWarps) {
                const int f = i / m.Ub, u = i - f * m.Ub;
                float ps = 0.f;
                if (f < nfv) {
                    const float *e = ebuf + f * Nst;
                    if (u == m.ublank)
                        for (int c = 0; c < (m.Nb + 31) / 32; ++c) ps += bpart[f * kLnBlankChunks + c];
                    const int n0 = csr[u], n1 = csr[u + 1];
                    for (int n = n0; n < n1; ++n) {
                        const int j = csr[wl.Nmax + 1 + n];
                        if (j < m.Nb) ps += e[j];
                    }
                    ps *= m.sc;
                }
                post[f * Upad + u] = ps;
            }
        }
        bar_compute();

        // ---- sweep 1: g = softmax * sc - posterior;  dn = g * gamma;  per-frame sums of dn and dn * n ----
        float4 dn[KMAX];
        float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
        const SlotIter first = it;
        const float *prow0 = post + (4 * h) * Upad;
        {
            SlotIter s = it;
#pragma unroll
            for (int k = 0; k < KMAX; ++k) {
                dn[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (k < K) {
                    if (k > 0) mbar_spin(&full[s.slot], s.phase);
                    const float4 zq = lds128(ring + s.slot * kLnBoxBytes + lane_off);
                    s.next(R);
                    const int v = kLnBoxRows * k + vrow;
                    const float g_ = gb[v], b_ = gb[Vt + v];
                    const unsigned word = bm_sm[v >> 5];
                    float p0 = 0.f, p1 = 0.f, p2 = 0.f, p3 = 0.f;
                    if ((word >> (v & 31)) & 1u) {                             // ~2% of the rows: ids the lattice emits
                        const int u = (int)bm_sm[nwt + (v >> 5)] + __popc(word & ((1u << (v & 31)) - 1u));
                        p0 = prow0[u]; p1 = prow0[Upad + u]; p2 = prow0[2 * Upad + u]; p3 = prow0[3 * Upad + u];
                    }
                    const float n0 = fmaf(zq.x, rs[0], mur[0]), n1 = fmaf(zq.y, rs[1], mur[1]);
                    const float n2 = fmaf(zq.z, rs[2], mur[2]), n3 = fmaf(zq.w, rs[3], mur[3]);
                    const float g0 = fmaf(ex2_approx(fmaf(fmaf(n0, g_, b_), LOG2E_HI, nl[0])), scs, -p0);
                    const float g1 = fmaf(ex2_approx(fmaf(fmaf(n1, g_, b_), LOG2E_HI, nl[1])), scs, -p1);
                    const float g2 = fmaf(ex2_approx(fmaf(fmaf(n2, g_, b_), LOG2E_HI, nl[2])), scs, -p2);
                    const float g3 = fmaf(ex2_approx(fmaf(fmaf(n3, g_, b_), LOG2E_HI, nl[3])), scs, -p3);
                    const float d0 = g0 * g_, d1 = g1 * g_, d2 = g2 * g_, d3 = g3 * g_;
                    s1[0] += d0; s1[1] += d1; s1[2] += d2; s1[3] += d3;
                    s2[0] = fmaf(d0, n0, s2[0]); s2[1] = fmaf(d1, n1, s2[1]); s2[2] = fmaf(d2, n2, s2[2]); s2[3] = fmaf(d3, n3, s2[3]);
                    const float tb = (g0 + g1) + (g2 + g3);                    // bias backward: sum over (b, t)
                    const float tg = fmaf(g0, n0, fmaf(g1, n1, fmaf(g2, n2, g3 * n3)));      // scale backward
                    dgb[k] += (h ? tb : tg) + __shfl_xor_sync(0xffffffffu, h ? tg : tb, 1);
                    dn[k] = make_float4(d0, d1, d2, d3);
                }
            }
            it = s;
        }
        // ---- the two per-frame sums of LayerNormalization's backward (asr/nn/layernorm.py:48-60) ----
        int fih;
        const Pair2 pr = reduce_frames16(Pair2{s1[0], s2[0]}, Pair2{s1[1], s2[1]}, Pair2{s1[2], s2[2]}, Pair2{s1[3], s2[3]}, lane,
                                         merge_pair2, fih);
        if (lane < 8) { const float v2[2] = {pr.a, pr.b}; red_store<2>(red, 4 * h + fih, w, v2); }
        bar_compute();
        if (w < kLnTT) {
            const float *src = red + (w * 16 + (lane & 15)) * 4;
            float a = src[0], b = src[1];
            if ((lane & 15) >= kLnWarps) { a = 0.f; b = 0.f; }
#pragma unroll
            for (int o = 1; o < 16; o <<= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
            if (lane == 0) { tot[w * 8 + 0] = a * inv_v; tot[w * 8 + 1] = b * inv_v; }
        }
        bar_compute();
        float c1r[4], c2r[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { c1r[j] = -tot[(4 * h + j) * 8 + 0] * rs[j]; c2r[j] = -tot[(4 * h + j) * 8 + 1] * rs[j]; }

        // ---- sweep 2: dz = rstd * (dn - mean_v(dn) - n * mean_v(dn * n)), written over the z it came from ----
        {
            SlotIter s = first;
#pragma unroll
            for (int k = 0; k < KMAX; ++k) {
                if (k < K) {
                    const uint32_t addr = ring + s.slot * kLnBoxBytes + lane_off;
                    const float4 zq = lds128(addr);
                    float4 o;
                    o.x = fmaf(fmaf(zq.x, rs[0], mur[0]), c2r[0], fmaf(dn[k].x, rs[0], c1r[0]));
                    o.y = fmaf(fmaf(zq.y, rs[1], mur[1]), c2r[1], fmaf(dn[k].y, rs[1], c1r[1]));
                    o.z = fmaf(fmaf(zq.z, rs[2], mur[2]), c2r[2], fmaf(dn[k].z, rs[2], c1r[2]));
                    o.w = fmaf(fmaf(zq.w, rs[3], mur[3]), c2r[3], fmaf(dn[k].w, rs[3], c1r[3]));
                    sts128(addr, o);
                    s.next(R);
                }
            }
        }
        fence_proxy_async_smem();     // the images are read by the TMA engine
        bar_compute();                // images complete; red / tot / post / tables are reused by the next tile
        if (tid == 0) mbar_arrive(&abbar[2]);      // store lane: this tile's boxes are ready
    }
    // ---- this CTA's share of dgamma / dbeta: one partial row per CTA ----
    const int Vp = K * kLnBoxRows;
    float *part = reinterpret_cast<float *>(p.ws + p.off_part) + (size_t)blockIdx.x * 2 * Vp + (size_t)h * Vp;
#pragma unroll
    for (int k = 0; k < KMAX; ++k)
        if (k < K) part[kLnBoxRows * k + vrow] = dgb[k];
}

// dgamma[v] = sum over CTAs of their partial rows, in CTA order (deterministic)
__global__ void ln_reduce_params_kernel(const float *part, int nparts, int Vp, int V, float *dgamma, float *dbeta) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= V) return;
    float g = 0.f, b = 0.f;
    for (int c = 0; c < nparts; ++c) {
        g += part[(size_t)c * 2 * Vp + v];
        b += part[(size_t)c * 2 * Vp + Vp + v];
    }
    if (dgamma) dgamma[v] = g;
    if (dbeta) dbeta[v] = b;
}

// ---------------------------------------------------------------------------------------------
// greedy argmax (the development loop, run/ctc/cnn/train.py:224-234: xp.argmax(y.data, axis=2) on the normalised output)
// ---------------------------------------------------------------------------------------------
constexpr int kLnNoRow = 0x7fffffff;      // "no candidate": loses to every real row, whatever its value
struct ArgMax {                           // best normalised value of a frame so far and its vocabulary row
    float v;
    int i;
    static __device__ __forceinline__ ArgMax shfl_xor(const ArgMax &a, int o) {
        ArgMax r;
        r.v = __shfl_xor_sync(0xffffffffu, a.v, o);
        r.i = __shfl_xor_sync(0xffffffffu, a.i, o);
        return r;
    }
};
// numpy.argmax order: a NaN above everything, then the larger value, then (equal values, or two NaNs) the smaller row.
// The merges run in an order that depends on which lane owns which rows, so ties are broken by the row, never by order.
__device__ __forceinline__ ArgMax merge_argmax(const ArgMax &a, const ArgMax &b) {
    const bool an = a.v != a.v, bn = b.v != b.v;
    const bool take_b = an != bn ? bn : (b.v > a.v || (!(b.v < a.v) && b.i < a.i));
    return take_b ? b : a;
}

// One read of z, no workspace: round 1 as in the forward kernel, then every thread keeps the best (value, row) of its four
// frames over its rows and the CTA merges them like the softmax statistics.  Rows v >= V are excluded by index: the
// value of a row is no protection in a frame whose values are all NaN.  A frame with a NaN or an infinity anywhere gives
// 0 (the reference's every normalised value is NaN then), and so does a frame of zeros (0/0).
template <int KMAX>
__global__ void __launch_bounds__(kLnThreads, 1) ln_argmax_kernel(const __grid_constant__ CUtensorMap tmap, LnParams p, LnSmem sm,
                                                                  int64_t *out) {
    extern __shared__ __align__(128) unsigned char smem[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + sm.off_full);
    uint64_t *empty = reinterpret_cast<uint64_t *>(smem + sm.off_empty);
    LnTileMeta *metas = reinterpret_cast<LnTileMeta *>(smem + sm.off_meta);
    float *red = reinterpret_cast<float *>(smem + sm.off_red);
    float *tot = reinterpret_cast<float *>(smem + sm.off_tot);
    float *gb = reinterpret_cast<float *>(smem + sm.off_gb);
    const uint32_t ring = smem_u32(smem + sm.off_ring);
    const ProblemDesc &d = p.d;
    const unsigned R = (unsigned)p.R;
    const int K = p.K;
    constexpr int Vt = KMAX * kLnBoxRows;
    if (threadIdx.x == 0) {
        for (unsigned i = 0; i < R; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], kLnWarps); }
        mbar_init_fence();
    }
    for (int i = threadIdx.x; i < Vt; i += blockDim.x) {
        gb[i] = i < d.V ? __ldg(p.gamma + i) : 0.f;
        gb[Vt + i] = i < d.V ? __ldg(p.beta + i) : 0.f;
    }
    __syncthreads();
    const int w = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31;
    if (w == kLnWarps) {
        if (lane == 0) ln_producer<kLnArgmax>(&tmap, nullptr, p, smem, sm);
        return;
    }
    const int r = lane >> 1, h = lane & 1;
    const int vrow = 16 * w + r;
    int nrows = 0;                                        // this thread's rows that exist: k < nrows
#pragma unroll
    for (int k = 0; k < KMAX; ++k) nrows += (k < K && kLnBoxRows * k + vrow < d.V) ? 1 : 0;
    const float fn = (float)nrows, inv_n = nrows > 0 ? 1.f / (float)nrows : 0.f, fmissing = (float)(KMAX - nrows);
    const uint32_t lane_off = (uint32_t)(w * 512 + lane * 16);

    SlotIter it = {0u, 0u};
    unsigned seq = 0;
    for (;;) {
        mbar_spin(&full[it.slot], it.phase);
        const LnTileMeta m = metas[seq % kLnMetaRing];
        ++seq;
        if (m.kind < 0) break;
        float4 z[KMAX];
        {
            SlotIter s = it;
#pragma unroll
            for (int k = 0; k < KMAX; ++k) {
                z[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (k < K) {
                    if (k > 0) mbar_spin(&full[s.slot], s.phase);
                    z[k] = lds128(ring + s.slot * kLnBoxBytes + lane_off);
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&empty[s.slot]);
                    s.next(R);
                }
            }
            it = s;
        }

        // ---- round 1 ----
        int fih = ln_frame_moments<KMAX>(z, fn, inv_n, fmissing, lane, h, w, red, [&](const Moments &a) {
            const float rstd = 1.f / sqrtf(fmaxf(a.m2, 0.f) / a.n);
            // a NaN or an infinity in the frame leaves a NaN mean or a NaN second moment (inf - inf); make the mean NaN
            // so that every value of the frame is NaN, as in the reference -- fmaxf above would have hidden a NaN m2
            tot[w * 8 + 0] = (a.mean != a.mean || a.m2 != a.m2) ? __int_as_float(0x7fc00000) : a.mean;
            tot[w * 8 + 1] = rstd;
        });
        bar_compute();

        // ---- round 2: a = gamma * (z - mean) * rstd + beta (asr/nn/nn.py:265); best (value, row) of each frame ----
        ArgMax am[4];
        {
            float rs[4], mur[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) { rs[j] = tot[(4 * h + j) * 8 + 1]; mur[j] = -tot[(4 * h + j) * 8 + 0] * rs[j]; }
            float bv[4];
            int bi[4];
            {                                             // row k = 0 (it exists unless V <= 16w + lane/2)
                const float g0 = gb[vrow], b0 = gb[Vt + vrow];
                const bool has = nrows > 0;
                bv[0] = has ? fmaf(fmaf(z[0].x, rs[0], mur[0]), g0, b0) : -INFINITY;
                bv[1] = has ? fmaf(fmaf(z[0].y, rs[1], mur[1]), g0, b0) : -INFINITY;
                bv[2] = has ? fmaf(fmaf(z[0].z, rs[2], mur[2]), g0, b0) : -INFINITY;
                bv[3] = has ? fmaf(fmaf(z[0].w, rs[3], mur[3]), g0, b0) : -INFINITY;
                bi[0] = bi[1] = bi[2] = bi[3] = has ? vrow : kLnNoRow;
            }
#pragma unroll
            for (int k = 1; k < KMAX; ++k) {
                if (k < nrows) {                          // rows ascend with k: a strict win keeps the first of equal values
                    const int row = kLnBoxRows * k + vrow;
                    const float gk = gb[row], bk = gb[Vt + row];
                    const float v[4] = {fmaf(fmaf(z[k].x, rs[0], mur[0]), gk, bk), fmaf(fmaf(z[k].y, rs[1], mur[1]), gk, bk),
                                        fmaf(fmaf(z[k].z, rs[2], mur[2]), gk, bk), fmaf(fmaf(z[k].w, rs[3], mur[3]), gk, bk)};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const bool take = v[j] > bv[j] || (v[j] != v[j] && bv[j] == bv[j]);
                        bv[j] = take ? v[j] : bv[j];
                        bi[j] = take ? row : bi[j];
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) { am[j].v = bv[j]; am[j].i = bi[j]; }
        }
        const ArgMax ar = reduce_frames16(am[0], am[1], am[2], am[3], lane, merge_argmax, fih);
        if (lane < 8) { const float v2[2] = {ar.v, __int_as_float(ar.i)}; red_store<2>(red, 4 * h + fih, w, v2); }
        bar_compute();
        if (w < kLnTT) {
            ArgMax b;
            const float *src = red + (w * 16 + (lane & 15)) * 4;
            b.v = src[0]; b.i = __float_as_int(src[1]);
            if ((lane & 15) >= kLnWarps) { b.v = -INFINITY; b.i = kLnNoRow; }
#pragma unroll
            for (int o = 1; o < 16; o <<= 1) b = merge_argmax(b, ArgMax::shfl_xor(b, o));
            const int t = m.t0 + w;
            if (lane == 0 && t < d.T) out[(size_t)m.b * d.T + t] = b.i;
        }
        bar_compute();            // protects red against the next tile
    }
}

static int ln_kmax(int K) { return K <= 5 ? 5 : (K <= 9 ? 9 : (K <= 15 ? 15 : 17)); }

// The backward kernel's shared-memory plan -- the one place that decides whether a shape's backward pass can run:
// launch_ln_backward launches with it and ln_supported refuses (at the forward call, before any work is enqueued) every
// shape whose ring would hold fewer than K + 2 boxes.  Everything but the ring is fixed by (V, Lmax, kind): two alpha/beta
// rows per frame of a tile, the merged posteriors, the node posteriors with their blank partials, the symbol tables, the
// gamma/beta table, the id bitmap and one box of zeros; the ring gets what is left.  The joint objective's plain-CTC
// lattice takes nothing here (phase (a) of ln_gradient_kernel reads it into registers): its plan is Gram-CTC's.
LnSmem plan_ln_backward(const WsLayout &w) {
    const int K = (w.V + kLnBoxRows - 1) / kLnBoxRows;
    const int Vt = ln_kmax(K) * kLnBoxRows;
    return plan_ln_smem((size_t)2 * kLnTT * w.Np * 8, (size_t)kLnTT * ((w.Umax + 3) & ~3),
                        (size_t)kLnTT * w.Np + (size_t)kLnTT * kLnBlankChunks, (size_t)2 * w.Nmax + 2, (size_t)2 * Vt,
                        (size_t)2 * (Vt / 32 + 1), kLnBoxBytes);
}

// Shared memory of the kernels that only stream tiles through the ring (forward, argmax): the gamma/beta table, the
// reductions' scratch and the ring.  smem_reserve: room to leave to a lattice CTA on the same SM, given up when the ring
// would then hold fewer than K + 2 boxes.
LnSmem plan_ln_stream(int K, size_t smem_reserve) {
    const size_t gbf = (size_t)2 * ln_kmax(K) * kLnBoxRows;
    LnSmem sm = plan_ln_smem(0, 0, 0, 0, gbf, 0, 0, smem_reserve);
    if (sm.R < K + 2) sm = plan_ln_smem(0, 0, 0, 0, gbf, 0, 0, 0);     // no room to share the SM
    if (sm.R > 2 * K + 4) {                       // more than two tiles' worth buys nothing; leave the rest to the L1
        sm.total -= (size_t)(sm.R - (2 * K + 4)) * kLnBoxBytes;
        sm.R = 2 * K + 4;
    }
    return sm;
}

// ---- host side ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void *sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(sym);
    });
    return fn;
}

// z viewed as a 3-D tensor (t fastest, then v, then b); a box is 8 frames x 256 rows of one utterance.  Rows and frames
// outside the tensor read as zeros.
bool make_z_map(CUtensorMap *map, const float *z, int B, int T, int V, int64_t zs_b, int64_t zs_v) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return false;
    // The encoder is a DRIVER entry point and wants the device's primary context current on the calling thread.  The
    // runtime binds it lazily, on a thread's first runtime call that needs it -- and backward runs on an autograd worker
    // thread that may not have made one yet (its buffers come out of the caller's caching allocator): bind it once.
    static thread_local bool bound = false;
    if (!bound) { cudaFree(nullptr); bound = true; }
    const cuuint64_t dims[3] = {(cuuint64_t)T, (cuuint64_t)V, (cuuint64_t)B};
    const cuuint64_t strides[2] = {(cuuint64_t)zs_v * 4, (cuuint64_t)zs_b * 4};
    const cuuint32_t box[3] = {(cuuint32_t)kLnTT, (cuuint32_t)kLnBoxRows, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(z), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// The fields every tile kernel reads (the backward-only ones zero; the argmax passes no workspace)
LnParams ln_params(const ProblemDesc &d, const LnLayout &ll, const void *ws, const float *z, int64_t zs_b, int64_t zs_v,
                   const float *gamma, const float *beta) {
    LnParams p;
    memset(&p, 0, sizeof(p));
    p.d = d; p.w = ll.w; p.ws = const_cast<unsigned char *>(static_cast<const unsigned char *>(ws));
    p.z = z; p.zs_b = zs_b; p.zs_v = zs_v; p.gamma = gamma; p.beta = beta;
    p.off_mu = ll.off_mu; p.off_rstd = ll.off_rstd; p.off_lse = ll.off_lse; p.off_part = ll.off_part;
    p.Tq = (d.T + 3) & ~3;
    p.K = (d.V + kLnBoxRows - 1) / kLnBoxRows;
    p.nTB = (d.T + kLnTT - 1) / kLnTT;
    return p;
}

template <typename Kern, typename... Args>
cudaError_t launch_ln(Kern kern, int grid, const LnSmem &sm, cudaStream_t stream, const Args &...args) {
    (void)cudaGetLastError();
    cudaError_t e = ensure_dynamic_smem(reinterpret_cast<const void *>(kern), sm.total);
    if (e != cudaSuccess) { note_failure_site("shared-memory opt-in"); return e; }
    kern<<<grid, kLnThreads, sm.total, stream>>>(args...);
    e = cudaGetLastError();
    if (e != cudaSuccess) note_failure_site("tile kernel launch");
    return e;
}

}  // namespace

LnLayout make_ln_layout(int kind, int B, int T, int V, int Lmax) {
    LnLayout l;
    l.w = make_layout(kind, B, T, V, Lmax);
    size_t o = l.w.total;
    const size_t BT = (size_t)B * (size_t)((T + 3) & ~3);          // rows of these arrays are 16-byte aligned (bulk-copied)
    l.off_mu = o;   o = align_up(o + sizeof(float) * BT, 256);
    l.off_rstd = o; o = align_up(o + sizeof(float) * BT, 256);
    l.off_lse = o;  o = align_up(o + sizeof(float) * BT, 256);
    const int K = (V + kLnBoxRows - 1) / kLnBoxRows;
    l.off_part = o; o = align_up(o + sizeof(float) * 2 * (size_t)K * kLnBoxRows * kLnMaxParts, 256);
    l.total = o;
    return l;
}

int ln_supported(int kind, int B, int T, int V, int Lmax, int64_t zs_v, int64_t zs_b, const void *z) {
    if (kind < 0 || kind > 2) return 0;
    if (V > 17 * kLnBoxRows) return 0;
    if (1 + (kind == 0 ? Lmax : 2 * Lmax) > kLnMaxCols) return 0;
    const int K = (V + kLnBoxRows - 1) / kLnBoxRows;
    if (plan_ln_backward(make_layout(kind, B, T, V, Lmax)).R < K + 2) return 0;
    if ((zs_v & 3) != 0 || (zs_b & 3) != 0 || (reinterpret_cast<uintptr_t>(z) & 15) != 0) return 0;
    return encode_tiled_fn() != nullptr;
}



cudaError_t launch_ln_forward(const ProblemDesc &d, const LnLayout &ll, void *ws, const float *z, int64_t zs_b, int64_t zs_v,
                              const float *gamma, const float *beta, size_t smem_reserve, cudaStream_t stream) {
    if ((long long)d.B * d.T == 0) return cudaSuccess;
    LnParams p = ln_params(d, ll, ws, z, zs_b, zs_v, gamma, beta);
    const LnSmem sm = plan_ln_stream(p.K, smem_reserve);
    if (sm.R < p.K + 2) return cudaErrorInvalidConfiguration;
    p.R = sm.R;
    CUtensorMap map;
    if (!make_z_map(&map, z, d.B, d.T, d.V, zs_b, zs_v)) return cudaErrorInvalidValue;
    long long tiles = (long long)d.B * p.nTB;
    int grid = (int)(tiles < sm_count() ? tiles : sm_count());
    if (grid < 1) grid = 1;
    switch (ln_kmax(p.K)) {
        case 5: return launch_ln(ln_softmax_gather_kernel<5>, grid, sm, stream, map, p, sm);
        case 9: return launch_ln(ln_softmax_gather_kernel<9>, grid, sm, stream, map, p, sm);
        case 15: return launch_ln(ln_softmax_gather_kernel<15>, grid, sm, stream, map, p, sm);
        default: return launch_ln(ln_softmax_gather_kernel<17>, grid, sm, stream, map, p, sm);
    }
}

cudaError_t launch_ln_backward(const GradParams &g, const LnLayout &ll, const void *ws, const float *z, int64_t zs_b, int64_t zs_v,
                               const float *gamma, const float *beta, float *dz, int64_t dzs_b, int64_t dzs_v, float *dgamma,
                               float *dbeta, cudaStream_t stream) {
    const ProblemDesc &d = g.d;
    if ((long long)d.B * d.T == 0) return cudaSuccess;
    LnParams p = ln_params(d, ll, ws, z, zs_b, zs_v, gamma, beta);
    p.grad_loss = g.grad_loss; p.per_utterance = g.per_utterance; p.scale = g.scale;
    p.dz = dz; p.dzs_b = dzs_b; p.dzs_v = dzs_v; p.dgamma = dgamma; p.dbeta = dbeta;
    const int Vp = p.K * kLnBoxRows;
    const LnSmem sm = plan_ln_backward(ll.w);
    if (sm.R < p.K + 2) { note_failure_site("shared-memory plan"); return cudaErrorInvalidConfiguration; }
    p.R = sm.R;
    CUtensorMap map, map_dz;
    if (!make_z_map(&map, z, d.B, d.T, d.V, zs_b, zs_v)) { note_failure_site("tensor map of z"); return cudaErrorInvalidValue; }
    if (!make_z_map(&map_dz, dz, d.B, d.T, d.V, dzs_b, dzs_v)) { note_failure_site("tensor map of dz"); return cudaErrorInvalidValue; }
    long long tiles = (long long)d.B * p.nTB;
    int grid = (int)(tiles < sm_count() ? tiles : sm_count());
    if (grid > kLnMaxParts) grid = kLnMaxParts;
    if (grid < 1) grid = 1;
    cudaError_t e;
    switch (ln_kmax(p.K)) {
        case 5: e = launch_ln(ln_gradient_kernel<5>, grid, sm, stream, map, map_dz, p, sm); break;
        case 9: e = launch_ln(ln_gradient_kernel<9>, grid, sm, stream, map, map_dz, p, sm); break;
        case 15: e = launch_ln(ln_gradient_kernel<15>, grid, sm, stream, map, map_dz, p, sm); break;
        default: e = launch_ln(ln_gradient_kernel<17>, grid, sm, stream, map, map_dz, p, sm); break;
    }
    if (e != cudaSuccess) return e;
    if (dgamma || dbeta) {
        const float *part = reinterpret_cast<const float *>(p.ws + p.off_part);
        ln_reduce_params_kernel<<<(d.V + 127) / 128, 128, 0, stream>>>(part, grid, Vp, d.V, dgamma, dbeta);
        e = cudaGetLastError();
        if (e != cudaSuccess) note_failure_site("dgamma/dbeta reduction launch");
    }
    return e;
}

cudaError_t launch_ln_argmax(const float *z, int64_t zs_b, int64_t zs_v, const float *gamma, const float *beta, int B, int T, int V,
                             int64_t *argmax_out, cudaStream_t stream) {
    if ((long long)B * T == 0) return cudaSuccess;
    ProblemDesc d;
    memset(&d, 0, sizeof(d));
    d.B = B; d.T = T; d.V = V;
    LnParams p = ln_params(d, LnLayout(), nullptr, z, zs_b, zs_v, gamma, beta);
    const LnSmem sm = plan_ln_stream(p.K, 0);
    if (sm.R < p.K + 2) { note_failure_site("shared-memory plan"); return cudaErrorInvalidConfiguration; }
    p.R = sm.R;
    CUtensorMap map;
    if (!make_z_map(&map, z, B, T, V, zs_b, zs_v)) { note_failure_site("tensor map of z"); return cudaErrorNotSupported; }
    const long long tiles = (long long)B * p.nTB;
    const int grid = (int)(tiles < sm_count() ? tiles : sm_count());
    switch (ln_kmax(p.K)) {
        case 5: return launch_ln(ln_argmax_kernel<5>, grid, sm, stream, map, p, sm, argmax_out);
        case 9: return launch_ln(ln_argmax_kernel<9>, grid, sm, stream, map, p, sm, argmax_out);
        case 15: return launch_ln(ln_argmax_kernel<15>, grid, sm, stream, map, p, sm, argmax_out);
        default: return launch_ln(ln_argmax_kernel<17>, grid, sm, stream, map, p, sm, argmax_out);
    }
}

}  // namespace b200ctc
