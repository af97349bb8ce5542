// common.cuh -- shared device helpers and the workspace layout of the B200 CTC / Gram-CTC library.
//
// Number format used by the lattice recursion ("scaled linear"): a probability is carried as a pair
// (m, e) of float32 meaning m * 2^e, with e integer-valued (exact up to 2^24) and m a plain mantissa
// that is pulled back into [1,2) every few frames.  One exponent PER NODE, so neither the range between
// nodes of one frame nor the decay along the utterance (T=800 frames x ~12 bits) can under/overflow, and
// the recursion needs no exp/log at all: aligning two values is a multiplication by an exact power of two.
// Probability zero is (0, SENT); any exponent below SENT_TEST means zero (the reference's log-space code
// uses -1e10 for log 0, gram_ctc.py:222).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace b200ctc {

constexpr float SENT = -1.0e30f;              // exponent of probability zero ("log 0")
constexpr float SENT_TEST = -1.0e29f;         // anything below this is treated as log 0
constexpr float LOG2E_HI = 1.44269502162933349609375f;      // float(log2 e)
constexpr float LOG2E_LO = 1.92596299112661746e-8f;         // log2 e - LOG2E_HI
// Per-frame softmax normaliser of the gradient kernels, (la, s): softmax(x) = 2^(x*LOG2E_HI - la) * s.  la + lb is the
// log2 normaliser as the lattice gets it, an unevaluated float pair; rounding la + lb to one float costs up to half an
// ulp of la in log2 p (6e-5 relative at |logits| ~ 1000), so lb goes into the per-frame scale s instead.  s also leaves
// out m*LOG2E_LO (m = the row maximum), as the row loop leaves out x*LOG2E_LO: what remains is (x - m)*LOG2E_LO,
// below 1e-6 wherever the softmax is not negligible.
__device__ __forceinline__ float2 grad_normaliser(float m, float la, float lb) {
    return make_float2(la, exp2f(fmaf(m, LOG2E_LO, -lb)));
}
constexpr double LN2_D = 0.693147180559945309417232121458;
constexpr int kProgBlock = 16;                // frames per progress counter = frames per lattice pipeline chunk
constexpr float RINT_MAGIC = 12582912.0f;     // 1.5 * 2^23: (x + M) - M == rint(x) for |x| < 2^22

// Per-utterance record written by the prep kernel and completed by the lattice kernel.
struct UttInfo {
    int Tb;        // clamped input length
    int Lb;        // clamped label length
    int Nb;        // lattice nodes: 2*Lb+1 (CTC) or 3*Lb+1 (Gram-CTC)
    int Ub;        // number of distinct symbols the lattice can emit (blank included), sorted by id
    float Ph;      // P = 2^Ph / Pl: integer exponent (+1e30 when the alignment is infeasible) ...
    float Pl;      // ... and the INVERSE of the mantissa in [1,2)  (0 when infeasible)
    float loss;    // -ln P, or 1e10 when infeasible (reference quirk, SURVEY.md 8a)
    int flags;     // bit0: lengths were out of range and got clamped
    int ublank;    // position of the blank id in the sorted distinct-symbol list
    int infeasible;  // written by the lattice CTA: 1 when no alignment exists
};

// Header at the start of the workspace: work-queue tickets for the row-streaming kernels.
struct WsHeader {
    unsigned int k1_ticket;    // next frame for the softmax/gather kernel
    unsigned int k3_ticket;    // next frame for the gradient kernel
    unsigned int k3_done;      // gradient warps that ran out of work (last one re-arms the queue)
    unsigned int k2_done;      // lattice CTAs that have published their loss (last one reduces the batch)
    unsigned int k2b_done;     // same for the second (plain CTC) lattice of a joint Gram-CTC + CTC call
    unsigned int stalled;      // a lattice CTA gave up waiting for emission rows of the softmax/gather kernel running next to
                               // it (seconds: the two kernels are not co-resident -- never seen, but it must not hang the GPU);
                               // the losses of the call are NaN then
};

// Workspace carve-up (all offsets in bytes from a 16-byte aligned base).
struct WsLayout {
    int kind, B, T, V, Lmax;
    int W;         // emission row width: [blank, label_0..label_{Lmax-1} (, bigram_0..)] padded to even.  An utterance with
                   // Lb labels fills EmissionColumns::count(Lb) of them (the bigram columns past Lb are not written): column c
                   // is the (m, e) pair emission_pair() gives for the id EmissionColumns::symbol(c, Lb), or (0, SENT) for a
                   // padded label column (id -1) and an id outside [0, V)
    int Nmax;      // lattice nodes for Lmax
    int Np;        // Nmax (+ boff) padded to a multiple of 4
    int boff;      // beta_t[j] is stored at bv[t][j + boff]: 1 for CTC (aligns the reversed direction's node pairs), else 0
    int Umax;      // upper bound on distinct symbols per utterance (blank + every non-blank-type node)
    int nwords;    // ceil(V / 32): words of the per-utterance "is a lattice symbol" bitmap
    int nblk;      // ceil(T / kProgBlock): progress counters per utterance
    size_t off_prog;   // [B][nblk] unsigned: emission rows of frames [16k, 16k+16) written so far (softmax/gather
                       // kernel -> lattice kernel, which may run concurrently with it)
    // joint Gram-CTC + CTC (run/gram_ctc/cnn/train.py:196-198, both losses on the same activations): the Gram-CTC
    // layout above plus the alpha/beta rows and utterance records of the plain-CTC lattice, which reads the same
    // emission rows (its symbols are the blank and unigram columns of the Gram-CTC row)
    int joint;         // 0 / 1
    int Nmax2, Np2;    // CTC lattice nodes for Lmax, padded like Np (its beta rows are stored one element up)
    size_t off_av2, off_bv2, off_utt2;
    size_t off_hdr, off_utt, off_lse, off_lp, off_av, off_bv, off_usym, off_uoff, off_unode, off_urec, off_bm, off_pc, total;
};

// The problem as the kernels see it (built by api.cu from the entry point's arguments)
struct ProblemDesc {
    int kind, B, T, V, Lmax, blank;   // kind: 0 = CTC, 1 = Gram-CTC (a joint call is 1 here plus a second, CTC lattice)
    const float *acts;
    int64_t stride_t, stride_b;
    const int32_t *labels, *bigrams, *input_lengths, *label_lengths;
    int concurrent; // the lattice kernel runs next to the softmax/gather kernel: the latter signals every finished
                    // frame (progress counters), the former waits on them, and tickets walk the frames from both ends
};

__host__ __device__ inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// An utterance's input or label length as every kernel reads it: clamped into [0, hi] (T or Lmax)
__host__ __device__ inline int clamp_length(int v, int hi) { return max(0, min(v, hi)); }

// kind: 0 = CTC, 1 = Gram-CTC, 2 = joint Gram-CTC + CTC (laid out as Gram-CTC plus a second lattice)
__host__ inline WsLayout make_layout(int kind, int B, int T, int V, int Lmax) {
    WsLayout w;
    const int joint = kind == 2 ? 1 : 0;
    if (joint) kind = 1;
    w.kind = kind; w.B = B; w.T = T; w.V = V; w.Lmax = Lmax;
    w.joint = joint;
    w.Nmax2 = 2 * Lmax + 1;
    w.Np2 = (w.Nmax2 + 1 + 3) & ~3;
    int width = 1 + (kind == 0 ? Lmax : 2 * Lmax);
    w.W = (width + 1) & ~1;
    w.Nmax = (kind == 0 ? 2 : 3) * Lmax + 1;
    w.boff = kind == 0 ? 1 : 0;
    w.Np = (w.Nmax + w.boff + 3) & ~3;
    w.Umax = w.Nmax - Lmax;                 // blank + (per-1)*Lmax entries
    w.nwords = (V + 31) / 32;
    w.nblk = (T + kProgBlock - 1) / kProgBlock;
    size_t o = 0;
    const size_t BT = (size_t)B * (size_t)T;
    w.off_hdr = o;   o = align_up(o + sizeof(WsHeader), 256);
    w.off_utt = o;   o = align_up(o + sizeof(UttInfo) * (size_t)B, 256);
    w.off_lse = o;   o = align_up(o + sizeof(float2) * BT, 256);     // grad_normaliser() per frame
    w.off_lp = o;    o = align_up(o + sizeof(float2) * BT * w.W, 256);
    w.off_av = o;    o = align_up(o + sizeof(float2) * BT * w.Np, 256);      // alpha_t[j] as (m, e)
    w.off_bv = o;    o = align_up(o + sizeof(float2) * BT * w.Np, 256);      // beta_t[j] (excludes emission at t), at [j + boff]
    w.off_usym = o;  o = align_up(o + sizeof(int) * (size_t)B * w.Nmax, 256);
    w.off_uoff = o;  o = align_up(o + sizeof(int) * (size_t)B * (w.Nmax + 1), 256);
    w.off_unode = o; o = align_up(o + sizeof(int) * (size_t)B * w.Nmax, 256);
    w.off_urec = o;  o = align_up(o + 16 * (size_t)B * w.Nmax, 256);         // int4 per distinct id, see prep.cuh
    w.off_bm = o;    o = align_up(o + sizeof(unsigned) * (size_t)B * w.nwords, 256);
    w.off_pc = o;    o = align_up(o + sizeof(int) * (size_t)B * w.nwords, 256);
    w.off_prog = o;  o = align_up(o + sizeof(unsigned) * (size_t)B * w.nblk, 256);
    w.off_av2 = w.off_bv2 = w.off_utt2 = 0;
    if (joint) {
        w.off_utt2 = o;  o = align_up(o + sizeof(UttInfo) * (size_t)B, 256);
        w.off_av2 = o;   o = align_up(o + sizeof(float2) * BT * w.Np2, 256);
        w.off_bv2 = o;   o = align_up(o + sizeof(float2) * BT * w.Np2, 256);
    }
    w.total = o;
    return w;
}

// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float lg2_approx(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// rint for |x| < 2^22 on the FMA pipe (FRND would go through the slow conversion unit)
__device__ __forceinline__ float rint_small(float x) {
    return __fsub_rn(__fadd_rn(x, RINT_MAGIC), RINT_MAGIC);
}

// 2^d for an integer-valued d <= 0, exact, on the FMA/ALU pipes; anything below -126 (SENT included) gives 0
__device__ __forceinline__ float pow2_nonpos(float d) {
    const float c = fmaxf(d, -127.f);
    return __uint_as_float((__float_as_uint(c + RINT_MAGIC) << 23) + 0x3f800000u);
}
// (m, e) -> the same value with m in [1,2); zero, NaN and Inf are left alone
__device__ __forceinline__ void renorm_pair(float &m, float &e) {
    const uint32_t b = __float_as_uint(m);
    const uint32_t x = (b >> 23) & 0xffu;
    if (x != 0u && x != 255u) {
        e += (float)((int)x - 127);
        m = __uint_as_float((b & 0x807fffffu) | 0x3f800000u);
    }
}
// alpha * beta / P for one lattice node (gram_ctc.py:290 "exp(label_prob - total)" before the per-symbol merge):
// a, b = (m, e) pairs, Ph / Pinv as in UttInfo.  ex2.approx is exact on integers (checked -140..115 on sm_100a,
// tools/ubench_step_linear.cu) and flushes to 0 below -126.
__device__ __forceinline__ float node_posterior(float2 a, float2 b, float Ph, float Pinv) {
    return (a.x * b.x) * ex2_approx((a.y + b.y) - Ph) * Pinv;
}

// ---- an utterance's lengths and its emission row (format: WsLayout::W) ----
// A missing length array means the full width (T or Lmax).
__device__ __forceinline__ int utt_input_length(const ProblemDesc &d, int b) {
    return clamp_length(d.input_lengths ? __ldg(d.input_lengths + b) : d.T, d.T);
}
__device__ __forceinline__ int utt_label_length(const ProblemDesc &d, int b) {
    return clamp_length(d.label_lengths ? __ldg(d.label_lengths + b) : d.Lmax, d.Lmax);
}
// The columns of utterance b's emission row: how many an utterance with Lb (clamped) labels fills, and the vocabulary id
// of column c (gram_ctc.py:24-32, :155), -1 for a padded label column
struct EmissionColumns {
    const int32_t *lab, *big;
    int Lmax, blank, gram;
    __device__ __forceinline__ EmissionColumns(const ProblemDesc &d, int b)
        : lab(d.labels + (size_t)b * d.Lmax), big(d.kind == 1 ? d.bigrams + (size_t)b * d.Lmax : nullptr), Lmax(d.Lmax),
          blank(d.blank), gram(d.kind == 1) {}
    __device__ __forceinline__ int count(int Lb) const { return 1 + (gram ? Lmax + Lb : Lb); }
    __device__ __forceinline__ int symbol(int c, int Lb) const {
        if (c == 0) return blank;
        if (c <= Lmax) return (c - 1 < Lb) ? __ldg(lab + c - 1) : -1;
        return __ldg(big + c - 1 - Lmax);
    }
};

// log2 normaliser of a row, max*log2(e) + log2(sum), as an unevaluated float pair
__device__ __forceinline__ void split_lse2(float m, float s, float &la, float &lb) {
    const float mh = m * LOG2E_HI;
    float ml = fmaf(m, LOG2E_HI, -mh);
    ml = fmaf(m, LOG2E_LO, ml);
    const float lg = log2f(s);
    const float a = mh + lg;                                  // TwoSum(mh, lg)
    const float bb = a - mh;
    const float err = (mh - (a - bb)) + (lg - bb);
    la = a;
    lb = err + ml;
}
// Emission probability p = 2^(x*log2(e) - lse2) in the lattice's (mantissa, integer exponent) format.  log2 p is first
// formed as integer hi + small lo, exact to ~1e-7 between symbols (lse2 comes as an unevaluated sum la + lb so that its
// own rounding does not enter); the mantissa is then 2^lo in [0.70, 1.42].
__device__ __forceinline__ float2 emission_pair(float x, float la, float lb) {
    const float ph = x * LOG2E_HI;
    float pl = fmaf(x, LOG2E_HI, -ph);
    pl = fmaf(x, LOG2E_LO, pl);
    const float dd = ph - la;                                 // TwoSum(ph, -la)
    const float bb = dd - ph;
    const float err = (ph - (dd - bb)) + (-la - bb);
    const float lo_full = (err + pl) - lb;
    const float hi = rintf(dd);
    const float lo = (dd - hi) + lo_full;
    if (dd < SENT_TEST) return make_float2(0.f, SENT);        // -inf activation: probability 0 (a NaN still propagates)
    return make_float2(exp2f(lo), hi);
}

// ---- frame progress between the softmax/gather kernel and a concurrently running lattice kernel ----
// Producer: called by ONE lane after a __syncwarp() that follows the warp's stores of the frame's emission row.
__device__ __forceinline__ void signal_frame_done(unsigned char *ws, const WsLayout &w, int b, int t) {
    unsigned *p = reinterpret_cast<unsigned *>(ws + w.off_prog) + (size_t)b * w.nblk + t / kProgBlock;
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(p) : "memory");
}
// Consumer (whole warp): how many of the blocks blk0, blk0 + step, blk0 + 2*step, ... (up to 32, inside [0, nblk))
// are complete, counted from the front.  Block k of an utterance with Tb frames is complete when its counter has
// reached min(kProgBlock, Tb - k*kProgBlock).  One L2 round trip for up to 32 blocks.
__device__ __forceinline__ int count_blocks_done(const unsigned char *ws, const WsLayout &w, int b, int Tb, int blk0,
                                                 int step, int lane) {
    const int nb = (Tb + kProgBlock - 1) / kProgBlock;
    const int blk = blk0 + step * lane;
    bool ok = false;
    if (blk >= 0 && blk < nb) {
        const unsigned *p = reinterpret_cast<const unsigned *>(ws + w.off_prog) + (size_t)b * w.nblk + blk;
        unsigned v;
        asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
        ok = v >= (unsigned)min(kProgBlock, Tb - blk * kProgBlock);
    }
    const unsigned m = __ballot_sync(0xffffffffu, ok);
    const int n = __ffs(~m) - 1;                      // leading run of complete blocks (32 if all)
    if (n > 0) asm volatile("fence.acq_rel.gpu;" ::: "memory");      // acquire: the rows behind the counters are visible from here on
    return n < 0 ? 32 : n;
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier + 1-D bulk async copy (TMA engine, SASS UBLKCP) ----
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// A few immediate retries (the usual case: the partner is a handful of cycles away), then polite polling, so that
// a warp that waits for long does not take issue slots from the warps it shares the SM with.
// non-blocking probe (try_wait may suspend the thread for a while when the phase is not complete yet)
__device__ __forceinline__ bool mbar_test_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    for (int i = 0; i < 8; ++i)
        if (mbar_try_wait(bar, parity)) return;
    while (!mbar_try_wait(bar, parity)) __nanosleep(64);
}
// same, but backs off between polls: for waits that are expected to block for a while, so that the
// polling does not compete with the warps it is waiting for
__device__ __forceinline__ void mbar_wait_backoff(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) __nanosleep(200);
}
// global -> shared bulk copy; bytes % 16 == 0, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// The same with an L2 eviction-priority hint.  The activation rows and the gradient rows are touched once per kernel and
// are many times the L2 (1.2 GB against 126 MB): marked evict-first they stop pushing out what IS reused across
// kernels -- the emission rows the lattice reads and the alpha/beta rows the gradient kernel reads (130 MB).
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void bulk_g2s_hint(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar, uint64_t policy) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
                 : "memory");
}
// shared -> global bulk copy (bulk-group completion)
__device__ __forceinline__ void bulk_s2g(void *dst_gmem, const void *src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem),
                 "r"(smem_u32(src_smem)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait_all() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// order generic-proxy accesses against async-proxy (bulk copy) accesses
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }
// the same, restricted to one state space: shared memory written by this thread and then read by a bulk store, or
// global memory written with ordinary stores and then read by a bulk load
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

__device__ __forceinline__ float4 ldg_stream4(const float4 *p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}
__device__ __forceinline__ void stg_stream4(float4 *p, const float4 &v) {
    asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}

#endif  // __CUDACC__

}  // namespace b200ctc
