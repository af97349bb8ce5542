// viterbi.cu -- forced alignment: the best path through the CTC / Gram-CTC lattice, i.e. the loss's recursion under the
// (max, x) semiring instead of (+, x), on the emission rows kernel 1 wrote; then its backtrace and the per-frame and
// per-label outputs (include/b200ctc.h, b200ctc_align).
//
// One CTA per utterance.  Scores are (m, e) pairs (common.cuh) with m kept in [1,2) every frame and probability zero as
// (0, SENT), so comparing two probabilities is a lexicographic (e, m) compare: exact, no exp/log, no scaling.  A frame
// is: pick the best predecessor (ties: smallest back-offset k), one FMUL with the emission mantissa, add the exponents,
// renormalise with integer exponent-bit operations.  The previous frame's scores sit in a shared-memory double buffer
// (one __syncthreads() per frame); every node's choice of k is stored as one byte per (frame, node) in the workspace's
// alpha region, row per frame.
#include <algorithm>

#include "common.cuh"
#include "kernels.h"

namespace b200ctc {

namespace {

constexpr int kFrontPad = 8;           // zero scores in front of node 0: j - k needs no bounds check (k <= 7)
constexpr int kBlk = 32;               // backtrace frames per staged window
constexpr int kWinW = 256;             // bytes per window row: the path moves at most 7 (Gram-CTC) nodes per frame, so a
                                       // row spans <= 7 * 31 + 1 nodes, read as 16-byte words from a 16-byte boundary
constexpr int kMaxThreads = 1024;

// backpointer rows ([b][t][P] bytes in the alpha region, which holds B*T*Np*8 >= B*T*P of them): 16-byte aligned
__host__ __device__ inline int bp_pitch(int Nmax) { return (Nmax + 15) & ~15; }

__device__ __forceinline__ bool better(float2 a, float2 b) {     // a > b as probabilities, both normalised
    return a.y > b.y || (a.y == b.y && a.x > b.x);
}

// Node j of utterance b: emission column of the row kernel 1 wrote (0 blank, 1 + i label i, 1 + Lmax + i bigram i),
// vocabulary id, and the mask of back-offsets k whose node j - k is a predecessor (bit 0, the self-loop, always).  The
// "ids differ" edges are those of the loss (lattice.cu, init_lane); j - k < 0 reads the zero front padding.
template <bool GRAM>
struct NodeGeo {
    int col, sym;
    unsigned mask;
};
template <bool GRAM>
__device__ __forceinline__ NodeGeo<GRAM> node_geo(const ProblemDesc &d, const int32_t *lab, const int32_t *big, int j) {
    NodeGeo<GRAM> g;
    if constexpr (!GRAM) {
        if (j & 1) {
            const int i = j >> 1;
            g.col = 1 + i;
            g.sym = lab[i];
            g.mask = 0x3u | ((i >= 1 && lab[i] != lab[i - 1]) ? 0x4u : 0u);
        } else {
            g.col = 0; g.sym = d.blank; g.mask = 0x3u;
        }
    } else {
        const int i = j / 3, type = j - 3 * i;
        if (type == 0) {
            g.col = 0; g.sym = d.blank; g.mask = 0x7u;
        } else if (type == 1) {
            g.col = 1 + i;
            g.sym = lab[i];
            g.mask = 0x7u | ((i >= 1 && lab[i] != lab[i - 1]) ? 0x8u : 0u);
        } else {
            g.col = 1 + d.Lmax + i;
            g.sym = big[i];
            g.mask = 0xa1u | ((i >= 2 && big[i] != big[i - 2]) ? 0x40u : 0u);
        }
    }
    return g;
}

// Label positions a node covers: [lo, hi] (CTC label i, Gram-CTC unigram i: i; bigram i: i - 1 and i); lo > hi for blank.
template <bool GRAM>
__device__ __forceinline__ void node_positions(int j, int &lo, int &hi) {
    if constexpr (!GRAM) {
        hi = j >> 1;
        lo = (j & 1) ? hi : hi + 1;
    } else {
        const int i = j / 3, type = j - 3 * i;
        hi = i;
        lo = type == 0 ? i + 1 : (type == 1 ? i : i - 1);
    }
}

// an emission pair as kernel 1 wrote it, normalised (m in [1,2), or (0, SENT))
__device__ __forceinline__ float2 normalised(float2 v) {
    renorm_pair(v.x, v.y);
    if (v.x == 0.f) v.y = SENT;
    return v;
}

// Emission rows of CH frames (CH * W pairs, contiguous in the workspace) -> one of the two shared-memory stages, by one
// bulk async copy (TMA); rows are 16-byte aligned because W is even.
__device__ __forceinline__ void stage_rows(float2 *dst, const float2 *lp, int W, int t0, int n, uint64_t *bar) {
    const uint32_t bytes = (uint32_t)n * (uint32_t)W * (uint32_t)sizeof(float2);
    fence_proxy_async_smem();                      // the stage's earlier generic reads before the async write
    mbar_arrive_expect_tx(bar, bytes);
    bulk_g2s(dst, lp + (size_t)t0 * W, bytes, bar);
}

template <bool GRAM, int NPT>
__global__ void __launch_bounds__(kMaxThreads) viterbi_kernel(AlignParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_node;
    __shared__ __align__(8) uint64_t full[2];
    const ProblemDesc &d = p.d;
    const int b = blockIdx.x;
    const int tid = threadIdx.x;
    // Lengths clamped as v < 0 ? 0 : min(v, hi), not with utt_input_length() / utt_label_length() (max(0, min(v, hi)), the
    // same value since T, Lmax >= 0): from those ptxas builds the CTC instantiations differently, and a CTC alignment took
    // 4 % longer (B = 64, T = 800, V = 3500 on a B200).
    const int Tin = d.input_lengths ? d.input_lengths[b] : d.T, Lin = d.label_lengths ? d.label_lengths[b] : d.Lmax;
    const int Tb = Tin < 0 ? 0 : min(Tin, d.T);
    const int Lb = Lin < 0 ? 0 : min(Lin, d.Lmax);
    const int Nb = (GRAM ? 3 : 2) * Lb + 1;
    const int Nmax = p.w.Nmax;
    const int stride = p.buf_stride;
    const int CH = p.chunk;
    const int W = p.w.W;
    float2 *buf = reinterpret_cast<float2 *>(smem_raw);                          // [2][stride]: scores of frames t, t+1
    float2 *stage = buf + 2 * stride;                                            // [2][CH][W]: emission rows
    unsigned char *win = reinterpret_cast<unsigned char *>(stage + 2 * (size_t)CH * W);   // [kBlk][kWinW] backtrace window
    const int32_t *lab = d.labels + (size_t)b * d.Lmax;
    const int32_t *big = GRAM ? d.bigrams + (size_t)b * d.Lmax : nullptr;
    const float2 *lp = reinterpret_cast<const float2 *>(p.ws + p.w.off_lp) + (size_t)b * d.T * p.w.W;
    const int P = bp_pitch(Nmax);
    unsigned char *bp = p.ws + p.w.off_av + (size_t)b * d.T * P;

    // virtual state before frame 0: all mass on node 0 (the loss's start nodes follow from the edges)
    for (int i = tid; i < 2 * stride; i += blockDim.x)
        buf[i] = i == kFrontPad ? make_float2(1.f, 0.f) : make_float2(0.f, SENT);

    if (tid == 0) {
        mbar_init(&full[0], 1u);
        mbar_init(&full[1], 1u);
        mbar_init_fence();
        for (int c = 0; c < 2 && c * CH < Tb; ++c) stage_rows(stage + (size_t)c * CH * W, lp, W, c * CH, min(CH, Tb - c * CH), &full[c]);
    }
    int col[NPT];
    unsigned mask[NPT];
    bool act[NPT];
#pragma unroll
    for (int r = 0; r < NPT; ++r) {
        const int j = NPT * tid + r;
        act[r] = j < Nb;
        col[r] = 0; mask[r] = 1u;
        if (act[r]) {
            const NodeGeo<GRAM> g = node_geo<GRAM>(d, lab, big, j);
            col[r] = g.col; mask[r] = g.mask;
        }
    }
    bool nan = false;
    __syncthreads();

    // ---- frame loop: a T-step dependent chain; the emission rows of the next chunk are in flight meanwhile ----
    for (int c = 0, t0 = 0; t0 < Tb; ++c, t0 += CH) {
        const float2 *ems = stage + (size_t)(c & 1) * CH * W;
        mbar_wait(&full[c & 1], (uint32_t)(c >> 1) & 1u);
        const int n = min(CH, Tb - t0);
        for (int u = 0; u < n; ++u) {
            const int t = t0 + u;
            const float2 *cur = buf + (t & 1) * stride + kFrontPad;
            float2 *nxt = buf + ((t + 1) & 1) * stride + kFrontPad;
            unsigned char *bprow = bp + (size_t)t * P;
#pragma unroll
            for (int r = 0; r < NPT; ++r) {
                if (!act[r]) continue;
                const int j = NPT * tid + r;
                float2 best = cur[j];
                int bk = 0;
#pragma unroll
                for (int k = 1; k <= (GRAM ? 7 : 2); ++k) {
                    if (GRAM && k == 4) continue;                                // no node has the predecessor j - 4
                    if ((mask[r] >> k) & 1u) {
                        const float2 c = cur[j - k];
                        if (better(c, best)) { best = c; bk = k; }
                    }
                }
                const float2 e = normalised(ems[u * W + col[r]]);
                nan |= e.x != e.x;
                float m = best.x * e.x;
                float ex = best.y + e.y;
                renorm_pair(m, ex);
                if (m == 0.f) ex = SENT;
                nxt[j] = make_float2(m, ex);
                bprow[j] = (unsigned char)bk;
            }
            __syncthreads();
        }
        // every thread is past its last read of this stage: refill it with chunk c + 2
        if (tid == 0 && t0 + 2 * CH < Tb)
            stage_rows(const_cast<float2 *>(ems), lp, W, t0 + 2 * CH, min(CH, Tb - t0 - 2 * CH), &full[c & 1]);
    }
    const bool any_nan = __syncthreads_or(nan) != 0;

    // ---- best end node (ties: the final blank, then N-2, then N-3) and the score ----
    if (tid == 0) {
        int jend = -1;
        float score;
        if (Tb == 0) {                                           // no frames: P = 1 iff there is nothing to emit
            score = Lb == 0 ? 0.f : 1e10f;
        } else {
            const float2 *fin = buf + (Tb & 1) * stride + kFrontPad;
            float2 best = make_float2(0.f, SENT);
            for (int i = 0; i < (GRAM ? 3 : 2); ++i) {
                const int j = Nb - 1 - i;
                if (j >= 0 && better(fin[j], best)) { best = fin[j]; jend = j; }
            }
            if (any_nan) {
                score = __int_as_float(0x7fc00000);
                jend = -1;
            } else if (jend < 0) {
                score = 1e10f;                                   // no alignment: what the loss returns
            } else {
                score = (float)(-(log((double)best.x) + (double)best.y * LN2_D));
            }
        }
        p.score[b] = score;
        s_node = jend;
    }
    __syncthreads();

    // ---- backtrace in windows of kBlk frames: the backpointers the path can reach are staged with one round of
    // 16-byte loads (independent, so their L2 latencies overlap), then one thread walks them in shared memory ----
    int node = s_node;
    const bool ok = node >= 0;
    int32_t *path = p.path + (size_t)b * d.T;
    constexpr int reach = GRAM ? 7 : 2;
    for (int tb = Tb - 1; ok && tb >= 0; tb -= kBlk) {
        const int tlo = max(0, tb - kBlk + 1);
        const int nrows = tb - tlo + 1;
        const int jlo = max(0, node - reach * (nrows - 1)) & ~15;
        const int nvec = (node + 16 - jlo) >> 4;                 // words covering nodes [jlo, node]
        for (int i = tid; i < nrows * nvec; i += blockDim.x) {
            const int r = i / nvec, c = i - r * nvec;
            reinterpret_cast<uint4 *>(win + r * kWinW)[c] =
                __ldcg(reinterpret_cast<const uint4 *>(bp + (size_t)(tlo + r) * P + jlo) + c);
        }
        __syncthreads();
        if (tid == 0) {
            int n = node;
            for (int t = tb; t >= tlo; --t) {
                path[t] = n;
                n -= win[(t - tlo) * kWinW + (n - jlo)];
            }
            s_node = n;
        }
        __syncthreads();
        node = s_node;
    }

    // ---- epilogue: ids, frame log-probabilities, label spans ----
    int64_t *ids = p.ids + (size_t)b * d.T;
    for (int t = tid; t < d.T; t += blockDim.x) {
        int64_t id = d.blank;
        float fl = 0.f;
        if (ok && t < Tb) {
            const int j = path[t];
            const NodeGeo<GRAM> g = node_geo<GRAM>(d, lab, big, j);
            id = g.sym;
            const float2 e = __ldg(lp + (size_t)t * W + g.col);
            fl = (float)(log((double)e.x) + (double)e.y * LN2_D);
        } else {
            path[t] = -1;
        }
        ids[t] = id;
        if (p.frame_logp) p.frame_logp[(size_t)b * d.T + t] = fl;
    }
    if (p.spans) {
        int2 *sp = reinterpret_cast<int2 *>(p.spans) + (size_t)b * d.Lmax;
        for (int i = tid; i < d.Lmax; i += blockDim.x) sp[i] = make_int2(-1, -1);
        __syncthreads();
        // every label position is covered by exactly one run of one node of a valid path
        for (int t = tid; ok && t < Tb; t += blockDim.x) {
            const int j = path[t];
            int lo, hi;
            node_positions<GRAM>(j, lo, hi);
            if (lo > hi) continue;
            const bool first = t == 0 || path[t - 1] != j;
            const bool last = t == Tb - 1 || path[t + 1] != j;
            for (int q = lo; q <= hi; ++q) {
                if (first) sp[q].x = t;
                if (last) sp[q].y = t + 1;
            }
        }
    }
}

template <bool GRAM, int NPT>
cudaError_t launch_one(const AlignParams &p, int threads, size_t smem, cudaStream_t stream) {
    const void *kern = reinterpret_cast<const void *>(viterbi_kernel<GRAM, NPT>);
    cudaError_t e = ensure_dynamic_smem(kern, smem);
    if (e != cudaSuccess) return e;
    viterbi_kernel<GRAM, NPT><<<p.d.B, threads, smem, stream>>>(p);
    return cudaGetLastError();
}

template <bool GRAM>
cudaError_t launch_kind(const AlignParams &p, int npt, int threads, size_t smem, cudaStream_t stream) {
    if (npt == 1) return launch_one<GRAM, 1>(p, threads, smem, stream);
    if (npt == 2) return launch_one<GRAM, 2>(p, threads, smem, stream);
    return launch_one<GRAM, 3>(p, threads, smem, stream);
}

constexpr size_t kStageBytes = 24 * 1024;   // per emission stage: 32 frames of the usual rows (W = 82 CTC, 122 Gram-CTC
                                            // at the bench shapes take 21 / 24 KB), at least one frame of any row

}  // namespace

size_t align_smem_bytes(const WsLayout &w, AlignGeometry *g) {
    AlignGeometry a;
    a.npt = (w.Nmax + kMaxThreads - 1) / kMaxThreads;
    a.threads = ((w.Nmax + a.npt - 1) / a.npt + 31) / 32 * 32;
    a.stride = (kFrontPad + a.npt * a.threads + 1) & ~1;
    const size_t row = sizeof(float2) * (size_t)w.W;
    a.chunk = (int)std::max<size_t>(1, std::min<size_t>(kBlk, kStageBytes / row));
    if (g) *g = a;
    return sizeof(float2) * (2 * (size_t)a.stride + 2 * (size_t)a.chunk * w.W) + (size_t)kBlk * kWinW;
}

cudaError_t launch_align(AlignParams p, cudaStream_t stream) {
    if (p.d.B == 0) return cudaSuccess;
    AlignGeometry g;
    const size_t smem = align_smem_bytes(p.w, &g);
    const int threads = g.threads, npt = g.npt;
    if (npt > 3) return cudaErrorInvalidValue;                  // validate() keeps Nmax <= 3072
    p.buf_stride = g.stride;
    p.chunk = g.chunk;
    return p.d.kind == 0 ? launch_kind<false>(p, npt, threads, smem, stream) : launch_kind<true>(p, npt, threads, smem, stream);
}

}  // namespace b200ctc
