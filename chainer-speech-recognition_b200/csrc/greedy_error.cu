// greedy_error.cu -- evaluation path after the greedy argmax: collapse, gram -> unigram expansion, edit
// distance and character error rate, on the device (SURVEY.md section 8f, rank 1).
//
// Replaces, in the reference:
//   asr/error.py:26-68   compute_minibatch_error: per utterance, drop blanks from the target (:33-37), collapse the
//                        argmax sequence (blank resets, repeats are skipped, :38-47), turn the predicted ids back into
//                        a string and re-tokenise it into unigram ids (:49-53, asr/vocab.py:99-126), accumulate
//                        the error rate (:55) and average over the batch (:68);
//   asr/error.py:7-24    compute_character_error_rate: Levenshtein distance / len(reference), len(hypothesis) when
//                        the reference is empty (:8-9).
// There it is a Python double loop per utterance on the host, every development batch
// (run/ctc/cnn/train.py:224-234).  Here: one CTA per utterance.
//   * collapse + expansion: keep[t] = tok[t] != blank && tok[t] != tok[t-1] (equivalent to the reference's
//     prev_token state machine: prev_token always equals the previous frame's token); the string round trip is a
//     table lookup id -> up to E unigram ids (the host builds the table once with the reference's own tokeniser,
//     asr/error.py of this package); offsets by warp scan;
//   * edit distance: anti-diagonal wavefront over the (R+1) x (H+1) table, three diagonals in shared memory;
//   * the batch mean is accumulated by the last CTA to finish, sequentially in float64 in batch order, i.e. with
//     the rounding of the reference's `sum_error += ...; sum_error / len(y_batch)`.
// The reference's table is numpy.uint8 (:10), so its distances wrap at 256; uint8_wrap != 0 reproduces that
// arithmetic bit for bit, 0 gives the true distance.
#include "common.cuh"
#include "kernels.h"

namespace b200ctc {

namespace {

constexpr int kErrThreads = 128;

// Levenshtein distance between r[0..R) (shared memory) and h[0..H) (global), by all threads of the CTA.
// diag: 3 * (R + 1) ints of shared memory.  Returns d[R][H] (valid in every thread).
__device__ int edit_distance_cta(const int *r, int R, const int32_t *h, int H, int *diag, int wrap8) {
    const int mask = wrap8 ? 0xff : 0x7fffffff;
    int *d2 = diag, *d1 = diag + (R + 1), *d0 = diag + 2 * (R + 1);      // diagonals k-2, k-1, k (indexed by i)
    for (int k = 0; k <= R + H; ++k) {
        const int ilo = max(0, k - H), ihi = min(R, k);
        for (int i = ilo + (int)threadIdx.x; i <= ihi; i += blockDim.x) {
            const int j = k - i;
            int v;
            if (i == 0) v = j & mask;                                     // asr/error.py:13
            else if (j == 0) v = i & mask;                                // :14
            else if (r[i - 1] == h[j - 1]) v = d2[i - 1];                 // :17-18
            else {
                const int sub = (d2[i - 1] + 1) & mask;                   // :20
                const int ins = (d1[i] + 1) & mask;                       // :21  d[i][j-1]
                const int del = (d1[i - 1] + 1) & mask;                   // :22  d[i-1][j]
                v = min(sub, min(ins, del));                              // :23
            }
            d0[i] = v;
        }
        __syncthreads();
        int *t = d2; d2 = d1; d1 = d0; d0 = t;
    }
    return d1[R];                                                         // the last diagonal written
}

__device__ void finish_utterance(int b, int B, int R, int H, int dist, int32_t *hyp_len, int32_t *ref_len,
                                 int32_t *distance, double *err_per_utt, double *err_mean, unsigned *done) {
    if (threadIdx.x != 0) return;
    const double e = (R == 0) ? (double)H : (double)dist / (double)R;     // asr/error.py:8-9, :24
    if (hyp_len) hyp_len[b] = H;
    if (ref_len) ref_len[b] = R;
    if (distance) distance[b] = dist;
    err_per_utt[b] = e;
    __threadfence();
    if (atomicAdd(done, 1u) + 1u == (unsigned)B) {                        // last CTA: batch mean, in batch order (:55, :68)
        __threadfence();
        double s = 0.0;
        for (int i = 0; i < B; ++i) s += __ldcg(err_per_utt + i);
        if (err_mean) *err_mean = s / (double)B;
        *done = 0u;
    }
}

__global__ void __launch_bounds__(kErrThreads) greedy_error_kernel(
    const int64_t *__restrict__ argmax, const int32_t *__restrict__ input_lengths, int B, int T,
    const int32_t *__restrict__ labels, int Lmax, int blank, const int32_t *__restrict__ expansion, int V, int E,
    int wrap8, int32_t *hyp, int Hmax, int32_t *hyp_len, int32_t *ref_len, int32_t *distance, double *err_per_utt,
    double *err_mean, unsigned *done) {
    extern __shared__ int sm[];
    __shared__ int s_R, s_H;
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int *r = sm;                                  // [Lmax]
    int *diag = sm + Lmax;                        // [3 * (Lmax + 1)]
    int32_t *h = hyp + (size_t)b * Hmax;

    if (warp == 0) {
        // ---- collapse + expansion (asr/error.py:38-53) ----
        int Tb = input_lengths ? clamp_length(input_lengths[b], T) : T;
        int base = 0, prev_last = blank;
        for (int t0 = 0; t0 < Tb; t0 += 32) {
            const int t = t0 + lane;
            const int tok = t < Tb ? (int)argmax[(size_t)b * T + t] : blank;
            int prev = __shfl_up_sync(0xffffffffu, tok, 1);
            if (lane == 0) prev = prev_last;
            const bool keep = t < Tb && tok != blank && tok != prev;
            int n = 0;
            if (keep && tok >= 0 && tok < V)
                while (n < E && expansion[(size_t)tok * E + n] >= 0) ++n;
            int incl = n;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            const int off = base + incl - n;
            for (int k = 0; k < n; ++k) h[off + k] = expansion[(size_t)tok * E + k];
            base += __shfl_sync(0xffffffffu, incl, 31);
            prev_last = __shfl_sync(0xffffffffu, tok, 31);
        }
        if (lane == 0) s_H = base;
    } else if (warp == 1) {
        // ---- target without blanks (:33-37) ----
        int base = 0;
        for (int l0 = 0; l0 < Lmax; l0 += 32) {
            const int l = l0 + lane;
            const int lab = l < Lmax ? labels[(size_t)b * Lmax + l] : blank;
            const bool keep = l < Lmax && lab != blank;
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (keep) r[base + __popc(m & ((1u << lane) - 1u))] = lab;
            base += __popc(m);
        }
        if (lane == 0) s_R = base;
    }
    __syncthreads();                              // also orders warp 0's global writes of h before the reads below
    const int R = s_R, H = s_H;
    const int dist = edit_distance_cta(r, R, h, H, diag, wrap8);
    finish_utterance(b, B, R, H, dist, hyp_len, ref_len, distance, err_per_utt, err_mean, done);
}

// explicit sequences: ref (B, Rmax) with ref_len, hyp (B, Hmax) with hyp_len
__global__ void __launch_bounds__(kErrThreads) edit_distance_kernel(
    const int32_t *__restrict__ ref, const int32_t *__restrict__ ref_len_in, int Rmax, const int32_t *__restrict__ hyp,
    const int32_t *__restrict__ hyp_len_in, int Hmax, int B, int wrap8, int32_t *distance, double *err_per_utt,
    double *err_mean, unsigned *done) {
    extern __shared__ int sm[];
    const int b = blockIdx.x;
    int *r = sm;
    int *diag = sm + Rmax;
    const int R = clamp_length(ref_len_in[b], Rmax), H = clamp_length(hyp_len_in[b], Hmax);
    for (int i = threadIdx.x; i < R; i += blockDim.x) r[i] = ref[(size_t)b * Rmax + i];
    __syncthreads();
    const int dist = edit_distance_cta(r, R, hyp + (size_t)b * Hmax, H, diag, wrap8);
    finish_utterance(b, B, R, H, dist, nullptr, nullptr, distance, err_per_utt, err_mean, done);
}

size_t err_smem(int Rmax) { return sizeof(int) * ((size_t)Rmax + 3 * ((size_t)Rmax + 1)); }

}  // namespace

cudaError_t launch_greedy_error(const int64_t *argmax, const int32_t *input_lengths, int B, int T, const int32_t *labels,
                                int Lmax, int blank, const int32_t *expansion, int V, int E, int wrap8, int32_t *hyp,
                                int32_t *hyp_len, int32_t *ref_len, int32_t *distance, double *err_per_utt,
                                double *err_mean, unsigned *done, cudaStream_t stream) {
    const size_t smem = err_smem(Lmax);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(greedy_error_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    greedy_error_kernel<<<B, kErrThreads, smem, stream>>>(argmax, input_lengths, B, T, labels, Lmax, blank, expansion, V, E,
                                                         wrap8, hyp, T * E, hyp_len, ref_len, distance, err_per_utt,
                                                         err_mean, done);
    return cudaGetLastError();
}

cudaError_t launch_edit_distance(const int32_t *ref, const int32_t *ref_len, int Rmax, const int32_t *hyp,
                                 const int32_t *hyp_len, int Hmax, int B, int wrap8, int32_t *distance,
                                 double *err_per_utt, double *err_mean, unsigned *done, cudaStream_t stream) {
    const size_t smem = err_smem(Rmax);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(edit_distance_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    edit_distance_kernel<<<B, kErrThreads, smem, stream>>>(ref, ref_len, Rmax, hyp, hyp_len, Hmax, B, wrap8, distance,
                                                          err_per_utt, err_mean, done);
    return cudaGetLastError();
}

}  // namespace b200ctc
