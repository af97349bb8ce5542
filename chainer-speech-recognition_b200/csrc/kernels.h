// kernels.h -- host-side launch interface between api.cu and the kernel translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "common.cuh"

namespace b200ctc {

// kernel 1: fused log-softmax statistics + label gather (+ optional greedy argmax)
// smem_reserve: shared memory to leave free per SM for a lattice CTA running next to this kernel (0 = none)
cudaError_t launch_softmax_gather(const ProblemDesc &d, const WsLayout &w, void *ws, int64_t *argmax_out,
                                  size_t smem_reserve, cudaStream_t stream);
cudaError_t launch_argmax(const float *acts, int64_t stride_t, int64_t stride_b, int B, int T, int V,
                          int64_t *argmax_out, cudaStream_t stream);

// shared by the two row-streaming kernels (defined in softmax_gather.cu)
struct RingLayout;
bool ring_usable(const void *base, const RingLayout &rl);

// ---- host-side caches (host_cache.cu): nothing below costs a driver call after its first use ----
// a launcher that fails names the step that failed; api.cu appends it to the error message
void note_failure_site(const char *where);
const char *failure_site();
int current_device();
int sm_count();                                                        // per device
// opt-in dynamic shared memory + maximum carve-out for `func`; cudaFuncSetAttribute only when more is needed than before
cudaError_t ensure_dynamic_smem(const void *func, size_t bytes);

// kernel 2: alpha/beta lattice recursion (+ symbol-table CTAs, + batch loss reduction by the last CTA)
struct LatticeParams {
    ProblemDesc d;
    WsLayout w;
    unsigned char *ws;
    float *loss_per_utt;     // (B)
    float *loss_reduced;     // (1): loss_scale * sum_b loss_b
    float loss_scale;
    int W;                   // warps per direction
    int S;                   // pipeline stages
    int second;              // 1: this is the plain-CTC lattice of a joint call -- no symbol-table CTAs, its own
                             //    completion counter, and its loss is ADDED to loss_per_utt (the Gram-CTC launch,
                             //    earlier in the stream, has written its own there) before the batch is reduced
};
// the view of a joint workspace that the plain-CTC lattice launch works on
WsLayout ctc_view_of_joint(const WsLayout &w);
int lattice_max_nodes(int kind);
// concurrent: the kernel is going to run next to the softmax/gather kernel (fewer pipeline stages, so that a
// lattice CTA fits beside a ring CTA); smem_out, if not NULL, receives the dynamic shared memory per CTA.
// With launch = false nothing is launched (planning call).
cudaError_t launch_lattice(LatticeParams p, cudaStream_t stream, int *status, bool concurrent = false,
                           size_t *smem_out = nullptr, bool launch = true);

// kernel 3: fused gradient
struct GradParams {
    ProblemDesc d;
    const float *grad_loss;
    int per_utterance;
    float scale;
    float *grad_out;
    int64_t gstride_t, gstride_b;
};
cudaError_t launch_gradient(const GradParams &g, const WsLayout &w, const void *ws, cudaStream_t stream);
// LayerNormalization fused into the loss (layernorm_loss.cu, SURVEY.md 8f rank 3): the kernels read the model's last
// convolution output z (B, V, T) in place instead of the normalised, transposed copy the reference hands to the loss
constexpr int kLnMaxParts = 160;          // CTAs of the backward kernel (>= SM count): rows of the dgamma/dbeta partial sums
struct LnLayout {
    WsLayout w;                           // the regular workspace ...
    size_t off_mu, off_rstd, off_lse, off_part;   // ... + per-frame mean, 1/std, log2 normaliser; per-CTA dgamma/dbeta partial rows
    size_t total;
};
LnLayout make_ln_layout(int kind, int B, int T, int V, int Lmax);
int ln_supported(int kind, int B, int T, int V, int Lmax, int64_t zs_v, int64_t zs_b, const void *z);
cudaError_t launch_ln_forward(const ProblemDesc &d, const LnLayout &ll, void *ws, const float *z, int64_t zs_b, int64_t zs_v,
                              const float *gamma, const float *beta, size_t smem_reserve, cudaStream_t stream);
cudaError_t launch_ln_backward(const GradParams &g, const LnLayout &ll, const void *ws, const float *z, int64_t zs_b,
                               int64_t zs_v, const float *gamma, const float *beta, float *dz, int64_t dzs_b, int64_t dzs_v,
                               float *dgamma, float *dbeta, cudaStream_t stream);
// greedy argmax of the normalised z (all T frames), one read of z and no workspace; the caller has checked V <= 4080 and
// 16-byte aligned rows.  cudaErrorNotSupported: the driver could not describe z as a TMA tensor
cudaError_t launch_ln_argmax(const float *z, int64_t zs_b, int64_t zs_v, const float *gamma, const float *beta, int B, int T, int V,
                             int64_t *argmax_out, cudaStream_t stream);

// forced alignment (viterbi.cu): best path through the lattice on the emission rows of kernel 1, backpointers in the
// workspace's alpha region
struct AlignParams {
    ProblemDesc d;
    WsLayout w;
    unsigned char *ws;
    float *score;            // (B)
    int32_t *path;           // (B,T)
    int64_t *ids;            // (B,T)
    float *frame_logp;       // (B,T) or NULL
    int32_t *spans;          // (B,Lmax,2) or NULL
    int buf_stride, chunk;   // set by launch_align
};
struct AlignGeometry {
    int threads, npt;        // block size, consecutive lattice nodes per thread
    int stride;              // pitch of a score row in shared memory (float2)
    int chunk;               // frames per emission stage
};
// dynamic shared memory of the alignment kernel for this layout, and its geometry (g may be NULL)
size_t align_smem_bytes(const WsLayout &w, AlignGeometry *g);
cudaError_t launch_align(AlignParams p, cudaStream_t stream);

// evaluation path: greedy collapse + gram expansion + edit distance + error rate (greedy_error.cu)
cudaError_t launch_greedy_error(const int64_t *argmax, const int32_t *input_lengths, int B, int T, const int32_t *labels,
                                int Lmax, int blank, const int32_t *expansion, int V, int E, int wrap8, int32_t *hyp,
                                int32_t *hyp_len, int32_t *ref_len, int32_t *distance, double *err_per_utt,
                                double *err_mean, unsigned *done, cudaStream_t stream);
cudaError_t launch_edit_distance(const int32_t *ref, const int32_t *ref_len, int Rmax, const int32_t *hyp,
                                 const int32_t *hyp_len, int Hmax, int B, int wrap8, int32_t *distance,
                                 double *err_per_utt, double *err_mean, unsigned *done, cudaStream_t stream);

}  // namespace b200ctc
