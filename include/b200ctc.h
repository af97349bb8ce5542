/*
 * b200ctc.h -- C ABI of the B200-native CTC / Gram-CTC loss (forward + backward).
 *
 * This is the drop-in boundary for the loss path of musyoku/chainer-speech-recognition:
 *   asr/loss/gram_ctc.py:300      gram_ctc(xs, label_unigram, label_bigram, blank_symbol,
 *                                          input_length, length_unigram, reduce)
 *   run/ctc/cnn/train.py:191      F.connectionist_temporal_classification(y, t, blank, x_len, t_len)
 *   run/ctc/cnn/train.py:232      xp.argmax(y.data, axis=2)            (greedy path)
 * The reference's binding for it is Python (a chainer.Function subclass); the replacement binding
 * is a ctypes stub (see INTEGRATION.md) that calls the functions below.
 *
 * Conventions
 *   - plain C types only; every pointer is a CUDA *device* pointer unless the name ends in _host;
 *   - the caller owns every buffer, including the workspace; the library keeps no device memory
 *     and no global state besides a thread-local last-error string, host-side lookup caches (SM
 *     count, per-kernel shared-memory opt-in, environment switches) and, per host thread and device,
 *     one internal side stream with two events (b200ctc_forward runs the lattice kernel on it next
 *     to the softmax kernel; forked from and joined back into `stream`, capturable in a CUDA graph;
 *     destroyed when the host thread exits);
 *   - every function returns a status code (B200CTC_OK == 0) and never throws;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*); no entry point synchronises the
 *     device or touches host copies of the data (host-array convenience wrappers live in the Python
 *     package, asr/loss/host.py, on top of these entry points);
 *   - activations and gradients need 4-byte alignment only: rows of any vocabulary size and pitch take
 *     the TMA path (the reference's vocabulary is 119 unigram ids + the bigrams that pass a count
 *     filter, asr/vocab.py:62-97 -- rarely a multiple of 4);
 *   - activations are float32, element (t, b, v) at acts[t*stride_t + b*stride_b + v] (vocabulary
 *     stride is 1), which covers the reference's stacked (T,B,V) layout (gram_ctc.py:272-273) and
 *     the decoder's (B,T,V) layout (asr/model/cnn.py:45-47) without a copy;
 *   - labels are int32, (B, Lmax) row-major, padded with any value (the data layer pads with the
 *     blank id, asr/data/processing.py:125-126); a Gram-CTC bigram id of -1 marks a bigram that is
 *     not in the inventory (asr/data/processing.py:139-146, gram_ctc.py:94-98);
 *   - input_lengths / label_lengths are int32 (B) or NULL for "full length" (gram_ctc.py:310-313).
 */
#ifndef B200CTC_H_
#define B200CTC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200CTC_VERSION 201

enum {
    B200CTC_OK = 0,
    B200CTC_INVALID_ARGUMENT = 1,   /* -> ValueError / TypeError in the Python shim              */
    B200CTC_UNSUPPORTED = 2,        /* shape outside what the kernels are instantiated for       */
    B200CTC_CUDA_ERROR = 3,         /* launch / runtime failure; message in b200ctc_last_error() */
    B200CTC_WORKSPACE_TOO_SMALL = 4,
    B200CTC_OUT_OF_MEMORY = 5       /* cudaErrorMemoryAllocation from a launch -> torch.cuda.OutOfMemoryError
                                       (buffers are the caller's, so this is rare; WORKSPACE_TOO_SMALL maps to the
                                       same Python exception, which is what the reference's batch-size search
                                       catches, run/ctc/cnn/train.py:204-211) */
};

/* JOINT: Gram-CTC loss + plain CTC loss of the same activations and unigram labels in one pass
 * (run/gram_ctc/cnn/train.py:196-198, `loss = gram_ctc(...); loss += F.connectionist_temporal_classification(...)`):
 * one softmax pass, one re-read and one gradient write instead of two of each.  loss outputs are the sums of the
 * two losses, the gradient is the gradient of the sum. */
enum { B200CTC_KIND_CTC = 0, B200CTC_KIND_GRAM = 1, B200CTC_KIND_JOINT = 2 };

/* flags for b200ctc_forward */
enum {
    B200CTC_FLAG_NONE = 0,
    B200CTC_FLAG_SERIAL = 1         /* run the lattice kernel behind the softmax/gather kernel instead of next to it
                                       (same results bit for bit; for debugging and for callers that must not have
                                       a second stream involved) */
};

int b200ctc_version(void);
const char *b200ctc_last_error(void);

/* Bytes of device workspace the forward/backward pair needs (replaces the reference's saved
 * `yseq` + `prob_trans`, gram_ctc.py:273,276).  16-byte aligned base required. */
int b200ctc_workspace_bytes(int kind, int B, int T, int V, int Lmax, size_t *bytes_out);

/*
 * Forward: replaces GramCTC.forward (gram_ctc.py:246-282) / Chainer's CTC forward.
 *   loss_per_utt  (B) float32, out: -log P(labels_b | x_b); exactly 1e10 for an infeasible
 *                 alignment (what the reference returns).
 *   loss_reduced  (1) float32, out: loss_scale * sum_b loss_per_utt[b], summed in a fixed order.
 *                 reduce='mean' (gram_ctc.py:281): loss_scale = 1 / B_global; on several GPUs the
 *                 caller all-reduces (sum) this one float across ranks.
 *   argmax_out    (B,T) int64 or NULL: greedy indices over the raw activations, first maximum
 *                 wins, NaN counts as maximal (numpy.argmax semantics, run/ctc/cnn/train.py:232).
 *   bigrams       NULL for kind == B200CTC_KIND_CTC.
 */
int b200ctc_forward(int kind,
                    const float *acts, int64_t stride_t, int64_t stride_b,
                    const int32_t *labels, const int32_t *bigrams,
                    const int32_t *input_lengths, const int32_t *label_lengths,
                    int blank, int B, int T, int V, int Lmax,
                    float *loss_per_utt, float *loss_reduced, float loss_scale, int64_t *argmax_out,
                    void *workspace, size_t workspace_bytes, unsigned flags, void *stream);

/*
 * Backward: replaces GramCTC.backward (gram_ctc.py:284-297).  Must follow a b200ctc_forward on the
 * same workspace and activations.
 *   grad_loss        device pointer: 1 float (per_utterance == 0, reduce='mean') or (B) floats
 *                    (per_utterance == 1, reduce='no'), the upstream gradient gy (gram_ctc.py:291-294).
 *   scale            extra factor applied to every element: 1/B_global for 'mean' (:292), 1 for 'no'.
 *   grad_out         float32, element (t,b,v) at grad_out[t*gstride_t + b*gstride_b + v]; every one of
 *                    the B*T*V elements is written, zeros for t >= input_lengths[b] (:296).
 */
int b200ctc_backward(int kind,
                     const float *acts, int64_t stride_t, int64_t stride_b,
                     const int32_t *labels, const int32_t *bigrams,
                     int blank, int B, int T, int V, int Lmax,
                     const float *grad_loss, int per_utterance, float scale,
                     float *grad_out, int64_t gstride_t, int64_t gstride_b,
                     const void *workspace, size_t workspace_bytes, void *stream);

/*
 * LayerNormalization fused into the loss (SURVEY.md 8f rank 3).  Every CTC / Gram-CTC model of the reference ends in
 * Convolution2D(.., vocab_size, ksize=1) -> LayerNormalization (run/ctc/cnn/model.py:85-88, asr/nn/nn.py:240-265,
 * asr/nn/layernorm.py:29-61), after which AcousticModel.__call__ makes a transposed copy of the whole tensor for the
 * loss (swapaxes/reshape/split_axis, asr/model/cnn.py:41-44).  These entry points take the convolution output itself:
 *   z        float32 (B, V, 1, T) as the model produces it: element (b, v, t) at z[b*zstride_b + v*zstride_v + t]
 *            (time stride 1); rows must be 16-byte aligned (base pointer, zstride_v % 4 == 0, zstride_b % 4 == 0)
 *   gamma, beta  float32 (V): LayerNormalization's scale and shift along the vocabulary axis
 * and compute  loss(gamma * (z - mean_v z) / std_v z + beta)  per frame, std = sqrt(mean_v (z - mean)^2), no epsilon
 * (asr/nn/layernorm.py:41-46).  Backward returns the gradient where the model needs it:
 *   dz       float32, same layout rules as z; every element is written (zeros for t >= input_lengths[b])
 *   dgamma, dbeta  float32 (V) or NULL: sums over all frames of the batch, in a fixed order (deterministic)
 * with LayerNormalization's backward (asr/nn/layernorm.py:48-60) and both transposes folded in: z is read once in
 * forward, once in backward, dz is written once.  loss outputs, grad_loss / per_utterance / scale as in
 * b200ctc_forward / b200ctc_backward.  kind may be B200CTC_KIND_JOINT: the loss outputs are then the sums of the
 * Gram-CTC and the plain-CTC loss, and dz / dgamma / dbeta are the gradients of that sum.
 * Returns B200CTC_UNSUPPORTED (use the unfused entry points) for V > 4080, more than 480 emission columns (1 + Lmax for
 * CTC, 1 + 2*Lmax for Gram-CTC and joint), unaligned rows, or an Lmax too long for the backward kernel's tile to fit in
 * shared memory at this V (at V = 4080: Lmax > 97 for CTC, Lmax > 63 for Gram-CTC and joint).  b200ctc_ln_forward
 * already refuses a shape whose backward pass could not run, so a caller can take the unfused path before any work is
 * enqueued.
 */
int b200ctc_ln_workspace_bytes(int kind, int B, int T, int V, int Lmax, size_t *bytes_out);
int b200ctc_ln_forward(int kind,
                       const float *z, int64_t zstride_b, int64_t zstride_v, const float *gamma, const float *beta,
                       const int32_t *labels, const int32_t *bigrams,
                       const int32_t *input_lengths, const int32_t *label_lengths,
                       int blank, int B, int T, int V, int Lmax,
                       float *loss_per_utt, float *loss_reduced, float loss_scale,
                       void *workspace, size_t workspace_bytes, unsigned flags, void *stream);
int b200ctc_ln_backward(int kind,
                        const float *z, int64_t zstride_b, int64_t zstride_v, const float *gamma, const float *beta,
                        const int32_t *labels, const int32_t *bigrams,
                        int blank, int B, int T, int V, int Lmax,
                        const float *grad_loss, int per_utterance, float scale,
                        float *dz, int64_t dzstride_b, int64_t dzstride_v, float *dgamma, float *dbeta,
                        const void *workspace, size_t workspace_bytes, void *stream);

/* Greedy path alone (run/ctc/cnn/train.py:232 and its 9 sibling call sites): out (B,T) int64. */
int b200ctc_greedy_argmax(const float *acts, int64_t stride_t, int64_t stride_b,
                          int B, int T, int V, int64_t *argmax_out, void *stream);

/*
 * Evaluation path after the greedy argmax (SURVEY.md 8f rank 1): replaces compute_minibatch_error
 * (asr/error.py:26-68) -- called on every development batch, run/ctc/cnn/train.py:231-233 -- and
 * compute_character_error_rate (asr/error.py:7-24).
 *   argmax        (B,T) int64: greedy ids (b200ctc_greedy_argmax / argmax_out of b200ctc_forward).
 *   input_lengths (B) int32 or NULL: frames to decode per utterance.  The reference decodes all T
 *                 frames of the padded batch (asr/error.py:40), i.e. NULL.
 *   labels        (B,Lmax) int32 targets padded with the blank id; blanks are dropped (:33-37).
 *   expansion     (V,E) int32: the unigram ids a vocabulary id stands for, padded with -1 -- the
 *                 reference's string round trip id -> token -> convert_sentence_to_unigram_ids
 *                 (:49-53, asr/vocab.py:99-126), tabulated once on the host.
 *   uint8_wrap    != 0: distances computed modulo 256 exactly as the reference's numpy.uint8 table
 *                 does (:10); 0: true Levenshtein distance.
 *   hyp_out       (B, T*E) int32 scratch/out: collapsed + expanded hypothesis; hyp_len (B) its length.
 *   ref_len, distance (B) int32 or NULL;  err_per_utt (B) float64: distance / ref_len, or hyp_len
 *                 for an empty target (:8-9);  err_mean (1) float64 or NULL: the batch mean, summed
 *                 in batch order in float64 like the reference's Python floats (:55, :68).
 *   workspace     B200CTC_ERROR_WORKSPACE_BYTES bytes.
 */
#define B200CTC_ERROR_WORKSPACE_BYTES 256
int b200ctc_greedy_error(const int64_t *argmax, const int32_t *input_lengths, int B, int T,
                         const int32_t *labels, int Lmax, int blank,
                         const int32_t *expansion, int V, int E, int uint8_wrap,
                         int32_t *hyp_out, int32_t *hyp_len, int32_t *ref_len, int32_t *distance,
                         double *err_per_utt, double *err_mean,
                         void *workspace, size_t workspace_bytes, void *stream);
/* Edit distance / error rate of explicit id sequences: ref (B,Rmax), hyp (B,Hmax), lengths (B). */
int b200ctc_edit_distance(const int32_t *ref, const int32_t *ref_len, int Rmax,
                          const int32_t *hyp, const int32_t *hyp_len, int Hmax, int B, int uint8_wrap,
                          int32_t *distance, double *err_per_utt, double *err_mean,
                          void *workspace, size_t workspace_bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* B200CTC_H_ */
