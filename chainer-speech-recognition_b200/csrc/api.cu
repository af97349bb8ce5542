// api.cu -- extern "C" entry points declared in include/b200ctc.h.
//
// Plain pointers and sizes in, status codes out; the caller (PyTorch via ctypes) owns every buffer.
// Reference interface replaced: asr/loss/gram_ctc.py:219-315 (GramCTC / gram_ctc) and Chainer's
// connectionist_temporal_classification as called from run/ctc/cnn/train.py:191.
#include <stdio.h>
#include <string.h>

#include "../../include/b200ctc.h"
#include "common.cuh"
#include "kernels.h"

using namespace b200ctc;

namespace {

// zeroes the workspace header (ticket counters) and the frame-progress counters in stream order
__global__ void zero_header_kernel(WsHeader *h, unsigned *prog, int nprog) {
    if (blockIdx.x == 0 && threadIdx.x == 0) { h->k1_ticket = 0u; h->k3_ticket = 0u; h->k3_done = 0u; h->k2_done = 0u; h->k2b_done = 0u; h->stalled = 0u; }
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nprog; i += gridDim.x * blockDim.x) prog[i] = 0u;
}

// Side stream on which the lattice kernel runs next to the softmax/gather kernel (fork/join by events, so the
// caller still sees one stream; capturable into a CUDA graph).  One per host thread and device, created on first
// use and destroyed with the thread: the only state the library holds besides the last-error string and the
// host-side lookup caches (host_cache.cu).
struct SideStream {
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};
constexpr int kMaxDevices = 64;
struct SideStreams {
    SideStream s[kMaxDevices];
    ~SideStreams() {
        for (int i = 0; i < kMaxDevices; ++i) {
            if (!s[i].stream) continue;
            // at process exit the runtime may already be gone: every call below then fails harmlessly
            cudaEventDestroy(s[i].fork);
            cudaEventDestroy(s[i].join);
            cudaStreamDestroy(s[i].stream);
            (void)cudaGetLastError();
        }
    }
};
thread_local SideStreams g_side;

SideStream *side_stream() {
    const int dev = current_device();
    if (dev < 0 || dev >= kMaxDevices) return nullptr;
    SideStream &s = g_side.s[dev];
    if (!s.stream) {
        if (cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess) { s.stream = nullptr; return nullptr; }
        if (cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming) != cudaSuccess) {
            cudaStreamDestroy(s.stream);
            if (s.fork) cudaEventDestroy(s.fork);
            s = SideStream();
            (void)cudaGetLastError();
            return nullptr;
        }
    }
    return &s;
}

thread_local char g_err[512] = "";

int fail(int code, const char *fmt, const char *a = "", long long x = 0, long long y = 0) {
    snprintf(g_err, sizeof(g_err), fmt, a, x, y);
    return code;
}

int check_cuda(cudaError_t e, const char *what) {
    if (e == cudaSuccess) return B200CTC_OK;
    const char *site = failure_site();
    snprintf(g_err, sizeof(g_err), "%s: %s%s%s", what, cudaGetErrorString(e), site[0] ? " at " : "", site);
    (void)cudaGetLastError();                       // do not leave the error behind for an unrelated later call
    return e == cudaErrorMemoryAllocation ? B200CTC_OUT_OF_MEMORY : B200CTC_CUDA_ERROR;
}

int validate(int kind, int B, int T, int V, int Lmax, int blank, bool need_blank) {
    if (kind != B200CTC_KIND_CTC && kind != B200CTC_KIND_GRAM && kind != B200CTC_KIND_JOINT)
        return fail(B200CTC_INVALID_ARGUMENT, "kind must be 0 (CTC), 1 (Gram-CTC) or 2 (joint)%s");
    if (B < 0 || T < 0 || V <= 0 || Lmax < 0)
        return fail(B200CTC_INVALID_ARGUMENT, "negative or empty dimension%s (B=%lld ...)", "", B);
    if ((long long)B * (long long)T >= (1ll << 31))
        return fail(B200CTC_UNSUPPORTED, "B*T = %s%lld frames exceeds 2^31", "", (long long)B * T);
    if (need_blank && (blank < 0 || blank >= V))
        return fail(B200CTC_INVALID_ARGUMENT, "blank symbol %s%lld outside [0, V=%lld)", "", blank, V);
    const int Nmax = (kind == 0 ? 2 : 3) * Lmax + 1;
    if (Nmax > lattice_max_nodes(kind))
        return fail(B200CTC_UNSUPPORTED, "lattice of %s%lld nodes exceeds the %lld this build instantiates", "", Nmax,
                    lattice_max_nodes(kind));
    return B200CTC_OK;
}

// LayerNormalization fused in front of the loss (layernorm_loss.cu): z (B, V, T) + gamma/beta instead of activations
struct LnInput {
    const float *z;
    int64_t zs_b, zs_v;
    const float *gamma, *beta;
};

int forward_impl(const LnInput *ln, int kind, const float *acts, int64_t stride_t, int64_t stride_b, const int32_t *labels,
                 const int32_t *bigrams, const int32_t *input_lengths, const int32_t *label_lengths, int blank, int B, int T,
                 int V, int Lmax, float *loss_per_utt, float *loss_reduced, float loss_scale, int64_t *argmax_out,
                 void *workspace, size_t workspace_bytes, unsigned flags, void *stream_) {
    int rc = validate(kind, B, T, V, Lmax, blank, true);
    if (rc) return rc;
    if (!ln && !acts && (size_t)B * T > 0) return fail(B200CTC_INVALID_ARGUMENT, "acts is NULL%s");
    if (ln) {
        if ((!ln->z && (size_t)B * T > 0) || !ln->gamma || !ln->beta) return fail(B200CTC_INVALID_ARGUMENT, "z, gamma or beta is NULL%s");
        if (argmax_out) return fail(B200CTC_UNSUPPORTED, "the fused LayerNormalization path has no greedy output%s");
        if (!ln_supported(kind, B, T, V, Lmax, ln->zs_v, ln->zs_b, ln->z))
            return fail(B200CTC_UNSUPPORTED, "fused LayerNormalization needs V <= 4080, <= 480 emission columns, a label length whose "
                                             "backward tile fits shared memory at this V, and 16-byte aligned rows of z "
                                             "(pitch %% 4 == 0)%s");
    }
    if (!labels && Lmax > 0) return fail(B200CTC_INVALID_ARGUMENT, "labels is NULL%s");
    if (kind != B200CTC_KIND_CTC && !bigrams && Lmax > 0) return fail(B200CTC_INVALID_ARGUMENT, "bigrams is NULL for Gram-CTC%s");
    if (!loss_per_utt || !loss_reduced || !workspace) return fail(B200CTC_INVALID_ARGUMENT, "output or workspace pointer is NULL%s");
    if ((reinterpret_cast<uintptr_t>(workspace) & 15) != 0) return fail(B200CTC_INVALID_ARGUMENT, "workspace must be 16-byte aligned%s");
    if ((reinterpret_cast<uintptr_t>(acts) & 3) != 0) return fail(B200CTC_INVALID_ARGUMENT, "acts must be 4-byte aligned%s");
    const LnLayout ll = ln ? make_ln_layout(kind, B, T, V, Lmax) : LnLayout();
    const WsLayout w = ln ? ll.w : make_layout(kind, B, T, V, Lmax);
    const size_t need = ln ? ll.total : w.total;
    if (workspace_bytes < need)
        return fail(B200CTC_WORKSPACE_TOO_SMALL, "workspace too small%s: %lld < %lld bytes", "", (long long)workspace_bytes,
                    (long long)need);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (B == 0) return check_cuda(cudaMemsetAsync(loss_reduced, 0, sizeof(float), stream), "memset");

    ProblemDesc d;
    d.kind = kind == B200CTC_KIND_CTC ? 0 : 1; d.B = B; d.T = T; d.V = V; d.Lmax = Lmax; d.blank = blank;
    d.acts = acts; d.stride_t = stride_t; d.stride_b = stride_b;
    d.labels = labels; d.bigrams = kind != B200CTC_KIND_CTC ? bigrams : nullptr;
    d.input_lengths = input_lengths; d.label_lengths = label_lengths;
    d.progress = 0;
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    const int nprog = B * w.nblk;
    zero_header_kernel<<<(nprog + 255) / 256 > 0 ? (nprog + 255) / 256 : 1, 256, 0, stream>>>(
        reinterpret_cast<WsHeader *>(ws + w.off_hdr), reinterpret_cast<unsigned *>(ws + w.off_prog), nprog);
    if ((rc = check_cuda(cudaGetLastError(), "workspace header reset"))) return rc;

    LatticeParams lp;
    lp.d = d; lp.w = w; lp.ws = ws;
    lp.loss_per_utt = loss_per_utt; lp.loss_reduced = loss_reduced; lp.loss_scale = loss_scale;
    lp.W = 0; lp.S = 0; lp.second = 0; lp.dbg_nostore = 0;
    int st = 0;
    // joint Gram-CTC + CTC: the plain-CTC lattice is a second launch behind the Gram-CTC one (same stream), on the
    // same emission rows; it adds its loss to loss_per_utt and reduces the batch
    LatticeParams lp2 = lp;
    if (w.joint) {
        lp2.d.kind = 0; lp2.d.bigrams = nullptr;
        lp2.w = ctc_view_of_joint(w);
        lp2.second = 1;
    }

    // The lattice kernel runs NEXT TO the softmax/gather kernel, on a side stream: the recursion is a latency-bound
    // dependent chain that needs a few warps per utterance, the softmax a bandwidth-bound stream over all SMs, and
    // the first feeds the second frame by frame through the progress counters (common.cuh).  Tickets walk the
    // frames from both ends, so alpha and beta both find their next rows ready; what remains exposed is the second
    // half of each direction after the last row has been produced.
    // No deadlock: the softmax kernel never waits on the lattice kernel, and the concurrent mode is only chosen when
    // every SM keeps room for a ring CTA whatever the lattice CTAs do: 2*B lattice CTAs can close an SM to the ring
    // kernel only two at a time (launch_softmax_gather sizes its ring for ONE lattice CTA beside it), so 2*B/2 < #SMs
    // leaves at least one SM per missing pair, and the ring kernel is persistent (any number of its CTAs makes progress).
    SideStream *side = nullptr;
    size_t lat_smem = 0;
    const bool concurrent_ok = B < sm_count() && T > 0 && !(flags & B200CTC_FLAG_SERIAL);
    if (concurrent_ok) {
        if ((rc = check_cuda(launch_lattice(lp, stream, &st, true, &lat_smem, false), "lattice kernel"))) return rc;
        if (!st) side = side_stream();
        st = 0;
    }
    if (side) {
        d.progress = 3;
#ifdef B200CTC_EXPERIMENT
        if (knobs().dbg_progress >= 0) d.progress = knobs().dbg_progress;
#endif
        lp.d = d;
        if ((rc = check_cuda(cudaEventRecord(side->fork, stream), "fork event"))) return rc;
        if (ln) {
            if ((rc = check_cuda(launch_ln_forward(d, ll, ws, ln->z, ln->zs_b, ln->zs_v, ln->gamma, ln->beta, lat_smem, stream),
                                 "layernorm softmax/gather kernel"))) return rc;
        } else if ((rc = check_cuda(launch_softmax_gather(d, w, ws, argmax_out, lat_smem, stream), "softmax/gather kernel"))) return rc;
        if ((rc = check_cuda(cudaStreamWaitEvent(side->stream, side->fork, 0), "fork wait"))) return rc;
        if ((rc = check_cuda(launch_lattice(lp, side->stream, &st, true), "lattice kernel"))) return rc;
        if (w.joint && !st) {
            lp2.d.progress = d.progress;
            if ((rc = check_cuda(launch_lattice(lp2, side->stream, &st, false), "CTC lattice kernel"))) return rc;
        }
        if ((rc = check_cuda(cudaEventRecord(side->join, side->stream), "join event"))) return rc;
        if ((rc = check_cuda(cudaStreamWaitEvent(stream, side->join, 0), "join wait"))) return rc;
    } else {
#ifdef B200CTC_EXPERIMENT
        if (knobs().dbg_progress >= 0) d.progress = knobs().dbg_progress & 64;      // streaming-rate experiment (softmax_gather.cu)
#endif
        if (ln) {
            if ((rc = check_cuda(launch_ln_forward(d, ll, ws, ln->z, ln->zs_b, ln->zs_v, ln->gamma, ln->beta, 0, stream),
                                 "layernorm softmax/gather kernel"))) return rc;
        } else if ((rc = check_cuda(launch_softmax_gather(d, w, ws, argmax_out, 0, stream), "softmax/gather kernel"))) return rc;
        if ((rc = check_cuda(launch_lattice(lp, stream, &st), "lattice kernel"))) return rc;
        if (w.joint && !st && (rc = check_cuda(launch_lattice(lp2, stream, &st), "CTC lattice kernel"))) return rc;
    }
    if (st) return fail(B200CTC_UNSUPPORTED, "lattice of %s%lld nodes does not fit the kernel's shared-memory pipeline", "", w.Nmax);
    return B200CTC_OK;
}

}  // namespace

#ifdef B200CTC_EXPERIMENT
namespace b200ctc {
void lattice_set_debug(long long *p);
void lattice_set_timeline(long long *p);
void softmax_set_timeline(long long *p);
void softmax_set_roles(long long *p);
void ln_set_debug(long long *p);
void gradient_set_timeline(long long *p);
}
#endif

extern "C" {

#ifdef B200CTC_EXPERIMENT
/* profiling hooks of the experiment build (tools/step_timeline.py, tools/lattice_timeline.py); not part of the ABI */
void b200ctc_debug_lattice(long long *p) { b200ctc::lattice_set_debug(p); }
void b200ctc_debug_k1_roles(long long *p) { b200ctc::softmax_set_roles(p); }
void b200ctc_debug_ln(long long *p) { b200ctc::ln_set_debug(p); }
void b200ctc_debug_timeline(long long *p) {
    b200ctc::softmax_set_timeline(p); b200ctc::lattice_set_timeline(p); b200ctc::gradient_set_timeline(p);
}
#endif

int b200ctc_version(void) { return B200CTC_VERSION; }

const char *b200ctc_last_error(void) { return g_err; }

int b200ctc_workspace_bytes(int kind, int B, int T, int V, int Lmax, size_t *bytes_out) {
    if (!bytes_out) return fail(B200CTC_INVALID_ARGUMENT, "bytes_out is NULL%s");
    int rc = validate(kind, B, T, V, Lmax, 0, false);
    if (rc) return rc;
    *bytes_out = make_layout(kind, B, T, V, Lmax).total;
    return B200CTC_OK;
}

int b200ctc_forward(int kind, const float *acts, int64_t stride_t, int64_t stride_b, const int32_t *labels,
                    const int32_t *bigrams, const int32_t *input_lengths, const int32_t *label_lengths, int blank,
                    int B, int T, int V, int Lmax, float *loss_per_utt, float *loss_reduced, float loss_scale,
                    int64_t *argmax_out, void *workspace, size_t workspace_bytes, unsigned flags, void *stream_) {
    return forward_impl(nullptr, kind, acts, stride_t, stride_b, labels, bigrams, input_lengths, label_lengths, blank, B, T, V, Lmax,
                        loss_per_utt, loss_reduced, loss_scale, argmax_out, workspace, workspace_bytes, flags, stream_);
}

int b200ctc_backward(int kind, const float *acts, int64_t stride_t, int64_t stride_b, const int32_t *labels,
                     const int32_t *bigrams, int blank, int B, int T, int V, int Lmax, const float *grad_loss,
                     int per_utterance, float scale, float *grad_out, int64_t gstride_t, int64_t gstride_b,
                     const void *workspace, size_t workspace_bytes, void *stream_) {
    int rc = validate(kind, B, T, V, Lmax, blank, true);
    if (rc) return rc;
    if ((size_t)B * T == 0) return B200CTC_OK;
    if (!acts || !grad_loss || !grad_out || !workspace) return fail(B200CTC_INVALID_ARGUMENT, "NULL pointer%s");
    if (((reinterpret_cast<uintptr_t>(acts) | reinterpret_cast<uintptr_t>(grad_out)) & 3) != 0)
        return fail(B200CTC_INVALID_ARGUMENT, "acts and grad_out must be 4-byte aligned%s");
    const WsLayout w = make_layout(kind, B, T, V, Lmax);
    if (workspace_bytes < w.total) return fail(B200CTC_WORKSPACE_TOO_SMALL, "workspace too small%s");
    GradParams g;
    g.d.kind = kind == B200CTC_KIND_CTC ? 0 : 1; g.d.B = B; g.d.T = T; g.d.V = V; g.d.Lmax = Lmax; g.d.blank = blank;
    g.d.acts = acts; g.d.stride_t = stride_t; g.d.stride_b = stride_b;
    g.d.labels = labels; g.d.bigrams = bigrams; g.d.input_lengths = nullptr; g.d.label_lengths = nullptr;
    g.d.progress = 0;
    g.grad_loss = grad_loss; g.per_utterance = per_utterance; g.scale = scale;
    g.grad_out = grad_out; g.gstride_t = gstride_t; g.gstride_b = gstride_b;
    return check_cuda(launch_gradient(g, w, workspace, static_cast<cudaStream_t>(stream_)), "gradient kernel");
}

int b200ctc_ln_workspace_bytes(int kind, int B, int T, int V, int Lmax, size_t *bytes_out) {
    if (!bytes_out) return fail(B200CTC_INVALID_ARGUMENT, "bytes_out is NULL%s");
    int rc = validate(kind, B, T, V, Lmax, 0, false);
    if (rc) return rc;
    *bytes_out = make_ln_layout(kind, B, T, V, Lmax).total;
    return B200CTC_OK;
}

int b200ctc_ln_forward(int kind, const float *z, int64_t zstride_b, int64_t zstride_v, const float *gamma, const float *beta,
                       const int32_t *labels, const int32_t *bigrams, const int32_t *input_lengths,
                       const int32_t *label_lengths, int blank, int B, int T, int V, int Lmax, float *loss_per_utt,
                       float *loss_reduced, float loss_scale, void *workspace, size_t workspace_bytes, unsigned flags,
                       void *stream_) {
    const LnInput ln = {z, zstride_b, zstride_v, gamma, beta};
    return forward_impl(&ln, kind, nullptr, 0, 0, labels, bigrams, input_lengths, label_lengths, blank, B, T, V, Lmax,
                        loss_per_utt, loss_reduced, loss_scale, nullptr, workspace, workspace_bytes, flags, stream_);
}

int b200ctc_ln_backward(int kind, const float *z, int64_t zstride_b, int64_t zstride_v, const float *gamma, const float *beta,
                        const int32_t *labels, const int32_t *bigrams, int blank, int B, int T, int V, int Lmax,
                        const float *grad_loss, int per_utterance, float scale, float *dz, int64_t dzstride_b,
                        int64_t dzstride_v, float *dgamma, float *dbeta, const void *workspace, size_t workspace_bytes,
                        void *stream_) {
    int rc = validate(kind, B, T, V, Lmax, blank, true);
    if (rc) return rc;
    if ((size_t)B * T == 0) {
        cudaStream_t st = static_cast<cudaStream_t>(stream_);
        if (dgamma && (rc = check_cuda(cudaMemsetAsync(dgamma, 0, sizeof(float) * V, st), "memset"))) return rc;
        if (dbeta && (rc = check_cuda(cudaMemsetAsync(dbeta, 0, sizeof(float) * V, st), "memset"))) return rc;
        return B200CTC_OK;
    }
    if (!z || !gamma || !beta || !grad_loss || !dz || !workspace) return fail(B200CTC_INVALID_ARGUMENT, "NULL pointer%s");
    if (!ln_supported(kind, B, T, V, Lmax, zstride_v, zstride_b, z) || (dzstride_v & 3) != 0 || (dzstride_b & 3) != 0 ||
        (reinterpret_cast<uintptr_t>(dz) & 15) != 0)
        return fail(B200CTC_UNSUPPORTED, "fused LayerNormalization needs V <= 4080, a label length whose backward tile fits shared "
                                         "memory at this V, and 16-byte aligned rows of z and dz%s");
    const LnLayout ll = make_ln_layout(kind, B, T, V, Lmax);
    if (workspace_bytes < ll.total) return fail(B200CTC_WORKSPACE_TOO_SMALL, "workspace too small%s");
    GradParams g;
    g.d.kind = kind == B200CTC_KIND_CTC ? 0 : 1; g.d.B = B; g.d.T = T; g.d.V = V; g.d.Lmax = Lmax; g.d.blank = blank;
    g.d.acts = nullptr; g.d.stride_t = 0; g.d.stride_b = 0;
    g.d.labels = labels; g.d.bigrams = bigrams; g.d.input_lengths = nullptr; g.d.label_lengths = nullptr;
    g.d.progress = 0;
    g.grad_loss = grad_loss; g.per_utterance = per_utterance; g.scale = scale;
    g.grad_out = nullptr; g.gstride_t = 0; g.gstride_b = 0;
    return check_cuda(launch_ln_backward(g, ll, workspace, z, zstride_b, zstride_v, gamma, beta, dz, dzstride_b, dzstride_v, dgamma,
                                         dbeta, static_cast<cudaStream_t>(stream_)),
                      "layernorm gradient kernel");
}

int b200ctc_greedy_argmax(const float *acts, int64_t stride_t, int64_t stride_b, int B, int T, int V,
                          int64_t *argmax_out, void *stream_) {
    if (B < 0 || T < 0 || V <= 0) return fail(B200CTC_INVALID_ARGUMENT, "bad dimensions%s");
    if ((size_t)B * T == 0) return B200CTC_OK;
    if (!acts || !argmax_out) return fail(B200CTC_INVALID_ARGUMENT, "NULL pointer%s");
    return check_cuda(launch_argmax(acts, stride_t, stride_b, B, T, V, argmax_out, static_cast<cudaStream_t>(stream_)),
                      "argmax kernel");
}

int b200ctc_greedy_error(const int64_t *argmax, const int32_t *input_lengths, int B, int T, const int32_t *labels,
                         int Lmax, int blank, const int32_t *expansion, int V, int E, int uint8_wrap, int32_t *hyp_out,
                         int32_t *hyp_len, int32_t *ref_len, int32_t *distance, double *err_per_utt, double *err_mean,
                         void *workspace, size_t workspace_bytes, void *stream_) {
    if (B < 0 || T < 0 || Lmax < 0 || V <= 0 || E <= 0) return fail(B200CTC_INVALID_ARGUMENT, "bad dimensions%s");
    if (B == 0) return B200CTC_OK;
    if ((!argmax && T > 0) || (!labels && Lmax > 0) || !expansion || (!hyp_out && T > 0) || !err_per_utt || !workspace)
        return fail(B200CTC_INVALID_ARGUMENT, "NULL pointer%s");
    if (workspace_bytes < B200CTC_ERROR_WORKSPACE_BYTES) return fail(B200CTC_WORKSPACE_TOO_SMALL, "workspace too small%s");
    if ((long long)T * E >= (1ll << 31)) return fail(B200CTC_UNSUPPORTED, "T*E too large%s");
    if (sizeof(int) * (4 * (size_t)Lmax + 3) > 200 * 1024) return fail(B200CTC_UNSUPPORTED, "target of %s%lld ids is too long", "", Lmax);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    int rc = check_cuda(cudaMemsetAsync(workspace, 0, sizeof(unsigned), stream), "counter reset");
    if (rc) return rc;
    return check_cuda(launch_greedy_error(argmax, input_lengths, B, T, labels, Lmax, blank, expansion, V, E, uint8_wrap ? 1 : 0,
                                          hyp_out, hyp_len, ref_len, distance, err_per_utt, err_mean,
                                          static_cast<unsigned *>(workspace), stream),
                      "greedy error kernel");
}

int b200ctc_edit_distance(const int32_t *ref, const int32_t *ref_len, int Rmax, const int32_t *hyp, const int32_t *hyp_len,
                          int Hmax, int B, int uint8_wrap, int32_t *distance, double *err_per_utt, double *err_mean,
                          void *workspace, size_t workspace_bytes, void *stream_) {
    if (B < 0 || Rmax < 0 || Hmax < 0) return fail(B200CTC_INVALID_ARGUMENT, "bad dimensions%s");
    if (B == 0) return B200CTC_OK;
    if ((!ref && Rmax > 0) || (!hyp && Hmax > 0) || !ref_len || !hyp_len || !err_per_utt || !workspace)
        return fail(B200CTC_INVALID_ARGUMENT, "NULL pointer%s");
    if (workspace_bytes < B200CTC_ERROR_WORKSPACE_BYTES) return fail(B200CTC_WORKSPACE_TOO_SMALL, "workspace too small%s");
    if (sizeof(int) * (4 * (size_t)Rmax + 3) > 200 * 1024) return fail(B200CTC_UNSUPPORTED, "reference of %s%lld ids is too long", "", Rmax);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    int rc = check_cuda(cudaMemsetAsync(workspace, 0, sizeof(unsigned), stream), "counter reset");
    if (rc) return rc;
    return check_cuda(launch_edit_distance(ref, ref_len, Rmax, hyp, hyp_len, Hmax, B, uint8_wrap ? 1 : 0, distance,
                                           err_per_utt, err_mean, static_cast<unsigned *>(workspace), stream),
                      "edit distance kernel");
}

}  // extern "C"
