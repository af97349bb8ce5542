// row_ring.cuh -- shared-memory ring of activation rows fed by the TMA engine.
//
// Both row-streaming kernels (softmax/gather and gradient) use the same structure: one CTA per SM,
// warp 0 is the producer, the other warps are consumers.
//   producer  draws frame tickets from a global counter (batches of kTicketBatch consecutive frames,
//             next batch prefetched); lane i of the producer warp owns frame i of the batch: the lanes
//             whose frame needs work are ranked by ballot, each claims the next ring slot in sequence
//             order, arms its mbarrier and issues a 1-D bulk async copy (cp.async.bulk, SASS UBLKCP) of
//             the whole V-float row -- several rows ahead of the consumers, so DRAM latency is covered by
//             the copy queue instead of by resident warps;
//   consumer  warp c handles row sequence numbers c, c+NC, c+2NC, ...: waits for the slot's "full"
//             barrier, works on the row out of shared memory, then releases the slot ("empty").
// Rows need only be 4-byte aligned (the reference's real vocabulary is 119 unigram ids + however many bigrams pass
// the count filter, asr/vocab.py:62-97 -- not a multiple of 4 in general): the producer copies the 16-byte aligned
// span that covers the row, RowMeta::off says where in the slot element 0 sits, and whoever stores a row back
// (gradient kernel) writes the unaligned ends with ordinary stores.  The span may reach up to 12 bytes in front of
// the first row and behind the last one: inside the allocation's own 256-byte granule, read only.
// Requirement (checked by the host dispatcher, which otherwise uses the plain LDG kernels): at least kMinSlots
// such spans fit in shared memory.
#pragma once
#include "common.cuh"
#include "kernels.h"

namespace b200ctc {

constexpr int kRingConsumers = 8;      // gradient kernel (the softmax/gather kernel runs kK1Consumers, softmax_gather.cu)
constexpr int kRingThreads = 32 * (1 + kRingConsumers);
constexpr int kTicketBatch = 8;       // frames per ticket; one producer lane per frame of the batch
constexpr int kMinSlots = 4;
constexpr int kMaxSlots = 16;
constexpr size_t kRingSmemBudget = 224 * 1024;

struct RowMeta {
    int b, t;
    int kind;      // 0: full work, 1: argmax only (padded frame), -1: stop
    unsigned seq;  // row sequence number currently occupying the slot (published before the barrier is armed)
    int off;       // the row's element 0 sits `off` floats into the slot (0..3: misalignment of the row in global memory)
    // per-row constants the producer fetches on the consumers' behalf (a dependent global load at the start of a
    // consumer's row is ~800 cycles during which the slot is held for nothing):
    int Lb;        // softmax/gather kernel: clamped label length of the utterance
    int pad_[3];
};

// bytes a slot needs for a row of V floats wherever it starts
__host__ __device__ inline size_t ring_row_bytes(int V) { return ((size_t)V * 4 + 12 + 15) & ~(size_t)15; }
#ifdef __CUDACC__
__device__ __forceinline__ int row_misalignment(const float *row) { return (int)((reinterpret_cast<uintptr_t>(row) >> 2) & 3); }
__device__ __forceinline__ uint32_t row_span_bytes(int off, int V) { return (uint32_t)(((off + V) * 4 + 15) & ~15); }
#endif

struct RingLayout {
    int consumers;         // active consumer warps = min(kRingConsumers, slots), see ring_acquire
    int batch;             // frames per ticket (<= slots)
    int slots;             // R
    size_t slot_bytes;     // row (+ per-row extras), multiple of 128
    size_t off_meta, off_full, off_empty, off_next, off_extra, total;
};

// smem_reserve: shared memory to leave free on the SM for a CTA of another kernel that is meant to run next to
// this one (the lattice kernel next to the softmax/gather kernel); 0 = none.
inline RingLayout make_ring(size_t slot_payload, size_t extra_bytes, size_t smem_reserve = 0, int consumers = kRingConsumers) {
    RingLayout r;
    r.slot_bytes = align_up(slot_payload, 128);
    const size_t fixed = (size_t)kMaxSlots * (sizeof(RowMeta) + 16) + extra_bytes + 256;
    long long budget = (long long)kRingSmemBudget;
    if (smem_reserve) {
        const long long room = 228 * 1024 - 2 * 1024 - (long long)smem_reserve;       // 1 KB per CTA is the driver's
        if (room < budget) budget = room;
    }
    long long n = (budget - (long long)fixed) / (long long)r.slot_bytes;
    if (n > kMaxSlots) n = kMaxSlots;
    r.slots = (int)(n < 0 ? 0 : n);
    r.batch = r.slots < kTicketBatch ? r.slots : kTicketBatch;
    r.consumers = r.slots < consumers ? r.slots : consumers;
    size_t o = r.slot_bytes * (size_t)r.slots;
    r.off_meta = o;  o += sizeof(RowMeta) * kMaxSlots;
    r.off_full = o;  o += 8 * kMaxSlots;
    r.off_empty = o; o += 8 * kMaxSlots;
    r.off_next = o;  o += 16;
    r.off_extra = align_up(o, 128);
    r.total = r.off_extra + extra_bytes;
    return r;
}

#ifdef __CUDACC__

struct Ring {
    unsigned char *base;
    RowMeta *meta;
    uint64_t *full, *empty;
    unsigned *next;        // next row sequence number to hand to a consumer
    int slots;
    int nc;                // active consumers (<= slots)
    int batch;             // frames per ticket = min(kTicketBatch, slots): a batch never waits on its own rows
    size_t slot_bytes;
    __device__ __forceinline__ unsigned char *slot(int s) const { return base + (size_t)s * slot_bytes; }
};

__device__ __forceinline__ Ring ring_setup(unsigned char *smem, const RingLayout &rl) {
    Ring r;
    r.base = smem;
    r.meta = reinterpret_cast<RowMeta *>(smem + rl.off_meta);
    r.full = reinterpret_cast<uint64_t *>(smem + rl.off_full);
    r.empty = reinterpret_cast<uint64_t *>(smem + rl.off_empty);
    r.next = reinterpret_cast<unsigned *>(smem + rl.off_next);
    r.slots = rl.slots;
    r.batch = rl.batch;
    r.nc = rl.consumers;
    r.slot_bytes = rl.slot_bytes;
    if (threadIdx.x == 0) {
        for (int i = 0; i < rl.slots; ++i) {
            mbar_init(&r.full[i], 1);
            mbar_init(&r.empty[i], 1);
            r.meta[i].seq = 0xffffffffu;
        }
        *r.next = 0u;
        mbar_init_fence();
    }
    __syncthreads();
    return r;
}

// Producer side: claim the slot for row sequence number q (waits until its previous occupant was released).
__device__ __forceinline__ int ring_claim(const Ring &r, unsigned q) {
    const int s = (int)(q % (unsigned)r.slots);
    const unsigned n = q / (unsigned)r.slots;
    if (n > 0) mbar_wait(&r.empty[s], (n - 1) & 1u);
    return s;
}

// Consumer side (whole warp): take the next row, whichever it is.  Rows are NOT dealt out round-robin: a row that has
// landed would then wait for "its" consumer while others idle -- at 66 % consumer utilisation that wait was as long
// as the processing itself and kept a third of the ring's slots out of flight (measured per warp, DESIGN.md §3).
__device__ __forceinline__ unsigned ring_next_row(const Ring &r, int lane) {
    unsigned q = 0;
    if (lane == 0) q = atomicAdd(r.next, 1u);
    return __shfl_sync(0xffffffffu, q, 0);
}

// Producer side, non-blocking: is the slot of row sequence number q free (its previous occupant released)?
__device__ __forceinline__ bool ring_slot_free(const Ring &r, unsigned q) {
    const int s = (int)(q % (unsigned)r.slots);
    const unsigned n = q / (unsigned)r.slots;
    return n == 0 || mbar_test_wait(&r.empty[s], (n - 1) & 1u);
}

// Consumer side: wait until row sequence number q has landed in its slot; returns the slot.
// An mbarrier parity wait can only tell "this phase" from "the one before", while rows complete out of order
// (a batch is issued by several lanes at once, each row is several bulk copies): a fast consumer may get here
// while the slot still belongs to an earlier row, and the parity of its own row would then alias to an older,
// already completed phase.  So the producer publishes the sequence number it is about to load into the slot
// (RowMeta::seq, written before it arms the barrier) and the consumer first waits to see ITS number there: from
// then on the barrier is in this row's phase and the parity wait is exact, whatever the skew between warps.
__device__ __forceinline__ int ring_acquire(const Ring &r, unsigned q) {
    const int s = (int)(q % (unsigned)r.slots);
    const unsigned n = q / (unsigned)r.slots;
    const volatile unsigned *seq = &r.meta[s].seq;
    while (*seq != q) __nanosleep(32);
    mbar_wait(&r.full[s], n & 1u);
    return s;
}

// Producer side: announce that slot s now belongs to row q (after the other RowMeta fields, before arming).
__device__ __forceinline__ void ring_publish(const Ring &r, int s, unsigned q) {
    __threadfence_block();
    *reinterpret_cast<volatile unsigned *>(&r.meta[s].seq) = q;
}

// Producer side (whole warp): tell every consumer to stop -- one stop record per consumer, in sequence order.
// Issued by lane 0 one after the other: the ring may have fewer slots than consumers, in which case a stop
// record can only be placed once an earlier one has been picked up (consumers release stop slots too).
__device__ __forceinline__ void ring_stop(const Ring &r, unsigned q, int lane) {
    if (lane == 0) {
        for (int c = 0; c < r.nc; ++c) {
            const int s = ring_claim(r, q + (unsigned)c);
            r.meta[s].kind = -1;
            ring_publish(r, s, q + (unsigned)c);
            mbar_arrive(&r.full[s]);
        }
    }
    __syncwarp();
}

#endif  // __CUDACC__

}  // namespace b200ctc
