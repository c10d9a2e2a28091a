// One-shot all-reduce of a few doubles over NVLink / NVSwitch peer memory -- the only exchange the frame-sharded
// SOT loss has (sum of the per-rank loss sums and frame counts, SURVEY.md 8e).  It sits between the forward and
// the backward launch of a ~0.75 ms step, so its latency is what multi-GPU scaling loses; a tiny kernel that
// stores into every peer's mailbox and spins on its own costs a few microseconds where an NCCL all-reduce
// (launch + protocol) costs tens.
//
// The stores can also be made by the SOT launch itself (its last CTA, `finish_mean` in sot_kernels.cuh: the compute
// kernel starts the exchange the moment its sum is complete) and collected by the wait-only form of this kernel.
//
// Mailbox (one per rank, symmetric allocation, peers mapped): [world][8 phases][kMaxVals + 1] doubles; entry
// [r][ph][kMaxVals] is the sequence number rank r wrote last into phase ph.  Call number `seq` (1, 2, ...) uses
// phase seq & 7.  When one kernel posts and collects (in stream), a rank can only start call seq + 2 after every
// peer has written call seq + 1, i.e. after every peer has finished reading call seq: two phases would do.  When
// the SOT launch posts and a side stream collects, the caller lets a rank post call s only after it has COLLECTED
// call s - 4 (`sharding.MeanExchange`: the ranks may drift four steps apart): then every peer has posted s - 4,
// hence collected s - 8 -- the slot that call s overwrites.  Eight phases.
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdlib>

#include "../../include/sot_b200.h"
#include "sot_internal.cuh"

namespace sot {

constexpr int kP2PMaxWorld = 16;
constexpr int kP2PMaxVals = 8;
constexpr int kP2PSlot = kP2PMaxVals + 1;  // doubles per (rank, phase)
constexpr int kP2PPhases = 8;

struct P2PArgs {
    double* mailbox[kP2PMaxWorld];  // mailbox[r] = rank r's mailbox as mapped into this process
    const double* in;
    double* out;
    // global-mean form (the sharded loss): values = (*in, local_count); results mean_out = sum / count and
    // inv_count_out = 1 / count as floats, ready for the caller -- no scalar-sized torch kernels around the exchange
    double local_count;
    float* mean_out;
    float* inv_count_out;
    int count, world, rank;
    unsigned long long seq;
    unsigned long long timeout_ns;
    // wait-only form: the stores into the peers' mailboxes were made by the last CTA of the SOT launch
    // (sot_kernels.cuh: finish_mean); this kernel only collects.  expected_count > 0: the counts must add up to it.
    int post;
    unsigned long long* seq_dev;  // nullable: call number = *seq_dev + 1, stored back at the end (graph replay)
    double expected_count;
    int* status;  // nullable: 1 = count mismatch, 2 = a peer never arrived
};

__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__global__ void __launch_bounds__(32) sot_p2p_allreduce_kernel(const P2PArgs a) {
    const int t = threadIdx.x;
    const unsigned long long seq = a.seq_dev != nullptr ? *a.seq_dev + 1ULL : a.seq;
    const int phase = static_cast<int>(seq & (kP2PPhases - 1));
    const double seq_val = static_cast<double>(seq);
    __shared__ int failed;
    if (t == 0) failed = 0;
    __syncwarp();
    if (t < a.world) {
        if (a.post) {
            // my values, then my sequence number, into slot [rank][phase] of peer t's mailbox
            double* dst = a.mailbox[t] + (static_cast<long long>(a.rank) * kP2PPhases + phase) * kP2PSlot;
            for (int i = 0; i < a.count; ++i) {
                const double v = (a.mean_out != nullptr && i == 1) ? a.local_count : a.in[i];
                asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(dst + i), "d"(v) : "memory");
            }
            __threadfence_system();
            asm volatile("st.release.sys.global.f64 [%0], %1;" ::"l"(dst + kP2PMaxVals), "d"(seq_val) : "memory");
        }
        // wait for rank t's contribution in my own mailbox
        const double* src = a.mailbox[a.rank] + (static_cast<long long>(t) * kP2PPhases + phase) * kP2PSlot;
        const unsigned long long t0 = global_ns();
        double seen;
        do {
            asm volatile("ld.acquire.sys.global.f64 %0, [%1];" : "=d"(seen) : "l"(src + kP2PMaxVals) : "memory");
            if (seen != seq_val && global_ns() - t0 > a.timeout_ns) {
                failed = 1;
                break;
            }
        } while (seen != seq_val);
    }
    __syncwarp();
    if (failed) {
        // A peer never arrived (timeout on NCCL's watchdog scale, minutes): fail LOUDLY -- the status word is
        // set for the host and the kernel traps, so the next CUDA call on this context returns an error
        // (a silent NaN would be all-reduced into every replica's weights by DDP).
        if (t == 0 && a.status != nullptr) {
            *a.status = 2;
            __threadfence_system();
        }
        __syncwarp();
        __trap();
    }
    if (t < a.count) {
        double s = 0.0;
        for (int r = 0; r < a.world; ++r) {  // fixed order: every rank gets the same bits
            double v;
            asm volatile("ld.relaxed.sys.global.f64 %0, [%1];"
                         : "=d"(v)
                         : "l"(a.mailbox[a.rank] + (static_cast<long long>(r) * kP2PPhases + phase) * kP2PSlot + t)
                         : "memory");
            s += v;
        }
        if (a.seq_dev != nullptr && t == 0) *a.seq_dev = seq;  // (every lane read the old value before the spin)
        if (a.out != nullptr) a.out[t] = s;
        if (a.mean_out != nullptr) {  // t = 0 holds the sum, t = 1 the count
            const double cnt = __shfl_sync((1u << a.count) - 1u, s, 1);
            if (t == 0) {
                const bool count_ok = !(a.expected_count > 0.0) || cnt == a.expected_count;
                *a.mean_out = count_ok ? static_cast<float>(s / cnt) : __int_as_float(0x7fc00000);
                if (a.inv_count_out != nullptr) *a.inv_count_out = static_cast<float>(1.0 / cnt);
                if (!count_ok && a.status != nullptr) *a.status = 1;
            }
        }
    }
}

}  // namespace sot

extern "C" {

int sot_p2p_mailbox_doubles(int32_t world) { return world * sot::kP2PPhases * sot::kP2PSlot; }

static int p2p_launch(sot::P2PArgs& a, void* const* mailboxes, int32_t world, int32_t rank, uint64_t seq, void* stream);

int sot_p2p_global_mean_device(const double* local_sum, double local_count, float* mean_out, float* inv_count_out,
                               void* const* mailboxes, int32_t world, int32_t rank, uint64_t seq, void* stream) {
    if (local_sum == nullptr || mean_out == nullptr || inv_count_out == nullptr || mailboxes == nullptr)
        return sot::fail(SOT_EINVAL, "sot_p2p_global_mean_device: NULL pointer");
    sot::P2PArgs a{};
    a.in = local_sum;
    a.local_count = local_count;
    a.mean_out = mean_out;
    a.inv_count_out = inv_count_out;
    a.count = 2;
    a.post = 1;
    return p2p_launch(a, mailboxes, world, rank, seq, stream);
}

int sot_p2p_wait_mean_device(float* mean_out, double expected_count, int32_t* status, void* const* mailboxes,
                             int32_t world, int32_t rank, uint64_t seq, uint64_t* seq_device, uint32_t timeout_ms,
                             void* stream) {
    if (mean_out == nullptr || mailboxes == nullptr)
        return sot::fail(SOT_EINVAL, "sot_p2p_wait_mean_device: NULL pointer");
    sot::P2PArgs a{};
    a.mean_out = mean_out;
    a.count = 2;
    a.post = 0;
    a.expected_count = expected_count;
    a.status = status;
    a.seq_dev = reinterpret_cast<unsigned long long*>(seq_device);
    if (seq_device != nullptr && seq == 0) seq = 1;  // (argument check below; the device value is what counts)
    if (timeout_ms > 0) a.timeout_ns = 1000000ULL * timeout_ms;
    return p2p_launch(a, mailboxes, world, rank, seq, stream);
}

int sot_p2p_allreduce_device(const double* in, double* out, int32_t count, void* const* mailboxes, int32_t world,
                             int32_t rank, uint64_t seq, void* stream) {
    if (in == nullptr || out == nullptr || mailboxes == nullptr)
        return sot::fail(SOT_EINVAL, "sot_p2p_allreduce_device: NULL pointer");
    if (count < 1 || count > sot::kP2PMaxVals)
        return sot::fail(SOT_EINVAL, "sot_p2p_allreduce_device: bad count");
    sot::P2PArgs a{};
    a.in = in;
    a.out = out;
    a.count = count;
    a.post = 1;
    return p2p_launch(a, mailboxes, world, rank, seq, stream);
}

static int p2p_launch(sot::P2PArgs& a, void* const* mailboxes, int32_t world, int32_t rank, uint64_t seq, void* stream) {
    const int32_t count = a.count;
    if (count < 1 || count > sot::kP2PMaxVals || world < 1 || world > sot::kP2PMaxWorld || rank < 0 || rank >= world ||
        seq == 0)
        return sot::fail(SOT_EINVAL, "sot_p2p_allreduce_device: bad count / world / rank / seq");
    for (int r = 0; r < world; ++r) {
        if (mailboxes[r] == nullptr) return sot::fail(SOT_EINVAL, "sot_p2p_allreduce_device: NULL mailbox");
        a.mailbox[r] = static_cast<double*>(mailboxes[r]);
    }
    a.world = world;
    a.rank = rank;
    a.seq = seq;
    if (a.timeout_ns == 0) {  // a late peer is normal (checkpointing, evaluation, a data-loader stall on one rank):
        unsigned long long ms = 600000ULL;  // wait on NCCL's watchdog scale, 10 minutes, unless told otherwise
        if (const char* env = getenv("SOT_P2P_TIMEOUT_MS")) {
            const long long v = atoll(env);
            if (v > 0) ms = static_cast<unsigned long long>(v);
        }
        a.timeout_ns = 1000000ULL * ms;
    }
    sot::sot_p2p_allreduce_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(a);
    return sot::launched(cudaGetLastError(), "sot_p2p_allreduce_kernel");
}

}  // extern "C"
