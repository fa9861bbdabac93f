// One-shot all-reduce of the `red` partials over NVLink / NVSwitch PEER MEMORY (SURVEY.md section 8e: the path's only exchange step).
//
// Every rank keeps its contribution `red` ([E (Kp x mld) | sum r^2 | Phi^T Phi | d omega], 129 KB at K = 27, m = 1000) in a buffer that
// all ranks of the node have mapped (CUDA VMM / fabric handles; torch.distributed._symmetric_memory does the rendezvous).  After the
// fused pass, instead of two NCCL calls (20-30 us of launch + protocol latency each, at a 0.4 - 3.5 ms step), each rank
//   1. signals "my red of epoch e is ready" by a release-store into every peer's flag pad                 (peer_signal_kernel)
//   2. waits until every peer has signalled e, then reads all ranks' buffers directly through NVLink and adds them in RANK ORDER
//      (every rank forms bit-identical sums: the replicated parameters stay bit-identical across ranks), and finally tells every peer
//      that it has consumed their buffer                                                                   (peer_gather_kernel)
//   3. at the start of the next step waits until every peer has consumed epoch e before its fused pass overwrites `red`
//                                                                                                          (peer_wait_consumed_kernel)
// Flags are monotonically increasing epochs (never reset), so CUDA-graph replays need no host involvement.  All spins carry a watchdog.
#include "common.cuh"

namespace desmo {

struct PeerArgs {
    int world, rank;
    const unsigned long long* red_ptrs;   // [world] peer-mapped address of every rank's red
    const unsigned long long* flag_ptrs;  // [world] peer-mapped address of every rank's flag pad: uint32 ready[world], consumed[world]
    unsigned* state;                      // local: [0] epoch of the last signalled step, [1] CTA completion counter of the gather
    float* out;
    long long count4;                     // float4 elements
};

__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ float4 ld_volatile_f4(const float4* p) {
    float4 v;
    asm volatile("ld.volatile.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
// spins until *flag >= target; a peer that never arrives (crashed rank) fails the launch after ~10 s instead of hanging the GPU
__device__ __forceinline__ void wait_flag(const unsigned* flag, unsigned target) {
    const unsigned long long t0 = globaltimer_ns();
    while ((int)(ld_acquire_sys(flag) - target) < 0) {
        __nanosleep(200);
        if (globaltimer_ns() - t0 > 10000000000ull) __trap();
    }
}

__global__ void peer_wait_consumed_kernel(const PeerArgs a) {
    const int q = threadIdx.x;
    if (q < a.world) {
        const unsigned e = a.state[0];
        const unsigned* mine = reinterpret_cast<const unsigned*>(a.flag_ptrs[a.rank]);
        wait_flag(mine + a.world + q, e);
    }
}

__global__ void peer_signal_kernel(const PeerArgs a) {
    const int q = threadIdx.x;
    const unsigned e = a.state[0] + 1;
    __threadfence_system();  // the red written by the preceding kernels of this stream is visible system-wide before the flag is
    __syncwarp();
    if (q < a.world) st_release_sys(reinterpret_cast<unsigned*>(a.flag_ptrs[q]) + a.rank, e);
    __syncwarp();
    if (q == 0) a.state[0] = e;
}

__global__ void __launch_bounds__(256) peer_gather_kernel(const PeerArgs a) {
    __shared__ unsigned e_s;
    __shared__ bool last_s;
    if (threadIdx.x == 0) e_s = a.state[0];
    __syncthreads();
    const unsigned e = e_s;
    if (threadIdx.x < a.world) wait_flag(reinterpret_cast<const unsigned*>(a.flag_ptrs[a.rank]) + threadIdx.x, e);
    __syncthreads();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.count4; i += (long long)gridDim.x * blockDim.x) {
        float4 s = ld_volatile_f4(reinterpret_cast<const float4*>(a.red_ptrs[0]) + i);
        for (int q = 1; q < a.world; ++q) {  // rank order: the same sum, bit for bit, on every rank
            const float4 v = ld_volatile_f4(reinterpret_cast<const float4*>(a.red_ptrs[q]) + i);
            s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
        }
        reinterpret_cast<float4*>(a.out)[i] = s;
    }
    // the last CTA to finish tells every peer that this rank no longer reads their buffer
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned prev = atomicAdd(a.state + 1, 1u);
        last_s = (prev == gridDim.x - 1);
        if (last_s) a.state[1] = 0;
    }
    __syncthreads();
    if (last_s && threadIdx.x < a.world) st_release_sys(reinterpret_cast<unsigned*>(a.flag_ptrs[threadIdx.x]) + a.world + a.rank, e);
}

static int peer_args(const desmo_peer* p, PeerArgs* a) {
    if (!p || p->world < 2 || p->world > DESMO_MAX_PEERS || p->rank < 0 || p->rank >= p->world || !p->red_ptrs || !p->flag_ptrs || !p->state) {
        set_error("desmo_peer: invalid descriptor (2 <= world <= %d, device tables and state required)", DESMO_MAX_PEERS);
        return DESMO_ERR_ARG;
    }
    a->world = p->world; a->rank = p->rank;
    a->red_ptrs = reinterpret_cast<const unsigned long long*>(p->red_ptrs);
    a->flag_ptrs = reinterpret_cast<const unsigned long long*>(p->flag_ptrs);
    a->state = p->state;
    a->out = nullptr; a->count4 = 0;
    return DESMO_OK;
}

}  // namespace desmo

using namespace desmo;

extern "C" int desmo_peer_begin_step(const desmo_peer* p, void* stream) {
    PeerArgs a;
    if (int rc = peer_args(p, &a)) return rc;
    peer_wait_consumed_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(a);
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}

extern "C" int desmo_peer_allreduce(const desmo_peer* p, int64_t count, float* red_sum, void* stream) {
    PeerArgs a;
    if (int rc = peer_args(p, &a)) return rc;
    if (!red_sum || count <= 0 || count % 4 != 0) { set_error("desmo_peer_allreduce: count must be a positive multiple of 4"); return DESMO_ERR_ARG; }
    a.out = red_sum;
    a.count4 = count / 4;
    cudaStream_t st = (cudaStream_t)stream;
    peer_signal_kernel<<<1, 32, 0, st>>>(a);
    const int grid = (int)((a.count4 + 255) / 256 < 64 ? (a.count4 + 255) / 256 : 64);
    peer_gather_kernel<<<grid, 256, 0, st>>>(a);
    DESMO_CUDA(cudaGetLastError());
    return DESMO_OK;
}
