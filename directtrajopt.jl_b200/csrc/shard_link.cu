// Knot-range shards of one long trajectory (SURVEY.md section 8e, partitioning B): the cross-rank traffic of an
// evaluation, all of it through peer memory (NVLink P2P stores into windows mapped with CUDA IPC), no collective library
// on the path:
//   * the one-knot halo: after uploading iterate e a shard PUSHES its first knot into the left neighbour's exchange
//     window (slot e & 1) and then publishes e there; the left neighbour's first kernel of iterate e waits for that flag.
//     Flow control is an acknowledgement the reader writes back into the pusher's window when it moves on to its next
//     iterate, so a fast rank can run at most one iterate ahead of the neighbour that still reads its knot.
//   * the two scalars every rank needs (objective: sum, constraint violation: max): one kernel writes {J, viol, seq} into
//     this rank's slot of EVERY peer's window and spins until all slots of its own window carry seq; the sum runs in
//     rank order on every rank (bit-identical results everywhere).
//   * the boundary Hessian block (time-dependent bilinear integrators with a linear control spline, whose interval k
//     reads u_{k+1}): interval k0 - 1 belongs to the left neighbour but adds to the (u, u) entries of knot k0 and to the
//     whole (knot k0 - 1, knot k0) cross block, which the right shard assembles.  Every Hessian evaluation the left
//     neighbour PUSHES the compact second-derivative row(s) of its last interval -- computed anyway, identical bits to the
//     unsharded evaluation -- into slot seq & 1 of the right neighbour's window and publishes seq (hs_push_kernel); the
//     right shard waits for seq right before it assembles its first knot, copies the block into the leading row of its
//     scratch and acknowledges (hs_receive_kernel).  seq counts Hessian evaluations since the link, so a linked shard's
//     Hessian evaluation s reads what its left neighbour's evaluation s produced: every rank evaluates every Hessian.
// A wait that sees no progress for kTimeoutNs sets XWin::err and gives up (reported by the host as DTO_ERR_CUDA).
#include "dto_internal.h"
#include <algorithm>
#include <cstdint>

namespace {

constexpr unsigned long long kTimeoutNs = 20ull * 1000ull * 1000ull * 1000ull;

__device__ __forceinline__ unsigned long long now_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// spin until *flag >= want; false on timeout
__device__ __forceinline__ bool wait_geq(const volatile unsigned long long* flag, unsigned long long want) {
    const unsigned long long t0 = now_ns();
    while (*flag < want) {
        if (now_ns() - t0 > kTimeoutNs) return false;
        __nanosleep(200);
    }
    return true;
}

// One kernel per new iterate: (a) copy the iterate into the resident buffer (dst != src: dto_upload_dev), all CTAs;
// (b) warp 0 of CTA 0: acknowledge the right neighbour's previous knot, push this shard's first knot to the left neighbour
// and publish the epoch; (c) wait_right: stay until the right neighbour's knot of this epoch has landed (shards linked across
// processes: the evaluation kernels that follow read it; one launch instead of copy + publish + wait).
__global__ void __launch_bounds__(256) shard_publish_kernel(XWin* own, XWin* left, XWin* right, double* __restrict__ dst,
                                                            const double* __restrict__ src, long long n, int vec2, int z,
                                                            unsigned long long epoch, int wait_right) {
    const bool proto = blockIdx.x == 0 && threadIdx.x < 32;
    const int lane = threadIdx.x;
    bool ok = true;
    if (proto) {
        if (right != nullptr && lane == 0) {  // everything of iterate epoch - 1 on this stream is done: its halo slot may be reused
            *(volatile unsigned long long*)&right->ack = epoch - 1;
            __threadfence_system();
        }
        if (left != nullptr) {
            if (lane == 0 && epoch >= 2) ok = wait_geq(&own->ack, epoch - 2);  // the reader left iterate epoch - 2 (same slot) behind
            ok = __shfl_sync(0xffffffffu, ok ? 1 : 0, 0) != 0;
            if (!ok) {
                if (lane == 0) own->err = 1;
            } else {
                double* slot = left->halo + (size_t)(epoch & 1) * z;
                for (int i = lane; i < z; i += 32) slot[i] = src[i];
                __threadfence_system();
                __syncwarp();
                if (lane == 0) {
                    *(volatile unsigned long long*)&left->halo_epoch = epoch;
                    __threadfence_system();
                }
            }
        }
    }
    if (dst != src) {
        const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x, nt = (long long)gridDim.x * blockDim.x;
        if (vec2) {
            const double2* s2 = reinterpret_cast<const double2*>(src);
            double2* d2 = reinterpret_cast<double2*>(dst);
            const long long n2 = n >> 1;
            for (long long e = t; e < n2; e += nt) d2[e] = s2[e];
            if (t == 0 && (n & 1)) dst[n - 1] = src[n - 1];
        } else {
            for (long long e = t; e < n; e += nt) dst[e] = src[e];
        }
    }
    if (proto && wait_right && right != nullptr && ok && lane == 0) {
        if (!wait_geq(&own->halo_epoch, epoch)) own->err = 2;
        __threadfence_system();
    }
}

__global__ void shard_wait_kernel(XWin* own, unsigned long long epoch) {
    if (!wait_geq(&own->halo_epoch, epoch)) own->err = 2;
    __threadfence_system();
}

// Hessian evaluation `seq`, pushing side (enqueued after the interval kernel that wrote the last local interval's rows):
// wait until the right neighbour has copied block seq - 2 (same slot) out, store this evaluation's rows into slot seq & 1
// of its window, then publish seq.
__global__ void __launch_bounds__(256) hs_push_kernel(XWin* own, XWin* right, HsRows rows, int z, long long hblk_len,
                                                      unsigned long long seq) {
    __shared__ int ok;
    if (threadIdx.x == 0) {
        ok = seq < 3 || wait_geq(&own->hs_ack, seq - 2);
        if (!ok) own->err = 4;
    }
    __syncthreads();
    if (!ok) return;
    double* slot = xwin_hblk(right, z) + (size_t)(seq & 1) * hblk_len;
    for (int r = 0; r < rows.n; ++r) {
        for (int e = threadIdx.x; e < rows.len[r]; e += blockDim.x) slot[e] = rows.row[r][e];
        slot += rows.len[r];
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        *(volatile unsigned long long*)&right->hs_seq = seq;
        __threadfence_system();
    }
}

// Hessian evaluation `seq`, receiving side (enqueued before the assembler launch of local knot 0): wait for the left
// neighbour's block of seq, copy it into the local rows, acknowledge it in the left neighbour's window.
__global__ void __launch_bounds__(256) hs_receive_kernel(XWin* own, XWin* left, HsRows rows, int z, long long hblk_len,
                                                         unsigned long long seq) {
    __shared__ int ok;
    if (threadIdx.x == 0) {
        ok = wait_geq(&own->hs_seq, seq);
        if (!ok) own->err = 5;
        __threadfence_system();
    }
    __syncthreads();
    if (!ok) return;
    const volatile double* slot = xwin_hblk(own, z) + (size_t)(seq & 1) * hblk_len;
    for (int r = 0; r < rows.n; ++r) {
        for (int e = threadIdx.x; e < rows.len[r]; e += blockDim.x) rows.row[r][e] = slot[e];
        slot += rows.len[r];
    }
    __syncthreads();  // every read of the slot is done before the slot is released
    if (threadIdx.x == 0) {
        __threadfence_system();
        *(volatile unsigned long long*)&left->hs_ack = seq;
        __threadfence_system();
    }
}

// store {J, viol, seq} into this rank's slot of every peer's window, wait for everybody's, reduce in rank order (one warp)
__device__ void exchange_scalars(XWin* own, XWin* const* __restrict__ peers, int rank, int world, unsigned long long seq, double myJ,
                                 double myV, double* __restrict__ J, double* __restrict__ viol) {
    const int lane = threadIdx.x & 31;
    const int par = (int)(seq & 1);
    if (lane < world) {
        volatile double* s = peers[lane]->scal[par][rank];
        s[0] = myJ;
        s[1] = myV;
        __threadfence_system();
        *(volatile unsigned long long*)&s[2] = seq;  // the tag goes last
        __threadfence_system();
    }
    bool ok = true;
    if (lane < world) ok = wait_geq((const volatile unsigned long long*)&own->scal[par][lane][2], seq);
    ok = __all_sync(0xffffffffu, ok);
    if (!ok) {
        if (lane == 0) own->err = 3;
        return;
    }
    __threadfence_system();
    if (lane == 0) {
        double sum = 0.0, mx = 0.0;
        for (int r = 0; r < world; ++r) {  // rank order on every rank: identical bits everywhere
            sum += ((volatile double*)own->scal[par][r])[0];
            mx = nan_max(mx, ((volatile double*)own->scal[par][r])[1]);
        }
        *J = sum;
        *viol = mx;
    }
}

__global__ void scalar_exchange_kernel(XWin* own, XWin* const* __restrict__ peers, int rank, int world, unsigned long long seq,
                                       double* __restrict__ J, double* __restrict__ viol) {
    exchange_scalars(own, peers, rank, world, seq, *J, *viol, J, viol);
}

// The shard's constraint violation (max(|g_eq|, max(0, g_ineq)) over its rows) AND the exchange in one launch: every CTA
// reduces its rows into scratch[0] (non-negative doubles order like their bit patterns, NaN above +inf); the CTA that arrives last at
// scratch[1] owns the complete maximum, exchanges {J, viol} with the peers and leaves the scratch words zeroed for the next call.
__global__ void __launch_bounds__(256) shard_scalars_kernel(XWin* own, XWin* const* __restrict__ peers, int rank, int world,
                                                            unsigned long long seq, long long n_cons, const double* __restrict__ g,
                                                            const int* __restrict__ row_is_eq, unsigned long long* __restrict__ scratch,
                                                            double* __restrict__ J, double* __restrict__ viol) {
    __shared__ double red[8];
    __shared__ int is_last;
    double m = 0.0;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < n_cons; r += (long long)gridDim.x * blockDim.x) {
        const double v = g[r];
        m = nan_max(m, row_is_eq[r] ? fabs(v) : nan_max(0.0, v));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = nan_max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = nan_max(m, red[w]);
        atomicMax(&scratch[0], (unsigned long long)__double_as_longlong(m));
        __threadfence();
        is_last = atomicAdd(&scratch[1], 1ull) == (unsigned long long)gridDim.x - 1;
    }
    __syncthreads();
    if (!is_last || threadIdx.x >= 32) return;
    __threadfence();
    double myV = 0.0;
    if (threadIdx.x == 0) {
        myV = __longlong_as_double((long long)atomicExch(&scratch[0], 0ull));
        scratch[1] = 0ull;
    }
    myV = __shfl_sync(0xffffffffu, myV, 0);
    exchange_scalars(own, peers, rank, world, seq, *J, myV, J, viol);
}

}  // namespace

void launch_shard_publish(XWin* own, XWin* left, XWin* right, double* dst, const double* src, long long n, int z,
                          unsigned long long epoch, bool wait_right, cudaStream_t st, long long* launches) {
    const bool vec2 = (((uintptr_t)dst | (uintptr_t)src) & 15) == 0;
    // a copy of n doubles at ~16 KB per CTA; in place: the protocol warp alone
    const unsigned grid = dst == src ? 1u : (unsigned)std::min<long long>(std::max<long long>(n / 2048, 1), 1184);
    shard_publish_kernel<<<grid, dst == src ? 32 : 256, 0, st>>>(own, left, right, dst, src, n, vec2 ? 1 : 0, z, epoch, wait_right ? 1 : 0);
    ++*launches;
}

void launch_shard_wait(XWin* own, unsigned long long epoch, cudaStream_t st, long long* launches) {
    shard_wait_kernel<<<1, 1, 0, st>>>(own, epoch);
    ++*launches;
}

void launch_hs_push(XWin* own, XWin* right, const HsRows& rows, int z, long long hblk_len, unsigned long long seq, cudaStream_t st,
                    long long* launches) {
    hs_push_kernel<<<1, 256, 0, st>>>(own, right, rows, z, hblk_len, seq);
    ++*launches;
}

void launch_hs_receive(XWin* own, XWin* left, const HsRows& rows, int z, long long hblk_len, unsigned long long seq, cudaStream_t st,
                       long long* launches) {
    hs_receive_kernel<<<1, 256, 0, st>>>(own, left, rows, z, hblk_len, seq);
    ++*launches;
}

void launch_scalar_exchange(XWin* own, XWin* const* peers, int rank, int world, unsigned long long seq, double* J, double* viol,
                            cudaStream_t st, long long* launches) {
    scalar_exchange_kernel<<<1, 32, 0, st>>>(own, peers, rank, world, seq, J, viol);
    ++*launches;
}

void launch_shard_scalars(XWin* own, XWin* const* peers, int rank, int world, unsigned long long seq, long long n_cons, const double* g,
                          const int* row_is_eq, unsigned long long* scratch, double* J, double* viol, cudaStream_t st, long long* launches) {
    const unsigned grid = (unsigned)std::min<long long>(std::max<long long>((n_cons + 2047) / 2048, 1), 592);
    shard_scalars_kernel<<<grid, 256, 0, st>>>(own, peers, rank, world, seq, n_cons, g, row_is_eq, scratch, J, viol);
    ++*launches;
}
