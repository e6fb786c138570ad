// Micro-benchmark: the hand-off of the fused gated MLP (ll2_kernel.cu) -- an all-gather of one K-slice of act (448 bf16 =
// 56 pieces of 16 bytes, the 8 act values of one w13 tile each) among the 16 CTAs of a thread-block cluster.  CTA r owns
// pieces [56 r / 16, 56 (r + 1) / 16) (3-4, one warp each, as in the kernel) and sends each to all 16 CTAs.  Two forms:
//   A  st.async.shared::cluster ... mbarrier::complete_tx into the peer, the receiver waits on its own mbarrier
//      (expect_tx of 896 bytes per round; two buffers + two barriers alternate by round parity);
//   B  st.shared::cluster into the peer, then barrier.cluster.arrive.release + wait.acquire (two buffers).
// Every round depends on the previous one (the pieces a CTA sends are a function of everything it received), so the time
// per round is the latency of one hand-off + a few instructions.  7 clusters run side by side, as in the kernel.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/micro/dsmem_allgather tools/micro/dsmem_allgather.cu
#include <cstdio>
#include <cuda_runtime.h>
#include <stdint.h>

constexpr int kC = 16, kPieces = 56, kThreads = 256;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t mapa(uint32_t a, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t n) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(n) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok = 0;
    for (uint32_t n = 0; !ok && n < (1u << 26); ++n)   // a lost hand-off shows up as disagreeing CTAs, not as a hang
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void st_async_v4(uint32_t a, uint4 v, uint32_t bar) {
    asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1,%2,%3,%4}, [%5];"
                 ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(bar) : "memory");
}
__device__ __forceinline__ void st_cluster_v4(uint32_t a, uint4 v) {
    asm volatile("st.shared::cluster.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cta_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }

template <int kForm>
__global__ void __launch_bounds__(kThreads, 1) allgather(int rounds, unsigned long long* ns_out, uint32_t* check) {
    __shared__ __align__(16) uint4 buf[2][kPieces];
    __shared__ __align__(8) uint64_t bar[2];
    __shared__ uint32_t seed;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t r = cta_rank();
    if (tid == 0) {
        mbar_init(smem_u32(&bar[0]), 1); mbar_init(smem_u32(&bar[1]), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        seed = r + 1;
    }
    cluster_sync_all();
    const int p0 = kPieces * r / kC, p1 = kPieces * (r + 1) / kC;
    unsigned long long t0 = 0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    uint32_t par[2] = {0u, 0u};
    for (int it = 0; it < rounds; ++it) {
        const int b = it & 1;
        const uint32_t bb = smem_u32(&bar[b]);
        if (kForm == 0 && tid == 0) mbar_expect_tx(bb, kPieces * 16);
        const int p = p0 + warp;
        if (p < p1 && lane < kC) {
            const uint32_t s = seed;
            const uint4 v = make_uint4(s + p, s ^ p, s * 3u + p, (uint32_t)it);
            const uint32_t dst = mapa(smem_u32(&buf[b][p]), (uint32_t)lane);
            if (kForm == 0) st_async_v4(dst, v, mapa(bb, (uint32_t)lane));
            else st_cluster_v4(dst, v);
        }
        if (kForm == 0) { mbar_wait(bb, par[b]); par[b] ^= 1u; }
        else cluster_sync_all();
        __syncthreads();   // every thread has seen the round before seed changes
        if (warp == 0) {   // the next round's pieces depend on all of this round's
            uint32_t acc = 0;
            for (int i = lane; i < kPieces; i += 32) acc += buf[b][i].x ^ buf[b][i].w;
            for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
            if (lane == 0) seed = acc;
        }
        __syncthreads();
    }
    unsigned long long t1 = 0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    if (tid == 0) { ns_out[blockIdx.x] = t1 - t0; check[blockIdx.x] = seed; }
    cluster_sync_all();   // no CTA leaves while a peer may still write into it
}

template <int kForm>
static double run(int clusters, int rounds, unsigned long long* d_ns, uint32_t* d_chk) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(clusters * kC);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = 200 * 1024;   // one CTA per SM, as in the decode kernel
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = kC; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, allgather<kForm>, rounds, d_ns, d_chk);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("launch failed: %s\n", cudaGetErrorString(e)); return -1.0; }
    unsigned long long ns[8 * kC];
    uint32_t chk[8 * kC];
    cudaMemcpy(ns, d_ns, sizeof(unsigned long long) * clusters * kC, cudaMemcpyDeviceToHost);
    cudaMemcpy(chk, d_chk, sizeof(uint32_t) * clusters * kC, cudaMemcpyDeviceToHost);
    unsigned long long mx = 0;
    for (int i = 0; i < clusters * kC; ++i) mx = ns[i] > mx ? ns[i] : mx;
    for (int c = 0; c < clusters; ++c)
        for (int i = 1; i < kC; ++i)
            if (chk[c * kC + i] != chk[c * kC]) { printf("cluster %d: CTAs disagree on the gathered data\n", c); return -1.0; }
    return (double)mx / rounds;
}

int main() {
    for (auto fn : {(const void*)allgather<0>, (const void*)allgather<1>})
    {
        cudaFuncSetAttribute(fn, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    }
    unsigned long long* d_ns; uint32_t* d_chk;
    cudaMalloc(&d_ns, sizeof(unsigned long long) * 8 * kC);
    cudaMalloc(&d_chk, sizeof(uint32_t) * 8 * kC);
    const int rounds = 20000;
    for (int clusters : {1, 7}) {
        for (int rep = 0; rep < 2; ++rep) {
            const double a = run<0>(clusters, rounds, d_ns, d_chk), b = run<1>(clusters, rounds, d_ns, d_chk);
            printf("%d cluster(s) x %d CTAs, 448 bf16 all-gather: st.async + mbarrier %7.1f ns/round | st.shared::cluster + cluster barrier %7.1f ns/round\n",
                   clusters, kC, a, b);
        }
    }
    cudaFree(d_ns); cudaFree(d_chk);
    return 0;
}
