// Integer-pipe probes: which instruction mix for a Threefry round issues fastest on sm_100a?
//   nvcc -O3 -gencode arch=compute_100a,code=sm_100a -o probe_int probe_int.cu && ./probe_int
#include <cstdio>
#include <cstdint>
#include <cstdlib>
#include <cuda_runtime.h>

__device__ __forceinline__ uint32_t rotl_shf(uint32_t x, int r) { return __funnelshift_l(x, x, r); }

// rotate through the FMA pipe: 64-bit product x * 2^r = {x >> (32-r), x << r}
__device__ __forceinline__ void mulwide(uint32_t x, uint32_t pow2, uint32_t& lo, uint32_t& hi) {
    asm volatile("{ .reg .u64 t; mul.wide.u32 t, %2, %3; mov.b64 {%0, %1}, t; }" : "=r"(lo), "=r"(hi) : "r"(x), "r"(pow2));
}
__device__ __forceinline__ uint32_t add_mad(uint32_t a, uint32_t b) {
    uint32_t d;
    asm volatile("mad.lo.u32 %0, %1, 1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
}

template <int V>
__device__ __forceinline__ void round_v(uint32_t& a, uint32_t& b, int r, int parity) {
    if (V == 0) { a += b; b = rotl_shf(b, r); b ^= a; }
    if (V == 1) { a += b; uint32_t lo, hi; mulwide(b, 1u << r, lo, hi); b = (lo | hi) ^ a; }
    if (V == 2) { a = add_mad(a, b); uint32_t lo, hi; mulwide(b, 1u << r, lo, hi); b = (lo | hi) ^ a; }
    if (V == 3) { if (parity) a = add_mad(a, b); else a += b; uint32_t lo, hi; mulwide(b, 1u << r, lo, hi); b = (lo | hi) ^ a; }
    if (V == 4) { a = add_mad(a, b); b = rotl_shf(b, r); b ^= a; }
    if (V == 6) { a = add_mad(a, b); if (parity == 3) { uint32_t lo, hi; mulwide(b, 1u << r, lo, hi); b = (lo | hi) ^ a; } else { b = rotl_shf(b, r); b ^= a; } }  // every 4th rotate through the FMA pipe
    if (V == 7) { a = add_mad(a, b); if (parity == 3) { uint32_t lo, hi; mulwide(b, 1u << r, lo, hi); b = add_mad(lo, hi) ^ a; } else { b = rotl_shf(b, r); b ^= a; } }  // same, halves joined by an add on the FMA pipe
    if (V == 5) { if (parity) { a += b; uint32_t lo, hi; mulwide(b, 1u << r, lo, hi); b = (lo | hi) ^ a; } else { a = add_mad(a, b); b = rotl_shf(b, r); b ^= a; } }
}

template <int V, int CH>
__global__ void probe(int iters, uint32_t* sink) {
    uint32_t a[CH], b[CH];
#pragma unroll
    for (int c = 0; c < CH; ++c) { a[c] = threadIdx.x + 17 * c; b[c] = blockIdx.x * 31 + c + 1; }
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int rs[4] = {13, 15, 26, 6};
#pragma unroll
            for (int c = 0; c < CH; ++c) round_v<V>(a[c], b[c], rs[k], V >= 6 ? k : (k & 1));
        }
    }
    uint32_t x = 0;
#pragma unroll
    for (int c = 0; c < CH; ++c) x ^= a[c] ^ b[c];
    sink[blockIdx.x * blockDim.x + threadIdx.x] = x;
}

template <int V, int CH>
void run(const char* name, int blocks) {
    uint32_t* sink;
    cudaMalloc(&sink, (size_t)blocks * 256 * 4);
    const int iters = 20000;
    probe<V, CH><<<blocks, 256>>>(iters, sink);
    cudaDeviceSynchronize();
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    float best = 1e9;
    for (int rep = 0; rep < 3; ++rep) {
        cudaEventRecord(e0);
        probe<V, CH><<<blocks, 256>>>(iters, sink);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms; cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best) best = ms;
    }
    const double rounds = (double)blocks * 256 * iters * 4 * CH;
    printf("%-44s CH=%d  %7.3f ms  %7.2f T rounds/s  (%.2f T instr/s at 3 instr/round)\n", name, CH, best, rounds / best / 1e9,
           3 * rounds / best / 1e9);
    cudaFree(sink);
}

// ---- whole Threefry-2x32-20 blocks at the play kernel's occupancy (512-thread CTAs, one per SM) ---------------------
// B0: the C code of g2048_rng.cuh before the change; ptxas folds each key injection and the round add after it into one
//     IADD3 (ALU pipe), and `ks + c` into an IADD3 with an immediate.
// B1: every add, key injections included, as mad.lo.u32 by an opaque 1 (FMA pipe); the `ks + c` sums computed once per
//     key, as the play kernel can (its action key hashes four blocks).
__device__ __forceinline__ uint32_t opaque_one() {
    uint32_t z;
    asm("mov.u32 %0, %%nctaid.z;" : "=r"(z));  // 1 for these launches; ptxas cannot see it as a constant
    return z;
}
__device__ __forceinline__ uint32_t madd(uint32_t a, uint32_t one, uint32_t b) {
    uint32_t d;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(one), "r"(b));
    return d;
}
struct KS { uint32_t k0, k1, k2, k0p2, k0p5, k1p3, k2p1, k2p4; };
__device__ __forceinline__ KS make_ks(uint32_t a, uint32_t b, uint32_t one) {
    KS s;
    s.k0 = a; s.k1 = b; s.k2 = a ^ b ^ 0x1BD11BDAu;
    s.k0p2 = madd(s.k0, one, 2u); s.k0p5 = madd(s.k0, one, 5u); s.k1p3 = madd(s.k1, one, 3u);
    s.k2p1 = madd(s.k2, one, 1u); s.k2p4 = madd(s.k2, one, 4u);
    return s;
}
template <int V>
__device__ __forceinline__ void tf_block(const KS& s, uint32_t one, uint32_t& x0, uint32_t& x1) {
    if (V == 0) {
#define PR(r) x0 += x1; x1 = rotl_shf(x1, r); x1 ^= x0;
        x0 += s.k0; x1 += s.k1;
        PR(13) PR(15) PR(26) PR(6) x0 += s.k1; x1 += s.k2 + 1u;
        PR(17) PR(29) PR(16) PR(24) x0 += s.k2; x1 += s.k0 + 2u;
        PR(13) PR(15) PR(26) PR(6) x0 += s.k0; x1 += s.k1 + 3u;
        PR(17) PR(29) PR(16) PR(24) x0 += s.k1; x1 += s.k2 + 4u;
        PR(13) PR(15) PR(26) PR(6) x0 += s.k2; x1 += s.k0 + 5u;
#undef PR
    } else {
#define MR(r) x0 = madd(x0, one, x1); x1 = rotl_shf(x1, r); x1 ^= x0;
        x0 = madd(x0, one, s.k0); x1 = madd(x1, one, s.k1);
        MR(13) MR(15) MR(26) MR(6) x0 = madd(x0, one, s.k1); x1 = madd(x1, one, s.k2p1);
        MR(17) MR(29) MR(16) MR(24) x0 = madd(x0, one, s.k2); x1 = madd(x1, one, s.k0p2);
        MR(13) MR(15) MR(26) MR(6) x0 = madd(x0, one, s.k0); x1 = madd(x1, one, s.k1p3);
        MR(17) MR(29) MR(16) MR(24) x0 = madd(x0, one, s.k1); x1 = madd(x1, one, s.k2p4);
        MR(13) MR(15) MR(26) MR(6) x0 = madd(x0, one, s.k2); x1 = madd(x1, one, s.k0p5);
#undef MR
    }
}
// one "step": the next key from the previous one (1 block), then four blocks under it (the action key's bits).
// CH independent key chains per thread: CH = 1 leaves 4 warps per scheduler with little to overlap the serial key
// block with (latency shows); CH = 2 doubles the independent work, so that pipe throughput alone decides.
template <int V, int CH>
__global__ void __launch_bounds__(512, 1) block_probe(int iters, uint32_t* sink) {
    const uint32_t one = opaque_one();
    uint32_t ka[CH], kb[CH], acc[CH];
#pragma unroll
    for (int h = 0; h < CH; ++h) { ka[h] = threadIdx.x * 0x9E3779B9u + h; kb[h] = blockIdx.x + 1u; acc[h] = 0; }
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int h = 0; h < CH; ++h) {
            KS s = make_ks(ka[h], kb[h], one);
            uint32_t y0 = 0u, y1 = (uint32_t)i;
            tf_block<V>(s, one, y0, y1);
            ka[h] = y0; kb[h] = y1;
            s = make_ks(ka[h], kb[h], one);
#pragma unroll
            for (uint32_t c = 0; c < 4; ++c) {
                uint32_t x0 = 0u, x1 = c;
                tf_block<V>(s, one, x0, x1);
                acc[h] ^= x0 ^ x1;
            }
            kb[h] ^= acc[h];
        }
    }
    uint32_t x = 0;
#pragma unroll
    for (int h = 0; h < CH; ++h) x ^= ka[h] ^ kb[h] ^ acc[h];
    sink[blockIdx.x * blockDim.x + threadIdx.x] = x;
}

// ---- which pipe takes an opcode: SHF.L.W chains (ALU) interleaved 1:1 with the opcode under test -------------------
// If the opcode runs on the ALU pipe the pair costs 2 ALU slots (4 cycles per warp), if it runs elsewhere 1 (2 cycles).
// O0: SHF only (the reference)   O1: + LOP3 (known ALU)   O2: + IMAD.IADD (known FMA)   O3: + IMAD.HI (opaque
// multiplier: a constant right shift through the FMA pipe)   O4: + PRMT   O5: VIADD (register + 32-bit immediate) inside the
// SHF chain (register rotate amount: with a constant one ptxas turns rotl(x + c) into LEA.HI)
// O6: + LEA.HI (`y + (x >> 28)`)   O7: + IADD3 (three register inputs)
template <int O>
__global__ void __launch_bounds__(512, 1) pipe_probe(int iters, uint32_t* sink) {
    const uint32_t one = opaque_one();
    const uint32_t mulhi = one << 28;  // umulhi(x, 2^28) = x >> 4
    uint32_t a[4], b[4], c = threadIdx.x ^ 0x5A5A5A5Au;
#pragma unroll
    for (int k = 0; k < 4; ++k) { a[k] = threadIdx.x * (k + 3u); b[k] = blockIdx.x + 7u * k; }
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                a[k] = (O == 5) ? rotl_shf(a[k] + (0x12345u + r), (int)(one * (5 + r))) : rotl_shf(a[k], 5 + r);
                if (O == 1) b[k] = (b[k] & c) ^ a[k];
                if (O == 2) b[k] = madd(b[k], one, a[k]);
                if (O == 3) { uint32_t d; asm("mad.hi.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(b[k]), "r"(mulhi), "r"(a[k])); b[k] = d; }
                if (O == 4) b[k] = __byte_perm(b[k], a[k], 0x6152);
                if (O == 6) b[k] = a[k] + (b[k] >> 28);
                if (O == 7) b[k] = b[k] + a[k] + c;
            }
        }
    }
    uint32_t x = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) x ^= a[k] ^ b[k];
    sink[blockIdx.x * blockDim.x + threadIdx.x] = x;
}

template <typename K>
float time_kernel(K kernel, int blocks, int iters, uint32_t* sink, int smem) {
    cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    kernel<<<blocks, 512, smem>>>(iters, sink);
    cudaDeviceSynchronize();
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    float best = 1e9;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0);
        kernel<<<blocks, 512, smem>>>(iters, sink);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms; cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best) best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return best;
}

void run_occupancy_probes(int sms) {
    uint32_t* sink;
    cudaMalloc(&sink, (size_t)sms * 512 * 4);
    const int smem = 160 * 1024;  // one 512-thread CTA per SM, as play3_kernel
    const int it_b = 20000;
    const double blocks_total = (double)sms * 512 * it_b * 5;
    for (int pass = 0; pass < 2; ++pass) {  // twice, so that drift of the box shows
        const float t0 = time_kernel(block_probe<0, 1>, sms, it_b, sink, smem);
        const float t1 = time_kernel(block_probe<1, 1>, sms, it_b, sink, smem);
        const float t2 = time_kernel(block_probe<0, 2>, sms, it_b / 2, sink, smem);
        const float t3 = time_kernel(block_probe<1, 2>, sms, it_b / 2, sink, smem);
        printf("B0 CH=1 Threefry blocks, C adds (IADD3 key injections)   %7.3f ms  %7.2f G blocks/s\n", t0, blocks_total / t0 / 1e6);
        printf("B1 CH=1 Threefry blocks, every add mad.lo (FMA pipe)     %7.3f ms  %7.2f G blocks/s  (B0/B1 time %.3f)\n", t1,
               blocks_total / t1 / 1e6, t0 / t1);
        printf("B0 CH=2 Threefry blocks, C adds (IADD3 key injections)   %7.3f ms  %7.2f G blocks/s\n", t2, blocks_total / t2 / 1e6);
        printf("B1 CH=2 Threefry blocks, every add mad.lo (FMA pipe)     %7.3f ms  %7.2f G blocks/s  (B0/B1 time %.3f)\n", t3,
               blocks_total / t3 / 1e6, t2 / t3);
    }
    const int it_o = 20000;
    const double pairs = (double)sms * 512 * it_o * 32;
    const char* names[8] = {"O0 SHF only", "O1 SHF + LOP3", "O2 SHF + IMAD.IADD", "O3 SHF + IMAD.HI (shift)", "O4 SHF + PRMT",
                            "O5 SHF + VIADD", "O6 SHF + LEA.HI", "O7 SHF + IADD3"};
    float t[8];
    t[0] = time_kernel(pipe_probe<0>, sms, it_o, sink, smem);
    t[1] = time_kernel(pipe_probe<1>, sms, it_o, sink, smem);
    t[2] = time_kernel(pipe_probe<2>, sms, it_o, sink, smem);
    t[3] = time_kernel(pipe_probe<3>, sms, it_o, sink, smem);
    t[4] = time_kernel(pipe_probe<4>, sms, it_o, sink, smem);
    t[5] = time_kernel(pipe_probe<5>, sms, it_o, sink, smem);
    t[6] = time_kernel(pipe_probe<6>, sms, it_o, sink, smem);
    t[7] = time_kernel(pipe_probe<7>, sms, it_o, sink, smem);
    for (int o = 0; o < 8; ++o)
        printf("%-28s %7.3f ms  %6.2f T pairs/s  time / O0 %.2f\n", names[o], t[o], pairs / t[o] / 1e9, t[o] / t[0]);
    cudaFree(sink);
}

int main() {
    int sms = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
    run_occupancy_probes(sms);
    if (getenv("PROBE_INT_ONLY_OCCUPANCY")) return 0;
    const int blocks = sms * 8;
    run<0, 4>("V0 add + SHF + LOP3 (C code)", blocks);
    run<1, 4>("V1 add + IMAD.WIDE rot + LOP3", blocks);
    run<2, 4>("V2 mad-add + IMAD.WIDE rot + LOP3", blocks);
    run<3, 4>("V3 alternating add/mad + IMAD.WIDE + LOP3", blocks);
    run<4, 4>("V4 mad-add + SHF + LOP3", blocks);
    run<5, 4>("V5 alternate (add,WIDE) / (mad,SHF)", blocks);
    run<6, 4>("V6 mad-add; SHF x3 + IMAD.WIDE x1 per 4 rounds", blocks);
    run<7, 4>("V7 same, halves joined by mad-add", blocks);
    run<0, 2>("V0", blocks); run<3, 2>("V3", blocks); run<5, 2>("V5", blocks);
    run<0, 8>("V0", blocks); run<3, 8>("V3", blocks); run<5, 8>("V5", blocks);
    return 0;
}
