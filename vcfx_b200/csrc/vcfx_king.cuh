// vcfx_king.cuh — KING-robust kinship counts on the tensor cores (tcgen05, sm_100a).
//
// Every count KING needs over all sample pairs is a product of 0/1 indicator matrices (include/vcfx_cuda.h, "pairwise
// relatedness"): CC = C Cᵀ, HH = H Hᵀ, AB = A Bᵀ, HC = H Cᵀ, with K = variants.  Two kernels per slab of rows:
//   king_planes_kernel  .bed rows (variant-major, 2 bits a call) -> the four int8 planes, sample-major, already in the
//                       shared-memory layout of the MMA (below), so that one tile is one contiguous block;
//   king_mma_kernel     one CTA per output tile: tcgen05.mma kind::i8 (u8 x u8 -> s32 in tensor memory) over the slab's
//                       K blocks, then the tile is added into the uint32 counts in global memory.
//
// Planes layout (DESIGN §2): plane p, K block kb (128 variants), sample s: 128 bytes at
//   planes + p * plane_stride + (kb * s_pad + s) * 128,
// one byte per variant, in the 128-byte swizzle of the UMMA K-major layout: the 16-byte chunk c (variants 16c .. 16c+15)
// of sample s sits at chunk position c ^ (s & 7).  Eight samples make one 1024-byte swizzle atom, so TM (TN) consecutive
// samples of one K block are a TM x 128 (TN x 128) K-major operand whose descriptor has SBO = 1024 and start = its first
// byte; the k-th 32-byte step of the block is start + 32 k (the hardware applies the swizzle to the address bits).
#pragma once

namespace vcfx {

constexpr uint32_t KING_KB = 128;                       // variants per K block = bytes of one plane row
constexpr uint32_t KING_TM = 128, KING_TN = 256;        // output tile: samples i (TMEM lanes) x samples j (TMEM columns)
constexpr uint32_t KING_UK = 32;                        // K of one kind::i8 instruction
constexpr uint32_t KING_STAGES = 4;
constexpr uint32_t KING_A_BYTES = KING_TM * KING_KB, KING_B_BYTES = KING_TN * KING_KB;
constexpr uint32_t KING_STAGE_BYTES = KING_A_BYTES + KING_B_BYTES;
constexpr uint32_t KING_SAMPLE_PAD = KING_TN;           // samples are padded to a multiple of both tile sides
constexpr uint64_t KING_MAX_S_PAD = (uint64_t)KING_TM << 14;   // a tile word holds the tile row in 14 bits: 2,097,152 samples
constexpr uint32_t KING_MMA_THREADS = 192;              // warp 0 loads, warp 1 issues the MMAs, warps 2-5 drain the tile
constexpr uint32_t KING_PLANES_THREADS = 256;
// 1024 bytes to align the ring to the swizzle atom, the ring, then 2 x STAGES + 1 mbarriers and the TMEM address
constexpr size_t KING_MMA_SMEM = 1024 + (size_t)KING_STAGES * KING_STAGE_BYTES + 8 * (2 * KING_STAGES + 1) + 8;
enum { KING_PA, KING_PH, KING_PB, KING_PC };             // planes: hom A2 (REF/REF), het, hom A1, called
enum { KING_CC, KING_HH, KING_AB, KING_HC };             // problems, in the order vcfx_cuda_king_counts writes them
// instruction descriptor: D = s32 (bits 4-5 = 2), A = B = u8 (bits 7-9, 10-12 = 0), both K-major (bits 15, 16 = 0),
// N >> 3 at bit 17, M >> 4 at bit 24
constexpr uint32_t KING_IDESC = (2u << 4) | ((KING_TN >> 3) << 17) | ((KING_TM >> 4) << 24);
static_assert(KING_TM == 128 && KING_TN % 16 == 0 && KING_TN <= 256, "kind::i8 with M = 128 takes N = 16 .. 256 in steps of 16");
static_assert(KING_MMA_SMEM <= 227u * 1024u, "the ring must fit one CTA's shared memory");

struct KingPlanesParams {
    const uint8_t *rows;      // n_rows .bed rows of row_bytes bytes
    uint8_t *planes;
    size_t plane_stride;      // bytes of one plane (the slab's capacity)
    uint32_t n_rows, row_bytes, n_samples, s_pad;
};

struct KingMmaParams {
    const uint8_t *planes;
    size_t plane_stride;
    uint32_t *acc;            // [4][s_pad][s_pad]
    const uint32_t *tiles;    // problem << 28 | tile row << 14 | tile column, one per CTA
    uint32_t s_pad, kblocks;
};

struct KingCountsParams {
    const uint32_t *acc;
    uint32_t *dst;            // [4][n][n]
    uint32_t n, s_pad;
};

// ---- PTX wrappers and their emulator twins -------------------------------------------------------------------------
#ifdef VCFX_EMU
// The emulator runs a CTA's threads one at a time and switches between warps only at warp collectives: an mbarrier is a
// real counter in shared memory and a wait is a vote of the whole warp, repeated until the phase has flipped (each vote
// lets the other warps run); tensor memory is one array (CTAs run one after the other); the MMA reads its operands from
// shared memory through the descriptors it is given, so a wrong descriptor or a wrong planes layout gives wrong counts
// here as well.  Shared addresses are offsets into the dynamic shared memory, which holds everything they address.
struct EmuBar { uint32_t expected : 15, phase : 1, pending : 16; int32_t tx; };
static_assert(sizeof(EmuBar) == 8, "an mbarrier is 8 bytes");
static uint32_t king_emu_tmem[128][512];
[[noreturn]] inline void king_emu_die(const char *what) { fprintf(stderr, "emu: %s\n", what); abort(); }
inline EmuBar *emu_bar(uint32_t a) { return reinterpret_cast<EmuBar *>(static_cast<char *>(emu::dyn_smem()) + a); }
inline void emu_bar_complete(EmuBar *b) {
    if (b->pending == 0 && b->tx == 0) { b->phase ^= 1u; b->pending = b->expected; }
}
__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)(static_cast<const char *>(p) - static_cast<const char *>(emu::dyn_smem())); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { EmuBar *b = emu_bar(bar); b->expected = count; b->pending = count; b->phase = 0; b->tx = 0; }
__device__ __forceinline__ void mbar_init_fence() {}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    EmuBar *b = emu_bar(bar);
    if (b->pending == 0) king_emu_die("mbarrier arrive with no pending arrival");
    b->tx += (int32_t)bytes; b->pending -= 1; emu_bar_complete(b);
}
// called by all 32 lanes of a warp
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    for (uint64_t spins = 0; !__all_sync(FULL, emu_bar(bar)->phase != parity); ++spins)
        if (spins > (1ull << 24)) king_emu_die("mbarrier wait never completes");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint32_t bar) {
    if ((bytes & 15) || ((uintptr_t)src & 15) || (smem_addr(dst) & 15)) king_emu_die("cp.async.bulk wants 16-byte sizes and addresses");
    memcpy(dst, src, bytes);
    EmuBar *b = emu_bar(bar); b->tx -= (int32_t)bytes; emu_bar_complete(b);
}
__device__ __forceinline__ void tmem_alloc(uint32_t slot, uint32_t cols) {
    if (cols < 32 || cols > 512 || (cols & (cols - 1))) king_emu_die("tcgen05.alloc wants a power of two in 32 .. 512 columns");
    if ((threadIdx.x & 31) == 0) *reinterpret_cast<uint32_t *>(static_cast<char *>(emu::dyn_smem()) + slot) = 0;   // lane 0, column 0
}
__device__ __forceinline__ void tmem_relinquish() {}
__device__ __forceinline__ void tmem_dealloc(uint32_t, uint32_t) {}
__device__ __forceinline__ void tc_fence_before() {}
__device__ __forceinline__ void tc_fence_after() {}
// K-major operand byte (row r, byte kk of the 32-byte K step) through a shared-memory descriptor: start (bits 0-13, >> 4),
// SBO (bits 32-45, >> 4), version 1 (bits 46-47), base offset 0 (bits 49-51), layout 2 = 128-byte swizzle (bits 61-63)
inline uint8_t emu_operand(uint64_t d, uint32_t r, uint32_t kk) {
    const uint32_t start = (uint32_t)(d & 0x3FFF) << 4, sbo = (uint32_t)((d >> 32) & 0x3FFF) << 4;
    if (((d >> 46) & 3) != 1 || ((d >> 49) & 7) != 0 || (d >> 61) != 2) king_emu_die("unsupported shared-memory descriptor");
    uint32_t a = start + (r >> 3) * sbo + (r & 7) * 128u + kk;
    a ^= ((a >> 7) & 7u) << 4;
    return static_cast<const uint8_t *>(emu::dyn_smem())[a];
}
__device__ __forceinline__ void umma_i8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, bool accumulate) {
    const uint32_t M = ((idesc >> 24) & 0x1F) << 4, N = ((idesc >> 17) & 0x3F) << 3;
    if (((idesc >> 4) & 3) != 2 || ((idesc >> 7) & 0x3F) != 0 || ((idesc >> 13) & 0xF) != 0 || (idesc & 0xF) != 0 || M != 128 || N == 0 || N > 256)
        king_emu_die("unsupported instruction descriptor (wants u8 x u8 -> s32, K-major, M = 128)");
    const uint32_t lane0 = d_tmem >> 16, col0 = d_tmem & 0xFFFF;
    if (lane0 != 0 || col0 + N > 512) king_emu_die("accumulator outside tensor memory");
    uint8_t a[128][32], b[256][32];
    for (uint32_t r = 0; r < M; ++r) for (uint32_t k = 0; k < KING_UK; ++k) a[r][k] = emu_operand(adesc, r, k);
    for (uint32_t r = 0; r < N; ++r) for (uint32_t k = 0; k < KING_UK; ++k) b[r][k] = emu_operand(bdesc, r, k);
    for (uint32_t i = 0; i < M; ++i)
        for (uint32_t j = 0; j < N; ++j) {
            int32_t s = 0;
            for (uint32_t k = 0; k < KING_UK; ++k) s += (int32_t)a[i][k] * (int32_t)b[j][k];
            uint32_t &dst = king_emu_tmem[i][col0 + j];
            dst = accumulate ? dst + (uint32_t)s : (uint32_t)s;
        }
}
__device__ __forceinline__ void umma_commit(uint32_t bar) { mbar_arrive_expect_tx(bar, 0); }   // the MMAs above are done
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    const uint32_t lane = (taddr >> 16) + (threadIdx.x & 31), col = taddr & 0xFFFF;
    if ((taddr >> 16) != 32 * ((threadIdx.x >> 5) & 3)) king_emu_die("a warp may only read its own quarter of the TMEM lanes");
    for (int i = 0; i < 32; ++i) v[i] = king_emu_tmem[lane][col + i];
}
__device__ __forceinline__ void tmem_ld_wait() {}
#else
__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count)); }
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    while (!done)
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_addr(dst)), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t slot, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(slot), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_i8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, bool accumulate) {
    asm volatile("{ .reg .pred p; setp.ne.b32 p, %4, 0;\n"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p; }"
                 :: "r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate) : "memory");
}
// arrives on the mbarrier once every MMA this thread issued before it has completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
#endif

// K-major, 128-byte swizzle operand descriptor for the tile starting at shared address `saddr` (1024-byte aligned)
__device__ __forceinline__ uint64_t king_smem_desc(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)1 << 16) /* LBO: unused with this swizzle */ |
           ((uint64_t)(1024 >> 4) << 32) /* SBO: 8 rows of 128 bytes */ | ((uint64_t)1 << 46) /* version */ | ((uint64_t)2 << 61);
}

// four 0/1 bytes from the low four bits of m
__device__ __forceinline__ uint32_t king_bytes4(uint32_t m) { return ((m & 0xFu) * 0x00204081u) & 0x01010101u; }
__device__ __forceinline__ uint4 king_bytes16(uint32_t m) {
    return make_uint4(king_bytes4(m), king_bytes4(m >> 4), king_bytes4(m >> 8), king_bytes4(m >> 12));
}

// One CTA per (K block, 128 samples): the 128 rows' 32 bytes of those samples go to shared memory (rows past n_rows and
// bytes past the row read as 01 = missing, which sets no plane), then each item is 16 variants of one sample, written as
// one 16-byte chunk of each plane.  32 consecutive items are four whole 128-byte plane rows: the stores are coalesced.
__global__ void __launch_bounds__(KING_PLANES_THREADS)
king_planes_kernel(const KingPlanesParams P) {
    __shared__ uint8_t tile[KING_KB][33];              // (33: the eight chunks of a warp read eight different banks)
    const uint32_t sblocks = P.s_pad / 128, kb = blockIdx.x / sblocks, sb = blockIdx.x % sblocks;
    for (uint32_t i = threadIdx.x; i < KING_KB * 32; i += KING_PLANES_THREADS) {
        const uint32_t v = i >> 5, x = i & 31, r = kb * KING_KB + v, byte = sb * 32 + x;
        tile[v][x] = (r < P.n_rows && byte < P.row_bytes) ? P.rows[(size_t)r * P.row_bytes + byte] : (uint8_t)0x55;
    }
    __syncthreads();
    for (uint32_t it = threadIdx.x; it < 128 * 8; it += KING_PLANES_THREADS) {
        const uint32_t sl = it >> 3, c = it & 7, s = sb * 128 + sl, sh = 2 * (sl & 3);
        uint32_t lo = 0, hi = 0;
#pragma unroll
        for (uint32_t j = 0; j < 16; ++j) {
            const uint32_t code = ((uint32_t)tile[c * 16 + j][sl >> 2] >> sh) & 3u;
            lo |= (code & 1u) << j; hi |= (code >> 1) << j;
        }
        // 11 hom A2, 10 het, 00 hom A1, 01 missing; samples past n_samples are padding whatever their bits
        const uint32_t keep = s < P.n_samples ? 0xFFFFu : 0u;
        const uint32_t a = hi & lo & keep, h = hi & ~lo & keep, b = ~hi & ~lo & keep, called = (hi | ~lo) & keep;
        const size_t off = ((size_t)kb * P.s_pad + s) * KING_KB + 16 * (c ^ (s & 7));
        *reinterpret_cast<uint4 *>(P.planes + KING_PA * P.plane_stride + off) = king_bytes16(a);
        *reinterpret_cast<uint4 *>(P.planes + KING_PH * P.plane_stride + off) = king_bytes16(h);
        *reinterpret_cast<uint4 *>(P.planes + KING_PB * P.plane_stride + off) = king_bytes16(b);
        *reinterpret_cast<uint4 *>(P.planes + KING_PC * P.plane_stride + off) = king_bytes16(called);
    }
}

// One CTA per output tile of one problem, over all K blocks of the slab.  Warp 0 (lane 0 issuing) streams the A and B operand
// tiles of each K block into a ring of KING_STAGES stages with cp.async.bulk (completion on the stage's "full" mbarrier);
// warp 1 (lane 0 issuing) issues four MMAs per stage into the 128 x 256 s32 accumulator in tensor memory and commits each stage
// back to its "empty" mbarrier; once the last MMA has completed ("acc" mbarrier), warps 2-5 each read their quarter of the
// TMEM lanes (32 rows) and add them into the counts.  A tile belongs to one CTA of a launch, so the adds need no atomics.
__global__ void __launch_bounds__(KING_MMA_THREADS, 1)
king_mma_kernel(const KingMmaParams P) {
#ifdef VCFX_EMU
    uint8_t *smem = static_cast<uint8_t *>(emu::dyn_smem());
#else
    extern __shared__ __align__(1024) uint8_t smem[];
#endif
    uint8_t *ring = smem + ((1024u - (smem_addr(smem) & 1023u)) & 1023u);
    const uint32_t bars = smem_addr(ring + KING_STAGES * KING_STAGE_BYTES);      // full[s], empty[s], acc: 8 bytes each
    const uint32_t full0 = bars, empty0 = bars + 8 * KING_STAGES, acc_bar = bars + 16 * KING_STAGES, slot = acc_bar + 8;
    const uint32_t *tmem_slot = reinterpret_cast<const uint32_t *>(ring + KING_STAGES * KING_STAGE_BYTES + 8 * (2 * KING_STAGES + 1));
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t t = P.tiles[blockIdx.x], prob = t >> 28, mi = (t >> 14) & 0x3FFF, nj = t & 0x3FFF;
    const uint32_t pa = prob == KING_CC ? KING_PC : prob == KING_AB ? KING_PA : KING_PH;
    const uint32_t pb = prob == KING_HH ? KING_PH : prob == KING_AB ? KING_PB : KING_PC;

    if (threadIdx.x == 0) {
        for (uint32_t s = 0; s < KING_STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        mbar_init(acc_bar, 1);
        mbar_init_fence();
    }
    if (warp == 1) { tmem_alloc(slot, KING_TN); tmem_relinquish(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    // warps 0 and 1 wait as whole warps (the emulator switches warps at warp collectives); lane 0 issues
    if (warp == 0) {
        const uint8_t *ga = P.planes + pa * P.plane_stride + (size_t)mi * KING_TM * KING_KB;
        const uint8_t *gb = P.planes + pb * P.plane_stride + (size_t)nj * KING_TN * KING_KB;
        const size_t kstep = (size_t)P.s_pad * KING_KB;
        for (uint32_t kb = 0; kb < P.kblocks; ++kb) {
            const uint32_t s = kb % KING_STAGES, ph = (kb / KING_STAGES) & 1u;
            mbar_wait(empty0 + 8 * s, ph ^ 1u);
            if (lane == 0) {
                uint8_t *st = ring + s * KING_STAGE_BYTES;
                mbar_arrive_expect_tx(full0 + 8 * s, KING_STAGE_BYTES);
                bulk_g2s(st, ga + kb * kstep, KING_A_BYTES, full0 + 8 * s);
                bulk_g2s(st + KING_A_BYTES, gb + kb * kstep, KING_B_BYTES, full0 + 8 * s);
            }
        }
    } else if (warp == 1) {
        for (uint32_t kb = 0; kb < P.kblocks; ++kb) {
            const uint32_t s = kb % KING_STAGES, ph = (kb / KING_STAGES) & 1u;
            mbar_wait(full0 + 8 * s, ph);
            if (lane == 0) {
                tc_fence_after();
                const uint32_t sa = smem_addr(ring + s * KING_STAGE_BYTES);
                const uint64_t da = king_smem_desc(sa), db = king_smem_desc(sa + KING_A_BYTES);
#pragma unroll
                for (uint32_t k = 0; k < KING_KB / KING_UK; ++k)       // k-th 32-byte step: start address + 32 k
                    umma_i8(tmem, da + 2 * k, db + 2 * k, KING_IDESC, (kb | k) != 0);
                umma_commit(empty0 + 8 * s);
            }
        }
        if (lane == 0) umma_commit(acc_bar);
    } else if (warp >= 2) {
        const uint32_t q = warp & 3;                              // a warp reads TMEM lanes 32 (warp % 4) .. + 31
        mbar_wait(acc_bar, 0);
        tc_fence_after();
        const uint32_t row = mi * KING_TM + 32 * q + lane;
        uint4 *dst = reinterpret_cast<uint4 *>(P.acc + ((size_t)prob * P.s_pad + row) * P.s_pad + (size_t)nj * KING_TN);
        for (uint32_t c = 0; c < KING_TN; c += 32) {
            uint32_t v[32];
            tmem_ld32(tmem + ((32 * q) << 16) + c, v);
            tmem_ld_wait();
#pragma unroll
            for (uint32_t j = 0; j < 8; ++j) {
                uint4 o = dst[c / 4 + j];
                o.x += v[4 * j]; o.y += v[4 * j + 1]; o.z += v[4 * j + 2]; o.w += v[4 * j + 3];
                dst[c / 4 + j] = o;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) { tc_fence_after(); tmem_dealloc(tmem, KING_TN); }
}

// the four n x n count matrices, row-major, from the padded accumulator: CC and HH were computed on and above the
// diagonal tiles only, so their (i, j) is read at (min, max)
__global__ void __launch_bounds__(256)
king_counts_kernel(const KingCountsParams P) {
    const size_t nn = (size_t)P.n * P.n, total = 4 * nn;
    for (size_t x = (size_t)blockIdx.x * 256 + threadIdx.x; x < total; x += (size_t)gridDim.x * 256) {
        const uint32_t prob = (uint32_t)(x / nn);
        const size_t r = x - prob * nn;
        uint32_t i = (uint32_t)(r / P.n), j = (uint32_t)(r - (size_t)i * P.n);
        if ((prob == KING_CC || prob == KING_HH) && i > j) { const uint32_t tmp = i; i = j; j = tmp; }
        P.dst[x] = P.acc[((size_t)prob * P.s_pad + i) * P.s_pad + j];
    }
}

}  // namespace vcfx
