// FP8 GEMM on the 5th-generation tensor cores:  C = epi( A[M,K] * B[N,K]^T ),  both operands
// K-major e4m3 bytes, fp32 accumulation in tensor memory.
//
// Replaces the reference's large-M routes: fp8_scaled_matmul_kernel (fp8_matmul.metal:99-147, one
// thread per output element, 2K single-byte loads each) and fp8_scaled_mm_fast
// (fp8_mps_native.py:213-267: two dequantise passes to fp16, two fp16 scale passes, an fp16 GEMM and
// an fp32 cast -- six launches and 3x the bytes), plus the patch's bias / scale_result / out_dtype
// passes (fp8_mps_patch.py:95-104).  One launch here.
//
// Structure (persistent, warp-specialised, one CTA per SM):
//   warp 4      TMA producer: cp.async.bulk.tensor 2D loads of a 128 x 128 B A tile and a BN x 128 B
//               B tile per k-block into a STAGES-deep 128B-swizzled shared-memory ring (mbarrier
//               complete_tx).  The reference's (N,K) weight layout is already the K-major form
//               tcgen05 wants, so neither operand is transposed.  TMA zero-fills out-of-range rows and
//               the K tail; 0x00 decodes to 0, so edges need no special code.
//   warp 5      MMA issuer: one thread issues tcgen05.mma.cta_group::1.kind::f8f6f4 (M=128, N=BN, K=32),
//               four per k-block; tcgen05.commit releases each smem slot and finally publishes the
//               accumulator.
//   warps 0-3   epilogue: tcgen05.ld (32 lanes x 32 columns per warp per step) -> ((acc*sa)*sb)+bias,
//               *scale_result -> out dtype -> 16-byte global stores.  Two accumulators of BN columns
//               live in TMEM (2*BN <= 512 columns) so the epilogue of tile i overlaps the main loop
//               of tile i+1.
// NaN bytes (0x7F/0xFF) make the hardware accumulator NaN where the reference decodes 0
// (metal:21); the epilogue recomputes exactly those outputs with the masked scalar loop.
#include <cuda.h>
#include <cstdio>
#include <mutex>
#include <type_traits>

#include "fp8_mm.cuh"
#include "fp8_async.cuh"

namespace fp8b {

constexpr int kBM = 128;          // rows of A per tile = UMMA M
constexpr int kBK = 128;          // bytes of K per stage = one 128B swizzle span
constexpr int kUmmaK = 32;        // bytes of K per tcgen05.mma (kind::f8f6f4)
// Epilogue warps: a multiple of 4 (one per TMEM lane quarter); with 8 the two warps of a quarter split the
// tile's columns.  Measured on C4 (256x256 pair tiles): 4 warps 113.1 us, 8 warps 119.3 us -> 4.
#ifndef FP8B_EPI_WARPS
#define FP8B_EPI_WARPS 4
#endif
constexpr int kNumEpiWarps = FP8B_EPI_WARPS;
constexpr int kEpiColSplits = kNumEpiWarps / 4;
// How the epilogue gets the tile to memory (template parameter MODE):
//   kStDirect  epilogue warps store with st.global (or multimem.st when C is a multicast address)
//   kStPeers   epilogue warps store every piece locally and into each peer's buffer with st.global (round-1 plan)
//   kStTma     epilogue warps only fill a swizzled shared-memory ring; a dedicated STORE warp pushes each
//              128-row x 128-byte box with cp.async.bulk.tensor (TMA store) to 1..8 destinations -- this rank's
//              buffer and, over NVLink, the same place in every peer's buffer.  The epilogue warps never wait on
//              the memory system, so the accumulator goes back to the MMA warp as soon as TMEM is drained.
enum { kStDirect = 0, kStPeers = 1, kStTma = 2 };
template <int MODE> constexpr bool is_push() { return MODE == kStTma; }
constexpr int kMaxDst = 8;
template <int MODE> constexpr int gemm_threads() { return 64 + 32 * kNumEpiWarps + (is_push<MODE>() ? 32 : 0); }

constexpr int kStoreBoxBytes = 128 * 128;       // one TMA-store box: 128 rows x 128 bytes, 128B-swizzled
#ifndef FP8B_TMA_SLOTS
#define FP8B_TMA_SLOTS 4                        // ring of 16 KB store boxes (kStTma); 2 leaves room for a sixth operand stage
#endif
constexpr int kStoreInflight = FP8B_TMA_SLOTS >= 4 ? 2 : 1;   // TMA-store groups that may still be reading shared memory
// Warp roles.  The epilogue takes the LOW warp ids and the two single-thread roles the HIGH ones: the warp
// scheduler favours higher warp ids among eligible warps, and the MMA issuer / TMA producer are latency-critical
// (with the roles the other way round the epilogue's ALU stream delayed MMA issue: 14.2K vs 12.4K cycles per tile).
constexpr int kWarpEpi0 = 0;                    // warps 0..kNumEpiWarps-1: epilogue (TMEM lane quarter = warp % 4)
constexpr int kWarpTma = kNumEpiWarps;          // TMA producer
constexpr int kWarpMma = kNumEpiWarps + 1;      // MMA issuer
constexpr int kWarpStore = kNumEpiWarps + 2;    // kStTma only: TMA-store issuer

// Profiling knobs (FP8B_GEMM_DEBUG bits, per-tile clock stamps) exist only in -DFP8B_PROFILE builds: the shipped
// library has no run-time switch that can change a result.
#ifdef FP8B_PROFILE
#define FP8B_DBG(p, bits) ((p).debug & (bits))
#else
#define FP8B_DBG(p, bits) 0
#endif

// CG = CTA-group size.  CG == 2: two CTAs of a cluster (an SM pair) compute one 256 x BN tile with
// tcgen05.mma.cta_group::2 -- each CTA stages its own 128 rows of A and only HALF of the B tile, so the
// shared-memory traffic per MMA (operand reads + TMA writes) drops from 24 KB to 16 KB per 128 cycles.
template <int BN, int CG, int MODE = kStDirect> struct GemmCfg {
    static constexpr int kABytes = kBM * kBK;
    static constexpr int kBRows = BN / CG;                         // B rows staged by one CTA
    static constexpr int kBBytes = kBRows * kBK;
    static constexpr int kStageBytes = kABytes + kBBytes;
    // epilogue staging: per epilogue warp 32 rows x 256 B, XOR-swizzled -- or the store ring
    static constexpr int kEpiStageBytes = is_push<MODE>() ? FP8B_TMA_SLOTS * kStoreBoxBytes : kNumEpiWarps * 8192;
    static constexpr int kStagesFit = (232448 - 1024 - 256 - kEpiStageBytes) / kStageBytes;
    static constexpr int kStages = kStagesFit > 8 ? 8 : kStagesFit;
    static constexpr int kTmemCols = (2 * BN > 256) ? 512 : 256;   // two accumulators; a power of two >= 32
    static constexpr int kBarBytes = 256;
    // layout: [operand ring | epilogue staging (1024-byte aligned) | barriers]
    static constexpr int kOffStaging = kStages * kStageBytes;
    static constexpr int kOffBar = kOffStaging + kEpiStageBytes;
    static constexpr int kSmemBytes = kOffBar + kBarBytes + 1024;   // +1024: manual alignment
    static_assert(kStageBytes % 1024 == 0, "operand stages must keep the 1024-byte swizzle alignment");
    static_assert((2 * kStages + 4 + 2 * FP8B_TMA_SLOTS) * 8 + 8 <= kBarBytes, "barrier block too small");
};

// kStTma: one tensor map per destination buffer, plus the optional completion signal: when the last CTA of
// the grid has pushed its last box, it stores `epoch` into sig[d] for every peer d (a flag in the PEER's memory).
struct StoreMaps {
    CUtensorMap m[kMaxDst];
    unsigned long long* sig[kMaxDst];        // sig[d]: where to tell destination d "rank's boxes have landed" (null: nobody)
    unsigned int* cta_counter;               // device counter, 0 between launches (reset by the last CTA)
    unsigned long long epoch;
    int n_sig;                               // 0: no signalling (the caller orders ranks itself)
};
struct NoStoreMaps { int unused; };
template <int MODE> struct StoreMapsOf { using type = NoStoreMaps; };
template <> struct StoreMapsOf<kStTma> { using type = StoreMaps; };

struct GemmParams {
    const uint8_t* A; const uint8_t* B;      // for the NaN fix-up only
    int M, N, K;
    int num_m_blocks, num_n_blocks, num_k_blocks;
    int raster_n;                            // tile order: 0 = M fastest (consecutive work items share a B tile), 1 = N fastest,
                                             // 2 = grouped: N fastest inside bands of kRasterGroup M-blocks (both operands large)
    int stage_tx;                            // bytes one CTA's two TMA loads deliver per stage (the A box is shorter when M < 128)
    int full_tiles;                          // work items [0, full_tiles) are BN-wide tiles ...
    int num_work;                            // ... items [full_tiles, num_work) are half-width tiles (last-wave split)
    Epi epi;
    int vec_store_ok;                        // C base and ldc allow 16-byte row-chunk stores
    int col_vec_ok;                          // scale_b / bias bases allow 16-byte broadcast loads
    int multicast;                           // kStDirect: C is an NVSwitch multicast address (multimem.st)
    int n_dst;                               // kStPeers: world size; kStTma: number of destinations
    const long long* peer_delta;             // kStPeers: device table of per-rank byte offsets from C
    int a_fmt, b_fmt;                        // operand formats: 0 = e4m3, 1 = e5m2
#ifdef FP8B_PROFILE
    long long* dbg;                          // FP8B_GEMM_DEBUG & 16: per-tile clock64 stamps of CTA 0 (else null)
    int debug;                               // FP8B_GEMM_DEBUG bits
#endif
};

// ------------------------------------------------------------------------------ PTX wrappers

__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" :: "l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 :: "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1) : "memory");
}

// TMA store of one box from shared memory (bulk async-group completion).  The tensor map may describe local HBM or
// a peer GPU's buffer mapped into this process: the copy engine of the SM does the NVLink writes.
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, uint32_t smem_src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 :: "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_group_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" :: "n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_group_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_dst), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, e4m3 x e4m3 -> f32
__device__ __forceinline__ void umma_f8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// mbarrier arrives once every tcgen05 op issued so far by this thread has completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
}

__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// The same wait, naming the registers an earlier tcgen05.ld is filling as in/out operands: with two loads in flight
// (software-pipelined epilogue) this is what keeps the compiler from scheduling a use of r[] above the wait.
__device__ __forceinline__ void tmem_ld_wait_for(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                   "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                   "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :: "memory");
}

// ---- cta_group::2 flavours (a CTA pair; rank 0 of the cluster is the leader) -------------------
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;      // clears the CTA-rank bit of a shared::cluster address -> even CTA

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// Execution barrier only: no memory ordering.  For the end of a kernel, where the release flavour would first wait for
// every global store of the epilogue to be acknowledged (measured: 2 000-4 000 cycles in the split-K kernel).
__device__ __forceinline__ void cluster_sync_relaxed() {
    asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.aligned;" ::: "memory");
}
// TMA load issued by either CTA of the pair; the bytes are accounted on the LEADER's mbarrier
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t smem_dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 :: "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar & kPeerBitMask), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" :: "r"(bar & kPeerBitMask) : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_dst), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2sm() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" :: "r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_f8_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrives on the barrier at this offset in BOTH CTAs of the pair once the MMAs issued so far retire
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 :: "r"(bar), "h"((uint16_t)3) : "memory");
}

// One lane of a fully converged warp; the compiler recognises the elect.sync predicate as "single thread",
// which lets it keep the tcgen05 / TMA operands in uniform registers without a per-lane waterfall loop.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xFFFFFFFF;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}

// K-major, 128B-swizzled shared-memory operand descriptor (PTX "matrix descriptor", sm_100 version 1):
//   [0,14)  start address >> 4        [16,30) leading byte offset >> 4 (unused for swizzled K-major: 1)
//   [32,46) stride byte offset >> 4 = 1024 B between 8-row groups      [46,48) version = 1
//   [61,64) layout = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// Instruction descriptor for kind::f8f6f4: D = f32 (bits 4-5 = 1), A format at [7,10), B format at [10,13)
// (0 = e4m3, 1 = e5m2; OR-ed in at run time from GemmParams::a_fmt / b_fmt), both K-major (bits 15,16 = 0),
// N >> 3 at [17,23), M >> 4 at [24,29).
__host__ __device__ constexpr uint32_t make_idesc(int m, int n) {
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// mc == 0: ordinary 16-byte global store.  mc != 0: `p` is an NVSwitch MULTICAST address and the store
// is replicated by the switch into the same offset of every GPU bound to the multicast object
// (multimem.st) -- the output tile reaches all ranks of an N-sharded linear in one instruction.
__device__ __forceinline__ void stg_v4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d, int mc) {
    if (mc)
        asm volatile("multimem.st.weak.global.v4.f32 [%0], {%1,%2,%3,%4};"
                     :: "l"(p), "f"(__uint_as_float(a)), "f"(__uint_as_float(b)), "f"(__uint_as_float(c)),
                        "f"(__uint_as_float(d)) : "memory");
    else
        asm volatile("st.global.v4.u32 [%0], {%1,%2,%3,%4};" :: "l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

__device__ __forceinline__ void sts_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" :: "r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void lds_v4(uint32_t addr, uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(addr) : "memory");
}

// Work item -> tile.  The last, partially filled wave of BN-wide tiles is cut into half-width tiles so that it
// takes about half a tile time and ends with a half-size epilogue (C4: 768 tiles on 74 CTA pairs = 10 full
// rounds + 28 tiles -> 56 half tiles in one short round).
constexpr int kRasterGroup = 8;
struct TileCoord { int m_blk; int n0; int width; };
__device__ __forceinline__ TileCoord decode_tile(const GemmParams& p, int t, int bn) {
    TileCoord c;
    int tt = t, half = -1;
    if (t >= p.full_tiles) {
        const int u = t - p.full_tiles;
        tt = p.full_tiles + (u >> 1);
        half = u & 1;
    }
    int n_blk;
    if (p.raster_n == 2) {
        // bands of kRasterGroup M-blocks, M fastest inside a band: the ~74 tiles in flight form a near-square patch of the
        // output, so a wave re-reads ~8 A-blocks + ~9 B-blocks from L2 instead of 2 + all of B
        const int per_band = kRasterGroup * p.num_n_blocks;
        const int band = tt / per_band, r = tt - band * per_band;
        const int m0 = band * kRasterGroup;
        const int rows = min(kRasterGroup, p.num_m_blocks - m0);
        c.m_blk = m0 + r % rows;
        n_blk = r / rows;
    }
    else if (p.raster_n) { n_blk = tt % p.num_n_blocks; c.m_blk = tt / p.num_n_blocks; }
    else { c.m_blk = tt % p.num_m_blocks; n_blk = tt / p.num_m_blocks; }
    c.width = half < 0 ? bn : bn >> 1;
    c.n0 = n_blk * bn + (half > 0 ? c.width : 0);
    return c;
}

// The epilogue arithmetic of one 32-column chunk, in the reference's order (acc * scale_a * scale_b [+ bias] [* scale_result],
// every step rounded to fp32), specialised on which optional terms exist so that the 32-element loop is branch-free:
// with the three run-time tests inside the loop the chunk compiled to ~1000 SASS instructions and the epilogue of a
// 128 x 256 accumulator took as long as its K = 3072 main loop (12 000 cycles, measured with the per-tile clock stamps).
template <bool SBV, bool BIAS, bool SR>
__device__ __forceinline__ void epi_math32(const uint32_t (&r)[32], float sa, float sb0, float sr, const float (&sbv)[32],
                                           const float (&bv)[32], float (&v)[32]) {
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        float x = __fmul_rn(__uint_as_float(r[j]), sa);
        x = __fmul_rn(x, SBV ? sbv[j] : sb0);
        if (BIAS) x = __fadd_rn(x, bv[j]);
        if (SR) x = __fmul_rn(x, sr);
        v[j] = x;
    }
}
// NaN anywhere in the 32 accumulators of a lane?  (four independent add chains instead of one 32-long one)
__device__ __forceinline__ bool any_nan32(const uint32_t (&r)[32]) {
    float s0 = 0.0f, s1 = 0.0f, s2 = 0.0f, s3 = 0.0f;
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
        s0 += __uint_as_float(r[j]); s1 += __uint_as_float(r[j + 1]);
        s2 += __uint_as_float(r[j + 2]); s3 += __uint_as_float(r[j + 3]);
    }
    const float s = (s0 + s1) + (s2 + s3);
    return s != s;
}

__device__ __forceinline__ int out_esz(int out_dtype) { return out_dtype == FP8B_F32 ? 4 : out_dtype == FP8B_OUT_E4M3FN ? 1 : 2; }

// The 32 epilogue values of one lane -> the output type, packed little-endian into the row's 16-byte pieces, each handed
// to store16(j, w0, w1, w2, w3) for piece j: 8 pieces (f32), 4 (f16 / bf16) or 2 (e4m3fn: the reference encoder,
// enc_prepare_f32 on the input, then the satfinite conversion).  Every vector epilogue of this file stores through it; each
// output type keeps its own compile-time piece loop, so no packed copy of the 32 values has to stay live.
template <typename Store16>
__device__ __forceinline__ void pack_out32(const float (&v)[32], int out_dtype, Store16&& store16) {
    if (out_dtype == FP8B_F32) {
#pragma unroll
        for (int j = 0; j < 8; ++j)
            store16(j, __float_as_uint(v[4 * j]), __float_as_uint(v[4 * j + 1]), __float_as_uint(v[4 * j + 2]),
                    __float_as_uint(v[4 * j + 3]));
    } else if (out_dtype == FP8B_OUT_E4M3FN) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            uint32_t w[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int c = 16 * j + 4 * i;
                w[i] = enc4_f32(v[c], v[c + 1], v[c + 2], v[c + 3]);
            }
            store16(j, w[0], w[1], w[2], w[3]);
        }
    } else {
        uint32_t pk[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            if (out_dtype == FP8B_BF16) {
                __nv_bfloat162 b = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
                pk[j] = *reinterpret_cast<uint32_t*>(&b);
            } else {
                __half2 h = __floats2half2_rn(v[2 * j], v[2 * j + 1]);
                pk[j] = *reinterpret_cast<uint32_t*>(&h);
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) store16(j, pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
    }
}

// Cold paths of the epilogue, out of line and working on local-memory copies, so that they cost the hot loop neither
// instructions nor instruction-cache footprint (with the NaN fix-up inlined 32 times per chunk the 128 x 256 epilogue took
// 8 100 cycles, without it 6 800; with the term dispatch hoisted out of the tile loop as well, 3 700).
static __device__ __noinline__ void fix_nan_chunk(uint32_t* r, const uint8_t* a_row, const uint8_t* b_rows, int K, int n_left,
                                                  int a_fmt, int b_fmt) {
    for (int j = 0; j < 32 && j < n_left; ++j) {
        const float a = __uint_as_float(r[j]);
        if (a != a) r[j] = __float_as_uint(slow_dot_fmt(a_row, b_rows + (size_t)j * K, K, a_fmt, b_fmt));
    }
}
static __device__ __noinline__ void load_col_params_edge(const Epi& e, int n0, int N, float* sbv, float* bv) {
    for (int j = 0; j < 32; ++j) {
        const int n = n0 + j;
        const bool ok = n < N;
        sbv[j] = (e.sb_stride && ok) ? e.sb[n] : 0.0f;
        bv[j] = (e.bias && ok) ? epi_bias(e, n) : 0.0f;
    }
}

// ------------------------------------------------------------------------------ kernel

// Per-column epilogue parameters of one 32-column chunk, loaded while the TMEM load is in flight: one broadcast
// 16-byte load per 4 columns when the chunk is full and the arrays are aligned, guarded scalar loads at the N edge.
__device__ __forceinline__ void load_col_params(const Epi& e, int n0, int N, bool vec, float (&sbv)[32], float (&bv)[32]) {
    if (vec) {
        if (e.sb_stride) {
            const float4* s4 = reinterpret_cast<const float4*>(e.sb + n0);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 t = s4[j];
                sbv[4 * j] = t.x; sbv[4 * j + 1] = t.y; sbv[4 * j + 2] = t.z; sbv[4 * j + 3] = t.w;
            }
        }
        if (e.bias) {
            if (e.bias_dtype == FP8B_F32) {
                const float4* b4 = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(e.bias) + n0);
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float4 t = b4[j];
                    bv[4 * j] = t.x; bv[4 * j + 1] = t.y; bv[4 * j + 2] = t.z; bv[4 * j + 3] = t.w;
                }
            } else {
                const uint4* b4 = reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(e.bias) + n0);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint4 t = b4[j];
                    const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        if (e.bias_dtype == FP8B_BF16) {
                            bv[8 * j + 2 * i] = __uint_as_float(w[i] << 16);
                            bv[8 * j + 2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
                        } else {
                            const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
                            bv[8 * j + 2 * i] = f.x; bv[8 * j + 2 * i + 1] = f.y;
                        }
                    }
                }
            }
        }
    } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            const int n = n0 + j;
            const bool ok = n < N;
            sbv[j] = (e.sb_stride && ok) ? e.sb[n] : 0.0f;
            bv[j] = (e.bias && ok) ? epi_bias(e, n) : 0.0f;
        }
    }
}

// MODE (see the enum above) selects how tiles leave the SM.  kStPeers / kStTma are separate instantiations, so the
// single-GPU and multicast kernels are untouched by the multi-destination code.
template <int BN, int CG, int MODE = kStDirect>
__global__ void __launch_bounds__(gemm_threads<MODE>(), 1)
fp8_gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a,
                        const __grid_constant__ CUtensorMap tmap_b,
                        const __grid_constant__ typename StoreMapsOf<MODE>::type smaps,
                        const GemmParams p)
{
    using Cfg = GemmCfg<BN, CG, MODE>;
    constexpr bool PEERS = MODE == kStPeers;
#ifdef FP8B_PROFILE
    long long* const dbg = p.dbg;
#endif
    constexpr int kTileM = kBM * CG;                 // rows of C per tile (per CTA pair when CG == 2)
    const uint32_t cta_rank = (CG == 2) ? cluster_ctarank() : 0u;
    const bool is_leader = cta_rank == 0;
    const int worker = (CG == 2) ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;       // tile-loop index
    const int num_workers = (CG == 2) ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    extern __shared__ uint8_t gemm_smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(gemm_smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* bar_mem = smem + Cfg::kOffBar;
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t bar_base = smem_u32(bar_mem);
    // barrier slots (8 bytes each): full[kStages], empty[kStages], tmem_full[2], tmem_empty[2], sfull[slots], sfree[slots]
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::kStages + s); };
    auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * Cfg::kStages + a); };
    auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * Cfg::kStages + 2 + a); };
    auto sfull_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::kStages + 4 + s); };
    auto sfree_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::kStages + 4 + FP8B_TMA_SLOTS + s); };
    volatile uint32_t* tmem_slot =
        reinterpret_cast<volatile uint32_t*>(bar_mem + 8 * (2 * Cfg::kStages + 4 + 2 * FP8B_TMA_SLOTS));
    const uint32_t stage_base = smem_base + Cfg::kOffStaging;      // epilogue staging (1024-byte aligned)

    const int warp = __shfl_sync(0xFFFFFFFFu, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31;
#ifdef FP8B_PROFILE
    if (dbg && blockIdx.x == 0 && threadIdx.x == 0) dbg[7] = clock64();       // kernel entry
#endif

    // Programmatic dependent launch: let the kernel that follows on the stream become resident as soon as SMs free up
    // (push modes: fp8b_peer_wait, so that its launch latency is behind it when the peers' completion flags arrive; a
    // chain of GEMMs: the next one's barrier / TMEM / descriptor set-up).  It still waits -- griddepcontrol.wait below --
    // for this grid to complete before it touches global memory.
    pdl_launch_dependents();

    if (warp == kWarpTma && lane == 0) {
        tma_prefetch_desc(&tmap_a);
        tma_prefetch_desc(&tmap_b);
    }
    if (warp == kWarpMma && lane == 0) {
        for (int s = 0; s < Cfg::kStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), kNumEpiWarps * CG); }
        if (is_push<MODE>())
            for (int s = 0; s < FP8B_TMA_SLOTS; ++s) { mbar_init(sfull_bar(s), kNumEpiWarps); mbar_init(sfree_bar(s), 1); }
        fence_mbar_init();
        fence_proxy_async_smem();
    }
    if (warp == kWarpEpi0) {
        if (CG == 2) { tmem_alloc_2sm(smem_u32(const_cast<uint32_t*>(tmem_slot)), Cfg::kTmemCols); tmem_relinquish_2sm(); }
        else { tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), Cfg::kTmemCols); tmem_relinquish(); }
    }
    tc_fence_before();
    if (CG == 2) cluster_sync_all();      // the peer's barriers must be initialised before anything signals them
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // Everything above touched only this CTA's shared / tensor memory.  From here on the kernel reads A, B, the scales
    // and the bias and writes C: the predecessor on the stream must have completed (no-op without the PDL attribute).
    pdl_wait();

    const int num_tiles = p.num_work;

    if (warp == kWarpTma) {
        // ===================== TMA producer =====================
        // The whole warp runs the loop (uniform control flow); one elected lane issues the TMA traffic.
        {
            const bool elected = elect_one();
            int stage = 0; uint32_t phase = 0;
#ifdef FP8B_PROFILE
            int issued = 0;
#endif
            for (int tile = worker; tile < num_tiles; tile += num_workers) {
                const TileCoord tc = decode_tile(p, tile, BN);
                const int m_idx = tc.m_blk * kTileM + (int)cta_rank * kBM;
                // each CTA of a pair stages width/CG rows of B (a half-width tile still loads the full box; the
                // MMA reads only the rows it needs)
                const int n_idx = tc.n0 + (int)cta_rank * (tc.width / CG);
                for (int kb = 0; kb < p.num_k_blocks; ++kb) {
                    mbar_wait(empty_bar(stage), phase ^ 1);
                    const uint32_t a_dst = smem_base + stage * Cfg::kStageBytes;
                    if (elected) {
#ifdef FP8B_PROFILE
                        if ((p.debug & 32) && issued >= Cfg::kStages) {
                            // profiling only: no TMA traffic after the ring is primed (results are garbage)
                            if (is_leader) mbar_arrive(full_bar(stage));
                        } else
#endif
                        if (CG == 2) {
                            // both CTAs load their halves; all bytes are accounted on the leader's barrier
                            if (is_leader) mbar_arrive_expect_tx(full_bar(stage), (uint32_t)p.stage_tx * CG);
                            tma_load_2d_2sm(a_dst, &tmap_a, full_bar(stage), kb * kBK, m_idx);
                            tma_load_2d_2sm(a_dst + Cfg::kABytes, &tmap_b, full_bar(stage), kb * kBK, n_idx);
                        } else {
                            mbar_arrive_expect_tx(full_bar(stage), (uint32_t)p.stage_tx);
                            tma_load_2d(a_dst, &tmap_a, full_bar(stage), kb * kBK, m_idx);
                            tma_load_2d(a_dst + Cfg::kABytes, &tmap_b, full_bar(stage), kb * kBK, n_idx);
                        }
                    }
                    __syncwarp();
#ifdef FP8B_PROFILE
                    ++issued;
#endif
                    if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == kWarpMma) {
        // ===================== MMA issuer =====================
        // Whole warp in the loop, one elected lane issues.  The loop body is kept minimal: the issuing thread
        // shares a scheduler with an epilogue warp, and every instruction it needs per k-block is latency the
        // tensor pipe may have to absorb (measured: a 90-instruction body cost 15 % of MMA throughput).
        if (is_leader) {
            constexpr uint32_t idesc = make_idesc(kTileM, BN);
            const uint32_t idesc_fmt = (uint32_t)p.a_fmt << 7 | (uint32_t)p.b_fmt << 10;
            const bool elected = elect_one();
            const uint64_t desc_a0 = make_smem_desc(smem_base);
            const uint64_t desc_b0 = make_smem_desc(smem_base + Cfg::kABytes);
            constexpr uint64_t kDescStage = (uint64_t)(Cfg::kStageBytes >> 4);      // start-address field per stage
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int tile = worker; tile < num_tiles; tile += num_workers) {
#ifdef FP8B_PROFILE
                const long long t_m0 = (dbg && blockIdx.x == 0) ? clock64() : 0;
#endif
                mbar_wait(tempty_bar(acc), acc_phase ^ 1);           // epilogue has drained this accumulator
                tc_fence_after();
#ifdef FP8B_PROFILE
                const long long t_m1 = (dbg && blockIdx.x == 0) ? clock64() : 0;
#endif
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
                const uint32_t idesc_t = ((tile < p.full_tiles) ? idesc : make_idesc(kTileM, BN / 2)) | idesc_fmt;
                for (int kb = 0; kb < p.num_k_blocks; ++kb) {
                    mbar_wait(full_bar(stage), phase);               // TMA bytes have landed
                    tc_fence_after();
                    if (elected) {
                        const uint64_t adesc = desc_a0 + kDescStage * (uint64_t)stage;
                        const uint64_t bdesc = desc_b0 + kDescStage * (uint64_t)stage;
#pragma unroll
                        for (int k = 0; k < kBK / kUmmaK; ++k) {     // +2 in the address field = +32 bytes of K
                            if (CG == 2) umma_f8_2sm(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc_t, (uint32_t)((kb | k) != 0));
                            else umma_f8(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc_t, (uint32_t)((kb | k) != 0));
                        }
                        // smem slot free (in both CTAs of a pair) once these MMAs retire
                        if (CG == 2) umma_commit_2sm(empty_bar(stage)); else umma_commit(empty_bar(stage));
                    }
                    __syncwarp();
                    if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
                }
                if (elected) {
                    if (CG == 2) umma_commit_2sm(tfull_bar(acc)); else umma_commit(tfull_bar(acc));   // accumulator complete
#ifdef FP8B_PROFILE
                    if (dbg && blockIdx.x == 0) {
                        const int ti = (tile - worker) / num_workers;
                        if (ti < 64) { dbg[ti * 8 + 0] = t_m0; dbg[ti * 8 + 1] = t_m1; dbg[ti * 8 + 2] = clock64(); dbg[ti * 8 + 3] = 0; }
                    }
#endif
                }
                __syncwarp();
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else if (is_push<MODE>() && warp == kWarpStore) {
        // ===================== store issuer (kStTma) =====================
        // Walks the same (tile, box) sequence as the epilogue warps.  Per box: wait until the four epilogue warps
        // have filled the slot, issue the stores to every destination, commit; then recycle the slot whose stores have
        // finished READING shared memory (the writes themselves stay in flight).
        if constexpr (MODE == kStTma) {
            const bool elected = elect_one();
            const int esz = out_esz(p.epi.out_dtype);
            const int cols_per_box = 128 / esz;
            uint32_t seq = 0;
            for (int tile = worker; tile < num_tiles; tile += num_workers) {
                const TileCoord tc = decode_tile(p, tile, BN);
                const int m_idx = tc.m_blk * kTileM + (int)cta_rank * kBM;
                for (int c = 0; c < tc.width; c += cols_per_box) {
                    const int n_box = tc.n0 + c;
                    if (n_box >= p.N) break;                      // warp-uniform; the epilogue skips the same boxes
                    const uint32_t slot = seq % FP8B_TMA_SLOTS;
                    mbar_wait(sfull_bar(slot), (seq / FP8B_TMA_SLOTS) & 1);
                    if (elected) {
                        if (m_idx < p.M) {
                            const uint32_t src = stage_base + slot * kStoreBoxBytes;
                            for (int d = 0; d < p.n_dst; ++d) tma_store_2d(&smaps.m[d], src, n_box * esz, m_idx);
                        }
                        bulk_commit_group();
                        bulk_wait_group_read<kStoreInflight>();
                        if (seq >= (uint32_t)kStoreInflight) mbar_arrive(sfree_bar((seq - kStoreInflight) % FP8B_TMA_SLOTS));
                    }
                    __syncwarp();
                    ++seq;
                }
            }
            if (elected) bulk_wait_group_all();                   // all writes performed before the CTA retires
            __syncwarp();
#ifdef FP8B_PROFILE
            if (dbg && blockIdx.x == 0 && lane == 0) dbg[15] = clock64();         // stores complete
#endif
        }
    } else if (is_push<MODE>()) {
        // ===================== epilogue, store-ring flavour (warps 0..3) =====================
        // tcgen05.ld -> scale/bias -> out dtype -> a box in shared memory.  Lane = row, 128 bytes per row,
        // 16-byte piece j of row r at r*128 + ((j ^ (r & 7)) * 16) -- conflict-free st.shared.v4 and exactly the layout the
        // SWIZZLE_128B tensor map of the store expects.  Column/row edges need no code: TMA clips the box.
        if constexpr (is_push<MODE>()) {
            const int q = warp & 3;
            const int row_in_tile = q * 32 + lane;
            const Epi& e = p.epi;
            const int a_fmt = p.a_fmt, b_fmt = p.b_fmt;
            const float sr = e.sr ? *e.sr : 1.0f;
            const float sb0 = e.sb[0];
            const int esz = out_esz(e.out_dtype);
            const int cols_per_box = 128 / esz;
            const uint32_t row_off = (uint32_t)row_in_tile * 128u;
            uint32_t seq = 0;
            int acc = 0; uint32_t acc_phase = 0;
            // Software-pipelined: the tcgen05.ld of chunk c+1 is in flight while chunk c is scaled, packed and
            // staged (two register sets).  Which optional epilogue terms exist (KIND) is a compile-time constant of the
            // whole tile loop -- one of eight copies runs -- and the cold paths (NaN fix-up, ragged column edge) are out
            // of line, so the hot loop is short and contiguous: a 128 x 256 accumulator is drained in 4 900 cycles
            // instead of 8 100-12 000.  That matters where the epilogue is exposed: the last tile of every CTA, i.e.
            // all of a small problem.
            auto run_tiles = [&](auto kind_c) {
                constexpr int KIND = decltype(kind_c)::value;
                constexpr bool SBV = (KIND & 1) != 0, BIAS = (KIND & 2) != 0, SR = (KIND & 4) != 0;
                for (int tile = worker; tile < num_tiles; tile += num_workers) {
                    const TileCoord tc = decode_tile(p, tile, BN);
                    const int m_idx = tc.m_blk * kTileM + (int)cta_rank * kBM;
                    const int n_idx = tc.n0;
                    const int m = m_idx + row_in_tile;
                    const bool m_ok = m < p.M;
                    const float sa = e.sa[(size_t)(m_ok ? m : 0) * e.sa_stride];
                    const int nch = tc.width >> 5;                    // 32-column chunks in this tile (2..8), warp-uniform
#ifdef FP8B_PROFILE
                    const long long t_e0 = (dbg && blockIdx.x == 0 && warp == kWarpEpi0 && lane == 0) ? clock64() : 0;
#endif
                    mbar_wait(tfull_bar(acc), acc_phase);
                    tc_fence_after();
#ifdef FP8B_PROFILE
                    const long long t_e1 = (dbg && blockIdx.x == 0 && warp == kWarpEpi0 && lane == 0) ? clock64() : 0;
#endif
                    const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN);
                    auto release_acc = [&]() {                        // every tcgen05.ld of this accumulator has completed
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) { if (CG == 2) mbar_arrive_leader(tempty_bar(acc)); else mbar_arrive(tempty_bar(acc)); }
                    };
                    auto chunk = [&](int c0, uint32_t (&r)[32]) {
                        const int n0 = n_idx + c0;
                        const int n_box = n_idx + (c0 & ~(cols_per_box - 1));
                        if (n_box >= p.N) return;                     // whole box outside the matrix (warp-uniform): the store warp skips it too
                        const bool box_first = (c0 & (cols_per_box - 1)) == 0;
                        const bool box_last = ((c0 + 32) & (cols_per_box - 1)) == 0 || c0 + 32 == tc.width;
                        const uint32_t slot = seq % FP8B_TMA_SLOTS;
                        if (box_first) mbar_wait(sfree_bar(slot), ((seq / FP8B_TMA_SLOTS) & 1) ^ 1);
                        if (n0 < p.N) {
                            float sbv[32];
                            float bv[32];
                            if (SBV || BIAS) {
                                if ((n0 + 32 <= p.N) && p.col_vec_ok) {
                                    load_col_params(e, n0, p.N, true, sbv, bv);
                                } else {                              // ragged edge / unaligned arrays (cold)
                                    float t_sb[32], t_b[32];
                                    load_col_params_edge(e, n0, p.N, t_sb, t_b);
#pragma unroll
                                    for (int j = 0; j < 32; ++j) { sbv[j] = t_sb[j]; bv[j] = t_b[j]; }
                                }
                            }
                            // NaN-byte fix-up (cold): a NaN accumulator can only come from a 0x7F/0xFF operand byte
                            if (__any_sync(0xFFFFFFFFu, m_ok && any_nan32(r))) {
                                uint32_t t[32];
#pragma unroll
                                for (int j = 0; j < 32; ++j) t[j] = r[j];
                                if (m_ok) fix_nan_chunk(t, p.A + (size_t)m * p.K, p.B + (size_t)n0 * p.K, p.K, p.N - n0,
                                                        a_fmt, b_fmt);
#pragma unroll
                                for (int j = 0; j < 32; ++j) r[j] = t[j];
                            }
                            float v[32];
                            epi_math32<SBV, BIAS, SR>(r, sa, sb0, sr, sbv, bv, v);
                            const uint32_t dst = stage_base + slot * kStoreBoxBytes + row_off;
                            const uint32_t sw = (uint32_t)(lane & 7);
                            // first 16-byte piece of this chunk inside the box row
                            const uint32_t piece0 = (uint32_t)(((c0 & (cols_per_box - 1)) * esz) >> 4);
                            pack_out32(v, e.out_dtype, [&](int j, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3) {
                                sts_v4(dst + (((piece0 + (uint32_t)j) ^ sw) << 4), w0, w1, w2, w3);
                            });
                        }
                        if (box_last) {
                            fence_proxy_async_smem();   // generic-proxy writes -> visible to the TMA (async proxy)
                            __syncwarp();
                            if (lane == 0) mbar_arrive(sfull_bar(slot));
                            ++seq;
                        }
                    };
                    uint32_t ra[32], rb[32];
                    __syncwarp();
                    tmem_ld_x32(t_row, ra);
#pragma unroll 1
                    for (int ch = 0; ch < nch; ch += 2) {
                        __syncwarp();                   // lanes may have diverged in chunk() (row mask, NaN fix-up);
                        tmem_ld_wait_for(ra);           // tcgen05.wait / .ld are warp-collective (.sync.aligned)
                        if (ch + 1 < nch) tmem_ld_x32(t_row + (uint32_t)((ch + 1) * 32), rb); else release_acc();
                        chunk(ch * 32, ra);
                        if (ch + 1 < nch) {
                            __syncwarp();
                            tmem_ld_wait_for(rb);
                            if (ch + 2 < nch) tmem_ld_x32(t_row + (uint32_t)((ch + 2) * 32), ra); else release_acc();
                            chunk((ch + 1) * 32, rb);
                        }
                    }
#ifdef FP8B_PROFILE
                    if (dbg && blockIdx.x == 0 && warp == kWarpEpi0 && lane == 0) {
                        const int ti = (tile - worker) / num_workers;
                        if (ti < 64) { dbg[ti * 8 + 4] = t_e0; dbg[ti * 8 + 5] = t_e1; dbg[ti * 8 + 6] = clock64(); }
                        dbg[23] = clock64();                                   // last epilogue end so far
                    }
#endif
                    if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                }
            };
            switch ((e.sb_stride ? 1 : 0) | (e.bias ? 2 : 0) | (e.sr ? 4 : 0)) {          // grid-uniform
                case 0: run_tiles(std::integral_constant<int, 0>{}); break;
                case 1: run_tiles(std::integral_constant<int, 1>{}); break;
                case 2: run_tiles(std::integral_constant<int, 2>{}); break;
                case 3: run_tiles(std::integral_constant<int, 3>{}); break;
                case 4: run_tiles(std::integral_constant<int, 4>{}); break;
                case 5: run_tiles(std::integral_constant<int, 5>{}); break;
                case 6: run_tiles(std::integral_constant<int, 6>{}); break;
                default: run_tiles(std::integral_constant<int, 7>{}); break;
            }
        }
    } else {
        // ===================== epilogue (warps 0..3) =====================
        const int q = warp & 3;                       // TMEM lane quarter this warp may read (warp id % 4)
        const int col_part = (warp - kWarpEpi0) >> 2;         // which slice of the tile's columns this warp drains
        const int row_in_tile = q * 32 + lane;
        const Epi& e = p.epi;
        const float sr = e.sr ? *e.sr : 1.0f;
        const float sb0 = e.sb[0];
        long long peer_delta[8];                     // PEERS: byte offset of every rank's buffer from the local one (0 = self)
        const int peer_world = PEERS ? p.n_dst : 0;
        if (PEERS) {
#pragma unroll
            for (int r = 0; r < 8; ++r) peer_delta[r] = r < peer_world ? p.peer_delta[r] : 0;
        }
        auto store16 = [&](void* ptr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
            if (PEERS) {
#pragma unroll
                for (int r = 0; r < 8; ++r)
                    if (r < peer_world) stg_v4(reinterpret_cast<uint8_t*>(ptr) + peer_delta[r], a, b, c, d, 0);
            } else {
                stg_v4(ptr, a, b, c, d, p.multicast);
            }
        };
        int acc = 0; uint32_t acc_phase = 0;
        for (int tile = worker; tile < num_tiles; tile += num_workers) {
            const TileCoord tc = decode_tile(p, tile, BN);
            const int m_idx = tc.m_blk * kTileM + (int)cta_rank * kBM;
            const int n_idx = tc.n0;
            const int cols_per_warp = tc.width / kEpiColSplits;      // BN / splits, or half of it in the split last wave
            const int m = m_idx + row_in_tile;
            const bool m_ok = m < p.M;
            const float sa = e.sa[(size_t)(m_ok ? m : 0) * e.sa_stride];
#ifdef FP8B_PROFILE
            const long long t_e0 = (dbg && blockIdx.x == 0 && warp == kWarpEpi0 && lane == 0) ? clock64() : 0;
#endif
            mbar_wait(tfull_bar(acc), acc_phase);
            tc_fence_after();
#ifdef FP8B_PROFILE
            const long long t_e1 = (dbg && blockIdx.x == 0 && warp == kWarpEpi0 && lane == 0) ? clock64() : 0;
#endif
            const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN);
#pragma unroll 1
            for (int c0 = col_part * cols_per_warp; c0 < (col_part + 1) * cols_per_warp; c0 += 32) {
                uint32_t r[32];
                __syncwarp();                         // lanes may have diverged on the row/column masks below
                tmem_ld_x32(t_row + c0, r);
                const int n0 = n_idx + c0;
                const bool full_chunk = (n0 + 32 <= p.N) && p.col_vec_ok;      // warp-uniform
                float sbv[32];
                float bv[32];
                if (full_chunk) load_col_params(e, n0, p.N, true, sbv, bv);
                tmem_ld_wait();
                if (c0 + 32 == (col_part + 1) * cols_per_warp) {   // this warp's last read of the accumulator: hand it back early
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) { if (CG == 2) mbar_arrive_leader(tempty_bar(acc)); else mbar_arrive(tempty_bar(acc)); }
                }
                if (n0 >= p.N) continue;              // warp-uniform
                if (FP8B_DBG(p, 2)) continue;

                // NaN-byte fix-up (cold): a NaN accumulator can only come from a 0x7F/0xFF operand byte
                float nan_probe = 0.0f;
#pragma unroll
                for (int j = 0; j < 32; ++j) nan_probe += __uint_as_float(r[j]);
                if (__any_sync(0xFFFFFFFFu, m_ok && nan_probe != nan_probe)) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float a = __uint_as_float(r[j]);
                        if (a != a && m_ok && n0 + j < p.N)
                            r[j] = __float_as_uint(slow_dot_fmt(p.A + (size_t)m * p.K, p.B + (size_t)(n0 + j) * p.K, p.K,
                                                                p.a_fmt, p.b_fmt));
                    }
                }
                if (full_chunk && p.vec_store_ok) {
                    float v[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        float x = __fmul_rn(__uint_as_float(r[j]), sa);
                        x = __fmul_rn(x, e.sb_stride ? sbv[j] : sb0);
                        if (e.bias) x = __fadd_rn(x, bv[j]);
                        if (e.sr) x = __fmul_rn(x, sr);
                        v[j] = x;
                    }
                    const int esz = out_esz(e.out_dtype);
                    const int ppc = 2 * esz;                             // 16-byte pieces per chunk per row: 8, 4 or 2
                    // Row groups of 256 bytes (256 e4m3fn, 128 16-bit or 64 fp32 columns) are staged through a per-warp
                    // XOR-swizzled shared-memory tile and written out with 16 lanes per row, so every
                    // store instruction covers 2 rows x 256 contiguous bytes (full 128-byte lines) -- for
                    // local HBM and, in multicast mode, for NVLink, where 16-byte-per-row scatter is fatal.
                    // chunks per row group: 256-byte row segments when the warp's column span allows it, else 128-byte
                    const int cpg_max = 8 / esz;
                    const int cpg = (cols_per_warp % (cpg_max * 32) == 0) ? cpg_max : cpg_max / 2;
                    const int ppr = cpg * ppc;                           // 16-byte pieces per staged row: 16 or 8
                    const int rel = (c0 - col_part * cols_per_warp) >> 5; // chunk index inside this warp's span
                    const int cg = rel & (cpg - 1);                      // chunk index inside its group
                    const int ng0 = n0 - cg * 32;                        // first column of the group
                    const bool staged = !FP8B_DBG(p, 1 | 4) && (ng0 + cpg * 32 <= p.N) &&
                                        ((rel - cg + cpg) * 32 <= cols_per_warp);   // warp-uniform; the whole group lies in this warp's span
                    if (staged) {
                        const uint32_t wbase = stage_base + (uint32_t)(warp - kWarpEpi0) * 8192u;
                        const uint32_t row_bytes = (uint32_t)ppr * 16u;
                        pack_out32(v, e.out_dtype, [&](int j, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3) {
                            const uint32_t phys = (uint32_t)((cg * ppc + j) ^ (lane & (ppr - 1)));
                            sts_v4(wbase + (uint32_t)lane * row_bytes + phys * 16u, w0, w1, w2, w3);
                        });
                        if (cg == cpg - 1) {
                            __syncwarp();
                            const int piece = lane & (ppr - 1);
                            const int rows_per_inst = 32 / ppr;          // 2 (256-byte rows) or 4 (128-byte rows)
                            uint8_t* cbase = reinterpret_cast<uint8_t*>(e.C) + (size_t)ng0 * esz + (size_t)piece * 16;
#pragma unroll 4
                            for (int i = 0; i < 32 / rows_per_inst; ++i) {
                                const int rr = rows_per_inst * i + lane / ppr;
                                const int gm = m_idx + q * 32 + rr;
                                uint32_t a0, a1, a2, a3;
                                lds_v4(wbase + (uint32_t)rr * row_bytes + (uint32_t)((piece ^ (rr & (ppr - 1))) * 16), a0, a1, a2, a3);
                                if (gm < p.M) store16(cbase + (size_t)gm * e.ldc * esz, a0, a1, a2, a3);
                            }
                            __syncwarp();
                        }
                    } else if (m_ok && !FP8B_DBG(p, 1)) {
                        uint8_t* dst = reinterpret_cast<uint8_t*>(e.C) + ((size_t)m * e.ldc + n0) * esz;
                        pack_out32(v, e.out_dtype, [&](int j, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3) {
                            store16(dst + 16 * j, w0, w1, w2, w3);
                        });
                    }
                } else if (m_ok) {
                    // edge chunk / unaligned output: scalar, bounds-checked
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const int n = n0 + j;
                        if (n < p.N) epi_store(e, m, n, epi_apply(e, __uint_as_float(r[j]), m, n));
                    }
                }
            }
#ifdef FP8B_PROFILE
            if (dbg && blockIdx.x == 0 && warp == kWarpEpi0 && lane == 0) {
                const int ti = (tile - worker) / num_workers;
                if (ti < 64) { dbg[ti * 8 + 4] = t_e0; dbg[ti * 8 + 5] = t_e1; dbg[ti * 8 + 6] = clock64(); }
            }
#endif
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }

    tc_fence_before();
    // Neither CTA of a pair may exit (or free TMEM) while its peer still signals it.  The store-ring modes keep the
    // release / acquire flavour -- the completion signal below is published by another thread than the one that waited for
    // the bulk stores, and nothing generic is pending there anyway; with st.global epilogues an execution-only barrier
    // spares the wait for every store of the last tile to be acknowledged.
    if (CG == 2) { if (is_push<MODE>()) cluster_sync_all(); else cluster_sync_relaxed(); }
    else __syncthreads();
#ifdef FP8B_PROFILE
    if (dbg && blockIdx.x == 0 && threadIdx.x == 0) dbg[31] = clock64();          // CTA end
#endif
    if (warp == kWarpEpi0) {
        tc_fence_after();
        if (CG == 2) tmem_dealloc_2sm(tmem_base, Cfg::kTmemCols); else tmem_dealloc(tmem_base, Cfg::kTmemCols);
    }
    if constexpr (is_push<MODE>()) {
        // Completion signal (fused closing barrier, send side).  Every store warp has waited for its bulk groups
        // (writes performed) before the CTA-wide barrier above.  One thread per CTA publishes that system-wide and
        // counts the CTA in; the last CTA of the grid tells every peer, with a release store into the PEER's flag word,
        // that all of this rank's boxes have landed.  fp8b_peer_wait on the peer acquires that flag.
        if (smaps.n_sig > 0 && threadIdx.x == 0) {
            asm volatile("fence.proxy.async;" ::: "memory");               // async-proxy (TMA) writes before generic-proxy signalling
            __threadfence_system();
            const unsigned int done = atomicAdd(smaps.cta_counter, 1u) + 1u;
            if (done == gridDim.x) {
                __threadfence_system();
                *smaps.cta_counter = 0u;                                     // ready for the next launch (stream-ordered)
                for (int d = 0; d < smaps.n_sig; ++d)
                    if (smaps.sig[d])
                        asm volatile("st.release.sys.global.u64 [%0], %1;" :: "l"(smaps.sig[d]), "l"(smaps.epoch) : "memory");
            }
        }
    }
}

// ------------------------------------------------------------------------------ split-K kernel (few tiles, long K)
//
// A problem with fewer 128 x 128 tiles than SMs leaves most of the GPU idle and every busy SM walks the whole of K alone
// (M = 32, K = N = 3072: 24 CTAs, 6 100 cycles of MMAs each).  Here a thread-block CLUSTER of S CTAs shares one tile: CTA r
// accumulates k-blocks [r, r+1) * KB / S into its own TMEM accumulator, then the cluster reduce-scatters over distributed
// shared memory -- CTA r sends column slice j of its partial tile to CTA j (bulk copies, shared memory to the peer's shared
// memory) and receives slice r of every partial -- and each CTA sums its slice in rank order (deterministic), applies the
// epilogue and stores it.  The reduction costs 64 KB of DSMEM traffic per CTA and spreads the epilogue over the S CTAs.
//   warps 0..3 epilogue (TMEM lane quarter = warp id), warp 4 TMA producer, warp 5 MMA issuer; one tile per cluster.
constexpr int kSkStages = 5;
constexpr int kSkStageBytes = 2 * kBM * kBK;                     // A 128 x 128 B + B 128 x 128 B
constexpr int kSkRecvBytes = kBM * 128 * 4;                      // S slots x 128 rows x (128 / S) fp32 columns = 64 KB
constexpr int kSkBarBytes = 128;
constexpr int kSkSmemBytes = kSkStages * kSkStageBytes + kSkRecvBytes + kSkBarBytes + 1024;
constexpr int kSkThreads = 192;

struct SplitKParams {
    const uint8_t* A; const uint8_t* B;      // for the NaN fix-up only
    int M, N, K;
    int num_n_blocks, num_k_blocks;
    int stage_tx;                            // bytes the two TMA loads of a stage deliver
    uint32_t idesc;                          // instruction descriptor incl. operand formats
    int a_fmt, b_fmt;
    Epi epi;
    int vec_store_ok;                        // C base and ldc allow 16-byte stores
    int col_vec_ok;                          // scale_b / bias bases allow 16-byte broadcast loads
    long long* dbg;                          // FP8B_PROFILE builds: clock stamps of CTA 0 (else null)
};

__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_smem_addr, uint32_t cta_rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(cta_rank));
    return r;
}
// shared memory of this CTA -> shared memory of a CTA of the cluster, completion counted in bytes on THAT CTA's mbarrier
__device__ __forceinline__ void bulk_copy_to_cta(uint32_t dst_cluster_addr, uint32_t src_local_addr, uint32_t bytes,
                                                 uint32_t cluster_bar_addr) {
    asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst_cluster_addr), "r"(src_local_addr), "r"(bytes), "r"(cluster_bar_addr) : "memory");
}
// ragged column edge / unaligned output: element-wise, bounds-checked (cold)
static __device__ __noinline__ void store_row_edge(const Epi& e, int m, int n0, int N, const float* v) {
    for (int j = 0; j < 32; ++j)
        if (n0 + j < N) epi_store(e, m, n0 + j, v[j]);
}
template <int S>
__global__ void __launch_bounds__(kSkThreads, 1)
fp8_gemm_splitk_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, const SplitKParams p)
{
    constexpr int kSlice = 128 / S;                  // output columns this CTA finishes
    static_assert(S == 2 || S == 4, "slices must be whole 32-column TMEM chunks (and >= 8 16-byte pieces per row for the swizzle)");
    extern __shared__ uint8_t gemm_smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(gemm_smem_raw) + 1023) & ~(uintptr_t)1023);
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t recv_base = smem_base + kSkStages * kSkStageBytes;
    const uint32_t bar_base = recv_base + kSkRecvBytes;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (kSkStages + s); };
    const uint32_t tfull_bar = bar_base + 8u * (2 * kSkStages);
    auto recv_bar = [&](int q) { return bar_base + 8u * (2 * kSkStages + 1 + q); };
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + kSkStages * kSkStageBytes + kSkRecvBytes + 8 * (2 * kSkStages + 5));

    const int warp = __shfl_sync(0xFFFFFFFFu, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int tile = (int)(blockIdx.x / S);
    const int n_blk = tile % p.num_n_blocks, m_blk = tile / p.num_n_blocks;
    const int m_idx = m_blk * kBM, n_idx = n_blk * 128;
    const int kb0 = (int)(((long long)p.num_k_blocks * rank) / S), kb1 = (int)(((long long)p.num_k_blocks * (rank + 1)) / S);

    pdl_launch_dependents();
#ifdef FP8B_PROFILE
    const bool stamp = p.dbg && blockIdx.x == 0 && threadIdx.x == 0;
    if (stamp) p.dbg[0] = clock64();
#endif
    if (warp == 4 && lane == 0) { tma_prefetch_desc(&tmap_a); tma_prefetch_desc(&tmap_b); }
    if (warp == 5 && lane == 0) {
        for (int s = 0; s < kSkStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        mbar_init(tfull_bar, 1);
        for (int q = 0; q < 4; ++q) mbar_init(recv_bar(q), 1);
        fence_mbar_init();
        // each receive barrier completes when warp q's block of every CTA of the cluster (S x 32 rows x kSlice fp32) has landed
        for (int q = 0; q < 4; ++q) mbar_arrive_expect_tx(recv_bar(q), (uint32_t)(S * 32 * kSlice * 4));
        fence_proxy_async_smem();
    }
    if (warp == 0) { tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), 128); tmem_relinquish(); }
    tc_fence_before();
    cluster_sync_all();                              // the peers' barriers exist before anybody arrives on them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();                                      // the predecessor on the stream has completed: global memory may be touched
#ifdef FP8B_PROFILE
    if (stamp) p.dbg[1] = clock64();
#endif

    if (warp == 4) {
        const bool elected = elect_one();
        int stage = 0; uint32_t phase = 0;
        for (int kb = kb0; kb < kb1; ++kb) {
            mbar_wait(empty_bar(stage), phase ^ 1);
            if (elected) {
                const uint32_t dst = smem_base + stage * kSkStageBytes;
                mbar_arrive_expect_tx(full_bar(stage), (uint32_t)p.stage_tx);
                tma_load_2d(dst, &tmap_a, full_bar(stage), kb * kBK, m_idx);
                tma_load_2d(dst + kBM * kBK, &tmap_b, full_bar(stage), kb * kBK, n_idx);
            }
            __syncwarp();
            if (++stage == kSkStages) { stage = 0; phase ^= 1; }
        }
    } else if (warp == 5) {
        const bool elected = elect_one();
        const uint64_t desc_a0 = make_smem_desc(smem_base);
        const uint64_t desc_b0 = make_smem_desc(smem_base + kBM * kBK);
        constexpr uint64_t kDescStage = (uint64_t)(kSkStageBytes >> 4);
        int stage = 0; uint32_t phase = 0;
        for (int kb = kb0; kb < kb1; ++kb) {
            mbar_wait(full_bar(stage), phase);
            tc_fence_after();
            if (elected) {
                const uint64_t adesc = desc_a0 + kDescStage * (uint64_t)stage, bdesc = desc_b0 + kDescStage * (uint64_t)stage;
#pragma unroll
                for (int k = 0; k < kBK / kUmmaK; ++k)
                    umma_f8(tmem_base, adesc + 2 * k, bdesc + 2 * k, p.idesc, (uint32_t)((kb != kb0) | (k != 0)));
                umma_commit(empty_bar(stage));
            }
            __syncwarp();
            if (++stage == kSkStages) { stage = 0; phase ^= 1; }
        }
        if (elected) umma_commit(tfull_bar);
        __syncwarp();
    } else {
        // ===================== epilogue warps: reduce-scatter over DSMEM, then finish this CTA's column slice =====================
        // Scatter: the partial tile is staged in the (now idle) operand ring as [destination CTA][warp][32 rows][kSlice fp32]
        // and every (warp, destination) block -- 32 * kSlice * 4 contiguous bytes -- travels as ONE bulk copy, shared memory
        // to the peer's shared memory, completing on the PEER's mbarrier.  (Per-lane st.shared::cluster of 16 bytes was
        // measured at 2 400 cycles per 32-column chunk: every lane writes a different row, nothing coalesces.)
        const int q = warp;                           // TMEM lane quarter
        const int row = q * 32 + lane;
        const int m = m_idx + row;
        const bool m_ok = m < p.M;
        const Epi& e = p.epi;
        const uint32_t sw = (uint32_t)(lane & 7);
        constexpr uint32_t kBlockBytes = 32u * kSlice * 4u;                   // one warp's rows of one slice
        const uint32_t lane_off = (uint32_t)lane * (uint32_t)(kSlice * 4);
        mbar_wait(tfull_bar, 0);                      // every MMA of this CTA has retired: TMEM complete, operand ring idle
        tc_fence_after();
#ifdef FP8B_PROFILE
        if (stamp) p.dbg[2] = clock64();
#endif
        const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16);
        // (destinations in the order rank+1, rank+2, ..., rank: every CTA of the cluster receives its blocks at about the
        // same time instead of CTA 0 first and CTA S-1 a whole scatter later)
#pragma unroll 1
        for (int i = 0; i < 128; i += 32) {
            const int c0 = (i + ((int)rank + 1) * kSlice) & 127;
            uint32_t r[32];
            __syncwarp();
            tmem_ld_x32(t_row + (uint32_t)c0, r);
            tmem_ld_wait_for(r);
            const uint32_t dst_cta = (uint32_t)(c0 / kSlice);
            const uint32_t blk = smem_base + (dst_cta * 4u + (uint32_t)q) * kBlockBytes;      // send[dst][q]
            const uint32_t piece0 = (uint32_t)((c0 % kSlice) >> 2);
#pragma unroll
            for (int j = 0; j < 8; ++j)
                sts_v4(blk + lane_off + (((piece0 + j) ^ sw) << 4), r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
            if ((c0 + 32) % kSlice == 0) {            // the block for dst_cta is complete: ship it
                fence_proxy_async_smem();             // generic-proxy writes -> visible to the bulk copy (async proxy)
                __syncwarp();
                if (lane == 0)
                    bulk_copy_to_cta(map_to_cta(recv_base + (rank * 4u + (uint32_t)q) * kBlockBytes, dst_cta), blk, kBlockBytes,
                                     map_to_cta(recv_bar(q), dst_cta));
            }
        }
#ifdef FP8B_PROFILE
        if (stamp) p.dbg[3] = clock64();
#endif
        // gather: block [s][q] of every CTA s of the cluster (this one included) has landed in recv[s][q]
        mbar_wait(recv_bar(q), 0);
#ifdef FP8B_PROFILE
        if (stamp) p.dbg[4] = clock64();
#endif
        const float sa = e.sa[(size_t)(m_ok ? m : 0) * e.sa_stride];
        const float sr = e.sr ? *e.sr : 1.0f;
        const float sb0 = e.sb[0];
        const int esz = out_esz(e.out_dtype);
        const int kind = (e.sb_stride ? 1 : 0) | (e.bias ? 2 : 0) | (e.sr ? 4 : 0);
#pragma unroll 1
        for (int c0 = 0; c0 < kSlice; c0 += 32) {
            const int n0 = n_idx + (int)rank * kSlice + c0;
            if (n0 >= p.N) break;                     // warp-uniform
            uint32_t acc[32];
#pragma unroll
            for (int s2 = 0; s2 < S; ++s2) {          // rank order: the sum is the same on every run
                const uint32_t src = recv_base + ((uint32_t)s2 * 4u + (uint32_t)q) * kBlockBytes + lane_off;
                const uint32_t piece0 = (uint32_t)(c0 >> 2);
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    uint32_t a0, a1, a2, a3;
                    lds_v4(src + (((piece0 + j) ^ sw) << 4), a0, a1, a2, a3);
                    if (s2 == 0) {
                        acc[4 * j] = a0; acc[4 * j + 1] = a1; acc[4 * j + 2] = a2; acc[4 * j + 3] = a3;
                    } else {
                        acc[4 * j] = __float_as_uint(__fadd_rn(__uint_as_float(acc[4 * j]), __uint_as_float(a0)));
                        acc[4 * j + 1] = __float_as_uint(__fadd_rn(__uint_as_float(acc[4 * j + 1]), __uint_as_float(a1)));
                        acc[4 * j + 2] = __float_as_uint(__fadd_rn(__uint_as_float(acc[4 * j + 2]), __uint_as_float(a2)));
                        acc[4 * j + 3] = __float_as_uint(__fadd_rn(__uint_as_float(acc[4 * j + 3]), __uint_as_float(a3)));
                    }
                }
            }
            const bool full = (n0 + 32 <= p.N);
            float sbv[32];
            float bv[32];
            if (kind & 3) {
                if (full && p.col_vec_ok) {
                    load_col_params(e, n0, p.N, true, sbv, bv);
                } else {                              // ragged edge / unaligned arrays (cold)
                    float t_sb[32], t_b[32];
                    load_col_params_edge(e, n0, p.N, t_sb, t_b);
#pragma unroll
                    for (int j = 0; j < 32; ++j) { sbv[j] = t_sb[j]; bv[j] = t_b[j]; }
                }
            }
            // NaN-byte fix-up (cold): recompute the element over the whole of K with the reference's masked decode
            if (__any_sync(0xFFFFFFFFu, m_ok && any_nan32(acc))) {
                uint32_t t[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) t[j] = acc[j];
                if (m_ok) fix_nan_chunk(t, p.A + (size_t)m * p.K, p.B + (size_t)n0 * p.K, p.K, p.N - n0, p.a_fmt, p.b_fmt);
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[j] = t[j];
            }
            float v[32];
            switch (kind) {                           // grid-uniform
                case 0: epi_math32<false, false, false>(acc, sa, sb0, sr, sbv, bv, v); break;
                case 1: epi_math32<true, false, false>(acc, sa, sb0, sr, sbv, bv, v); break;
                case 2: epi_math32<false, true, false>(acc, sa, sb0, sr, sbv, bv, v); break;
                case 3: epi_math32<true, true, false>(acc, sa, sb0, sr, sbv, bv, v); break;
                case 4: epi_math32<false, false, true>(acc, sa, sb0, sr, sbv, bv, v); break;
                case 5: epi_math32<true, false, true>(acc, sa, sb0, sr, sbv, bv, v); break;
                case 6: epi_math32<false, true, true>(acc, sa, sb0, sr, sbv, bv, v); break;
                default: epi_math32<true, true, true>(acc, sa, sb0, sr, sbv, bv, v); break;
            }
            if (!m_ok) continue;
            if (full && p.vec_store_ok) {
                uint8_t* dst = reinterpret_cast<uint8_t*>(e.C) + ((size_t)m * e.ldc + n0) * esz;
                pack_out32(v, e.out_dtype, [&](int j, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3) {
                    stg_v4(dst + 16 * j, w0, w1, w2, w3, 0);
                });
            } else {
                float t[32];                          // (a local copy: v itself stays in registers on the hot path)
#pragma unroll
                for (int j = 0; j < 32; ++j) t[j] = v[j];
                store_row_edge(e, m, n0, p.N, t);
            }
        }
    }
    // Nobody writes into this CTA's shared memory any more: its own gather has seen every peer's arrival.  A CTA's
    // own remote stores and arrives precede its gather wait only in program order, so all CTAs leave together.
#ifdef FP8B_PROFILE
    if (stamp) p.dbg[5] = clock64();
#endif
    tc_fence_before();
    cluster_sync_relaxed();               // (data moved under mbarriers; this only keeps every CTA's shared memory alive)
#ifdef FP8B_PROFILE
    if (stamp) p.dbg[6] = clock64();
#endif
    if (warp == 0) { tc_fence_after(); tmem_dealloc(tmem_base, 128); }
}

// Receive side of the fused closing barrier: returns (completes) when every peer's flag has reached `epoch`, i.e. every
// peer's push kernel has finished writing into this rank's buffer -- and, through griddepcontrol.wait, when this rank's own
// push kernel (its predecessor on the stream) has completed.  Launched with the PDL attribute: it is resident and
// polling long before the flags arrive.  A peer that never signals trips the watchdog instead of hanging the GPU.
__global__ void fp8_peer_wait_kernel(const unsigned long long* __restrict__ flags, int world, int rank, unsigned long long epoch)
{
    const int r = threadIdx.x;
    if (r < world && r != rank) {
        unsigned long long t0 = 0, v = 0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        unsigned int spins = 0;
        for (;;) {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flags + r) : "memory");
            if (v >= epoch) break;
            if ((++spins & 0xFFF) == 0) {
                unsigned long long t1;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                if (t1 - t0 > 20000000000ull) __trap();                      // 20 s
            }
        }
    }
    __syncthreads();
    pdl_wait();                                                              // our own push kernel has completed and flushed
}


// ------------------------------------------------------------------------------ host side

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

typedef CUresult (*PFN_ctxGetCurrent)(CUcontext*);

static void* driver_fn(const char* name)
{
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    return cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess ? p
                                                                                                                             : nullptr;
}

static PFN_encodeTiled get_encode_fn()
{
    static PFN_encodeTiled fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] { fn = reinterpret_cast<PFN_encodeTiled>(driver_fn("cuTensorMapEncodeTiled")); });
    return fn;
}

// The encoder is a driver call and needs a current context.  A host thread whose first call into the library finds its
// kernel attribute already set (by another thread) has made no runtime call that binds one -- cudaGetDevice does not --
// and the encode then fails with CUDA_ERROR_INVALID_CONTEXT (seen on a B200 with six threads starting together).  A
// thread without a current context gets the current device's primary context, as the runtime's own calls would give
// it; a context the caller made current is left alone.
static cudaError_t ensure_current_context()
{
    static PFN_ctxGetCurrent get_current = nullptr;
    static std::once_flag once;
    std::call_once(once, [] { get_current = reinterpret_cast<PFN_ctxGetCurrent>(driver_fn("cuCtxGetCurrent")); });
    CUcontext ctx = nullptr;
    if (get_current && get_current(&ctx) == CUDA_SUCCESS && ctx) return cudaSuccess;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    return e == cudaSuccess ? cudaSetDevice(dev) : e;        // cudaSetDevice makes the primary context current
}

// A tensor map is a pure function of (base, rows, row bytes, pitch, box): a serving loop calls the same few
// weights and buffers over and over, so the encoded maps are kept in a small per-thread direct-mapped cache (the
// analogue of the reference bridge's one-time pipeline cache, fp8_bridge.cpp:103-141).  A map holds only addresses
// and extents, never data, so a stale entry for a freed-and-reallocated pointer with the same geometry is still right.
struct MapKey {
    const void* base; uint64_t rows, row_bytes, pitch; uint32_t box_rows, box_bytes;
    bool operator==(const MapKey& o) const {
        return base == o.base && rows == o.rows && row_bytes == o.row_bytes && pitch == o.pitch &&
               box_rows == o.box_rows && box_bytes == o.box_bytes;
    }
};
struct MapSlot { MapKey key; CUtensorMap map; bool valid; };
constexpr int kMapCacheSlots = 64;

// rows x row_bytes uint8 matrix with a row pitch, box = box_rows x box_bytes (<= 128), 128B swizzle.
static bool get_tensor_map(CUtensorMap* out, const void* base, uint64_t rows, uint64_t row_bytes, uint64_t pitch,
                           uint32_t box_rows, uint32_t box_bytes)
{
    static thread_local MapSlot cache[kMapCacheSlots];
    const MapKey key = {base, rows, row_bytes, pitch, box_rows, box_bytes};
    uint64_t h = reinterpret_cast<uintptr_t>(base) >> 4;
    h ^= rows * 0x9E3779B97F4A7C15ull; h ^= row_bytes * 0xC2B2AE3D27D4EB4Full; h ^= pitch << 7; h ^= (uint64_t)box_rows << 40;
    h ^= h >> 29;
    MapSlot& s = cache[h % kMapCacheSlots];
    if (s.valid && s.key == key) { *out = s.map; return true; }
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) { t_last_cuda_error = (int)cudaErrorSymbolNotFound; return false; }
    if (cudaError_t e = ensure_current_context()) { t_last_cuda_error = (int)e; return false; }
    cuuint64_t dims[2] = {(cuuint64_t)row_bytes, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)pitch};
    cuuint32_t box[2] = {(cuuint32_t)box_bytes, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base),
                     dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { t_last_cuda_error = (int)r; return false; }       // a CUresult (fp8b_last_cuda_error)
    s.key = key; s.map = *out; s.valid = true;
    return true;
}

// operand: rows x K bytes, row-major; box = box_rows x 128 bytes
static bool encode_operand_map(CUtensorMap* map, const uint8_t* base, int rows, int K, int box_rows)
{
    return get_tensor_map(map, base, (uint64_t)rows, (uint64_t)K, (uint64_t)K, (uint32_t)box_rows, (uint32_t)kBK);
}

bool tcgen05_supported(const MMArgs& a)
{
    // TMA: 16-byte aligned bases and a row pitch (K bytes) that is a multiple of 16.
    return a.M >= 1 && a.N >= 1 && a.K >= 16 && (a.K % 16 == 0) && aligned(a.A, 16) && aligned(a.B, 16);
}

// TMA-store epilogue: every destination base, the row pitch and the row length must be multiples of 16 bytes
static bool tma_store_ok(const MMArgs& a, void* const* dsts, int n_dst)
{
    const size_t esz = dtype_size(a.out_dtype);
    if ((a.ldc * esz) % 16 != 0) return false;
    // TMA stores move 16-byte units: a row of the column block that does not end on one would be rounded UP and the
    // store would write past column N (seen: three columns of a neighbour's shard zeroed)
    if (((size_t)a.N * esz) % 16 != 0) return false;
    for (int d = 0; d < n_dst; ++d)
        if (!aligned(dsts[d], 16)) return false;
    return true;
}

static void fill_signal(StoreMaps& sm, const MMArgs& a)
{
    sm.n_sig = 0; sm.cta_counter = nullptr; sm.epoch = 0;
    for (int d = 0; d < kMaxDst; ++d) sm.sig[d] = nullptr;
    if (!a.sig) return;
    sm.n_sig = a.n_dst;
    for (int d = 0; d < sm.n_sig; ++d) sm.sig[d] = reinterpret_cast<unsigned long long*>(a.sig->flags[d]);
    sm.cta_counter = a.sig->cta_counter;
    sm.epoch = a.sig->epoch;
}

int launch_peer_wait(const uint64_t* flags, int world, int rank, uint64_t epoch, cudaStream_t st)
{
    return launch_ex(fp8_peer_wait_kernel, dim3(1), dim3(32), 0, st, 1, 1, /*pdl=*/true,
                     reinterpret_cast<const unsigned long long*>(flags), world, rank, (unsigned long long)epoch);
}

template <int BN, int CG, int MODE = kStDirect>
static int launch_tcgen05_cfg(const MMArgs& a)
{
    using Cfg = GemmCfg<BN, CG, MODE>;
    static std::atomic<int> attr_done[64];
    if (int rc = ensure_max_smem(fp8_gemm_tcgen05_kernel<BN, CG, MODE>, Cfg::kSmemBytes, attr_done)) return rc;

    CUtensorMap tmap_a, tmap_b;
    // A problem shorter than one tile loads only its own rows (rounded up to the 8-row swizzle atom): a 128-row box over
    // a matrix of <= 40 rows was measured to run the main loop at HALF speed (M = 32: 16.2 us, M = 48: 11.8 us for
    // K = 3072, N = 12288).  The rows of the stage beyond the box keep stale shared memory; they only feed accumulator
    // rows >= M, which are never stored (and are masked out of the NaN probe).
    const int a_box_rows = a.M < kBM ? ((a.M + 7) / 8) * 8 : kBM;
    if (!encode_operand_map(&tmap_a, a.A, a.M, a.K, a_box_rows)) return FP8B_ERR_CUDA;
    if (!encode_operand_map(&tmap_b, a.B, a.N, a.K, Cfg::kBRows)) return FP8B_ERR_CUDA;

    const size_t esz = dtype_size(a.out_dtype);
    GemmParams p;
    p.A = a.A; p.B = a.B; p.M = a.M; p.N = a.N; p.K = a.K;
    p.num_m_blocks = (a.M + kBM * CG - 1) / (kBM * CG);
    p.num_n_blocks = (a.N + BN - 1) / BN;
    p.num_k_blocks = (a.K + kBK - 1) / kBK;
    {   // Tile order.  N fastest: the tiles in flight complete whole output rows together (DRAM-page- and NVLink-friendly
        // writes; the C4 shard at w = 2: 53.2 vs 58.6 us) and re-read B once per 256-row block from L2 -- fine while B
        // stays L2-resident.  Otherwise the smaller operand is the one to re-read.
        const int forced_r = tune(kTuneGemmRaster, 0);
        const size_t b_bytes = (size_t)a.N * a.K, a_bytes = (size_t)a.M * a.K;
        const bool n_fast = b_bytes <= ((size_t)48 << 20) || b_bytes <= a_bytes;
        // Both operands too large to sit in L2 beside each other (8192^3: 67 MB each): grouped order.
        const bool grouped = a_bytes > ((size_t)32 << 20) && b_bytes > ((size_t)32 << 20) && p.num_m_blocks > kRasterGroup;
        p.raster_n = forced_r ? (forced_r == 3 ? 2 : forced_r == 2) : grouped ? 2 : n_fast;
    }
    const int tiles_all = p.num_m_blocks * p.num_n_blocks;
    const int workers_cap = device_info().sm_count / CG;
    p.full_tiles = tiles_all;
    p.num_work = tiles_all;
    {   // split the partially filled last wave into half-width tiles when that makes it one SHORT round
        const int rem = tiles_all % workers_cap;
        bool can_split = (BN % 64 == 0) && ((BN / 2 / CG) % 8 == 0) && tiles_all > workers_cap;
        if (MODE == kStTma) can_split = can_split && ((BN / 2) * esz) % 128 == 0;      // half tiles must be whole store boxes
#ifdef FP8B_PROFILE
        can_split = can_split && !(tune_int("FP8B_GEMM_DEBUG", 0) & 8);
#endif
        if (can_split && rem > 0 && 2 * rem <= workers_cap) {
            p.full_tiles = tiles_all - rem;
            p.num_work = tiles_all + rem;
        }
    }
    p.epi = make_epi(a);
    p.vec_store_ok = aligned(a.C, 16) && ((a.ldc * esz) % 16 == 0);
    p.col_vec_ok = (a.sb_len == 1 || aligned(a.sb, 16)) && (!a.bias || aligned(a.bias, 16));
    p.multicast = a.store == Store::Multicast;
    p.n_dst = a.n_dst;
    p.peer_delta = reinterpret_cast<const long long*>(a.peer_deltas);
    p.a_fmt = a.a_fmt; p.b_fmt = a.b_fmt;
    p.stage_tx = a_box_rows * kBK + Cfg::kBBytes;
    typename StoreMapsOf<MODE>::type smaps;
    if constexpr (MODE == kStTma) {
        // (BN * esz) % 128: a tile must be whole 128-byte boxes, or a box store would cover the next tile's columns
        if (!tma_store_ok(a, a.dsts, a.n_dst) || (BN * esz) % 128 != 0) return FP8B_ERR_UNSUPPORTED;
        for (int d = 0; d < a.n_dst; ++d)
            if (!get_tensor_map(&smaps.m[d], a.dsts[d], (uint64_t)a.M, (uint64_t)a.N * esz, (uint64_t)a.ldc * esz, 128, 128))
                return FP8B_ERR_CUDA;
        for (int d = a.n_dst; d < kMaxDst; ++d) smaps.m[d] = smaps.m[0];
        fill_signal(smaps, a);
    } else {
        smaps.unused = 0;
    }
#ifdef FP8B_PROFILE
    p.debug = tune_int("FP8B_GEMM_DEBUG", 0);
    p.dbg = nullptr;
    if (p.debug & 16) {                      // profiling only: allocates and synchronises
        static long long* dbuf = nullptr;
        if (!dbuf) cudaMalloc(&dbuf, 64 * 8 * sizeof(long long));
        cudaMemset(dbuf, 0, 64 * 8 * sizeof(long long));
        p.dbg = dbuf;
    }
#endif
    // multimem.st / peer stores have no sub-word form: both modes need every chunk on the 16-byte path
    if (!is_push<MODE>() && a.store != Store::Local && !(p.vec_store_ok && p.col_vec_ok && a.N % 32 == 0))
        return FP8B_ERR_UNSUPPORTED;

    const int workers = p.num_work < workers_cap ? p.num_work : workers_cap;      // one CTA (or CTA pair) per SM (pair)
    // Programmatic dependent launch (FP8B_OPT_PDL): the prologue overlaps the predecessor's tail.  Worth nothing on C4
    // (104.17 vs 104.12 us back to back: power-limited, idle gaps only buy clock) but a fixed ~2 us on small problems.
    const int rc = launch_ex(fp8_gemm_tcgen05_kernel<BN, CG, MODE>, dim3(workers * CG), dim3(gemm_threads<MODE>()),
                             Cfg::kSmemBytes, a.st, CG, 1, g_opt_pdl.load(std::memory_order_relaxed) != 0,
                             tmap_a, tmap_b, smaps, p);
#ifdef FP8B_PROFILE
    if (rc == FP8B_OK && p.dbg) {
        long long h[64 * 8];
        cudaDeviceSynchronize();
        cudaMemcpy(h, p.dbg, sizeof(h), cudaMemcpyDeviceToHost);
        printf("CTA 0: kernel entry -> first MMA wait %lld cycles; last epilogue end -> stores complete %lld; -> CTA end %lld\n",
               h[0] - h[7], h[15] ? h[15] - h[23] : 0, h[31] - (h[15] ? h[15] : h[23]));
        printf("tile | mma: wait_tempty  issue+run (of which waiting for TMA) | epi: wait_tfull  drain+store | epi_end - mma_end\n");
        for (int t = 0; t < 64 && h[t * 8 + 2]; ++t)
            printf("%4d | %8lld %8lld (%8lld) | %8lld %8lld | %8lld   (mma start %lld)\n", t, h[t * 8 + 1] - h[t * 8 + 0],
                   h[t * 8 + 2] - h[t * 8 + 1], h[t * 8 + 3], h[t * 8 + 5] - h[t * 8 + 4], h[t * 8 + 6] - h[t * 8 + 5],
                   h[t * 8 + 6] - h[t * 8 + 2], h[t * 8 + 0] - h[0]);
    }
#endif
    return rc;
}

// Split-K plan (fp8_gemm_splitk_kernel): clusters of S CTAs, one 128 x 128 tile each.
template <int S>
static int launch_splitk(const MMArgs& a)
{
    static std::atomic<int> attr_done[64];
    if (int rc = ensure_max_smem(fp8_gemm_splitk_kernel<S>, kSkSmemBytes, attr_done)) return rc;
    const int a_box_rows = a.M < kBM ? ((a.M + 7) / 8) * 8 : kBM;      // see launch_tcgen05_cfg
    CUtensorMap tmap_a, tmap_b;
    if (!encode_operand_map(&tmap_a, a.A, a.M, a.K, a_box_rows)) return FP8B_ERR_CUDA;
    if (!encode_operand_map(&tmap_b, a.B, a.N, a.K, 128)) return FP8B_ERR_CUDA;
    const size_t esz = dtype_size(a.out_dtype);
    SplitKParams p;
    p.A = a.A; p.B = a.B; p.M = a.M; p.N = a.N; p.K = a.K;
    p.num_n_blocks = (a.N + 127) / 128;
    p.num_k_blocks = (a.K + kBK - 1) / kBK;
    p.stage_tx = a_box_rows * kBK + 128 * kBK;
    p.idesc = make_idesc(kBM, 128) | ((uint32_t)(a.a_fmt ? 1 : 0) << 7) | ((uint32_t)(a.b_fmt ? 1 : 0) << 10);
    p.a_fmt = a.a_fmt; p.b_fmt = a.b_fmt;
    p.epi = make_epi(a);
    p.vec_store_ok = aligned(a.C, 16) && ((a.ldc * esz) % 16 == 0);
    p.col_vec_ok = (a.sb_len == 1 || aligned(a.sb, 16)) && (!a.bias || aligned(a.bias, 16));
    p.dbg = nullptr;
#ifdef FP8B_PROFILE
    if (tune_int("FP8B_GEMM_DEBUG", 0) & 16) {     // profiling only: allocates and synchronises
        static long long* dbuf = nullptr;
        if (!dbuf) cudaMalloc(&dbuf, 8 * sizeof(long long));
        cudaMemset(dbuf, 0, 8 * sizeof(long long));
        p.dbg = dbuf;
    }
#endif
    const long tiles = (long)((a.M + kBM - 1) / kBM) * p.num_n_blocks;
    if (p.num_k_blocks < S || tiles * S > 65535L * 16) return FP8B_ERR_UNSUPPORTED;
    const int rc = launch_ex(fp8_gemm_splitk_kernel<S>, dim3((unsigned)(tiles * S)), dim3(kSkThreads), kSkSmemBytes, a.st, S, 1,
                             g_opt_pdl.load(std::memory_order_relaxed) != 0, tmap_a, tmap_b, p);
#ifdef FP8B_PROFILE
    if (rc == FP8B_OK && p.dbg) {
        long long h[8];
        cudaDeviceSynchronize();
        cudaMemcpy(h, p.dbg, sizeof(h), cudaMemcpyDeviceToHost);
        printf("split-K x%d, CTA 0 thread 0 (cycles): prologue %lld | main loop %lld | scatter %lld | wait for peers %lld | "
               "reduce+store %lld | final cluster sync %lld\n", S, h[1] - h[0], h[2] - h[1], h[3] - h[2], h[4] - h[3], h[5] - h[4],
               h[6] - h[5]);
    }
#endif
    return rc;
}

// How many CTAs should share one tile (0 = the ordinary plans).  Split K when all clusters fit on the GPU at once and K
// is long enough to pay for the reduction (~2 000 cycles of scatter / wait / gather).  Calibrated on the sweep in
// profiles/r2_splitk_calibration.log (us, no split / 2 / 4): M=32 K=N=3072 8.9 / 8.1 / 7.1; M=128 K=8192 N=2048 18.0 / 12.9 /
// 9.6; M=32 K=14336 N=4096 28.3 / 19.8 / 16.0; M=256 K=N=3072 9.7 / 8.8 / 13.7 (192 CTAs: two waves); K=1024: never a gain.
// FP8B_OPT_TUNE_GEMM_SPLITK: 1 = never, 2 / 4 = force.
static int pick_split_k(const MMArgs& a)
{
    const int forced = tune(kTuneGemmSplitK, 0);
    if (forced == 1) return 0;
    const int kb = (a.K + kBK - 1) / kBK;
    if (forced == 2 || forced == 4) return kb >= forced ? forced : 0;
    const long tiles = (long)((a.M + kBM - 1) / kBM) * ((a.N + 127) / 128);
    const int sms = device_info().sm_count;
    if (tiles * 4 <= sms && kb >= 16) return 4;
    if (tiles * 2 <= sms && kb >= 24) return 2;
    return 0;
}

constexpr int kDefaultGemmStore = 2;      // epilogue of plain fp8b_scaled_mm calls: 1 = st.global from the epilogue warps, 2 = TMA
                                          // store (C4: 109.7 vs 112.0 us in the same bench run; falls back to 1 when C is not TMA-storable)

// Tile configuration: 1 = 128x256 one CTA, 2 = 128x128 one CTA, 3 = 256x256 pair, 4 = 256x128 pair, 5 = 256x192 pair.
// The TMA-store epilogue needs tiles of whole 128-byte boxes; only 256x192 with 1-byte (e4m3fn) elements is not.
static bool tile_whole_boxes(int cfg, int out_dtype)
{
    const int width = cfg == 5 ? 192 : (cfg == 1 || cfg == 3) ? 256 : 128;
    return (width * dtype_size(out_dtype)) % 128 == 0;
}

static int pick_tile_cfg(const MMArgs& a)
{
    const int sms = device_info().sm_count;
    const bool pairs_only = a.store == Store::Peers;         // the peer-store plan exists for CTA pairs only
    // Small problems (one round of 128 x 128 tiles, or two short ones): one-CTA tiles.  A CTA pair spends ~1 300 more cycles
    // in its prologue (cluster barrier) and its larger tile leaves a longer exposed epilogue; measured (us, chosen pair
    // config -> 128 x 128): 512^3 4.9 -> 4.4, 1024^3 6.2 -> 5.7, 2048 x 512 x 2048 8.5 -> 7.2, M=333 K=N=4096 13.1 -> 12.1;
    // with a long K and two rounds the pairs' cheaper main loop wins again (M=1000 K=N=3072: 12.9 vs 13.9).
    const long tiles128 = (long)((a.M + kBM - 1) / kBM) * ((a.N + 127) / 128);
    if (!pairs_only && (tiles128 <= sms || (tiles128 <= 2L * sms && a.K <= 1024))) return 2;
    if (a.M > 128 && a.N > 128) {
        // CTA pairs.  Pick the tile width minimising rounds x time-per-tile.  A tile costs a fixed ~1.5 us (accumulator
        // hand-over, pipeline fill) plus a part proportional to K that was measured at K = 3072 as 10.5 / 9.3 / 8.65 us
        // per tile for widths 256 / 192 / 128 (L2->SM traffic of the operands, not MMA time, dominates, so narrow
        // tiles are barely cheaper).  Only the ratios matter.
        // Pushing to peers the kernel is bound by NVLink, not by the tensor pipe, and the link idles until the first tiles
        // are complete: narrower tiles (256 x 128) halve that ramp at no cost in exchange time (measured at w = 2:
        // 103.4 us against 106.4 us with 256 x 256 tiles; profiles/r2_scaling.md).
        if (a.store == Store::Push && a.n_dst > 1) return 4;
        // a push whose TMA-store boxes do not tile 256x192 leaves that configuration out
        const bool no_192 = a.store == Store::Push && !tile_whole_boxes(5, a.out_dtype);
        const long mt = (a.M + 255) / 256;
        const int pairs = sms / 2;
        const double kf = (double)a.K / 3072.0;
        auto cost = [&](int width) {
            const double t3072 = width == 256 ? 10.5 : width == 192 ? 9.3 : 8.65;
            const long tiles = mt * ((a.N + width - 1) / width);
            return (1.5 + kf * (t3072 - 1.5)) * (double)((tiles + pairs - 1) / pairs);
        };
        int cfg = 3;
        double best = cost(256);
        if (!no_192 && cost(192) < best) { best = cost(192); cfg = 5; }
        if (cost(128) < best) { best = cost(128); cfg = 4; }
        return cfg;
    }
    const long t_256 = (long)((a.M + kBM - 1) / kBM) * ((a.N + 255) / 256);
    return (a.N > 128 && t_256 >= 2L * sms) ? 1 : 2;
}

// Tile configuration -> kernel instantiation.  The peer-store epilogue is built for the CTA-pair configurations only.
template <int MODE>
static int launch_cfg(int cfg, const MMArgs& a)
{
    switch (cfg) {
        case 3: return launch_tcgen05_cfg<256, 2, MODE>(a);
        case 4: return launch_tcgen05_cfg<128, 2, MODE>(a);
        case 5: return launch_tcgen05_cfg<192, 2, MODE>(a);
    }
    if constexpr (MODE == kStPeers) return FP8B_ERR_UNSUPPORTED;
    else return cfg == 1 ? launch_tcgen05_cfg<256, 1, MODE>(a) : launch_tcgen05_cfg<128, 1, MODE>(a);
}

int launch_gemm_tcgen05(const MMArgs& a)
{
    if (!tcgen05_supported(a)) return FP8B_ERR_UNSUPPORTED;
    // Tile choice.  Prefer CTA pairs (256-row tiles) whenever M and N are large enough for them,
    // 256-wide when that still leaves >= ~2 waves of tiles, else 128-wide (finer tail).
    // fp8b_set_option(FP8B_OPT_TUNE_GEMM_CFG) -- a result-neutral tuning knob -- forces one.
    const int forced = tune(kTuneGemmCfg, 0);
    const int cfg = forced ? forced : pick_tile_cfg(a);
    switch (a.store) {
        case Store::Multicast: return launch_cfg<kStDirect>(cfg, a);
        case Store::Peers: return launch_cfg<kStPeers>(cfg, a);
        case Store::Push: return launch_cfg<kStTma>(cfg, a);      // store-ring epilogue, 1..8 destinations
        case Store::Local: break;
    }
    if (!forced) {                            // few tiles and a long K -> several CTAs per tile
        const int split = pick_split_k(a);
        if (split == 4) return launch_splitk<4>(a);
        if (split == 2) return launch_splitk<2>(a);
    }
    // TMA-store epilogue to the one output, else the st.global epilogue (same bits)
    if (tune(kTuneGemmStore, kDefaultGemmStore) == 2 && tma_store_ok(a, &a.C, 1) && tile_whole_boxes(cfg, a.out_dtype)) {
        MMArgs t = a;
        t.store = Store::Push; t.n_dst = 1; t.dsts = &a.C;
        return launch_cfg<kStTma>(cfg, t);
    }
    return launch_cfg<kStDirect>(cfg, a);
}

}  // namespace fp8b
