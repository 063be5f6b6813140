// BALF detector forward on the sm_100a tensor cores: precision 1 ("tf32": single-rounded fp16 / tf32 operands) and precision 2
// ("f16x3": every operand an fp16 hi + lo pair, three MMAs per product -- template flag PX, see BranchG).
//
// Same semantics and kernel decomposition as the fp32 path in detector.cu (reference:
// balf/model/mlp_ma_decoder.py:201-244 Down, :119-149 multi-axis gMLP, :25-117 grid / block gMLP,
// :151-199 channel attention; balf/model/decoder.py:16-30 head), but every Linear layer and both
// token-mixing products are tcgen05.mma (kind::f16 on fp16 operands -- the same 11-bit significand as tf32 --
// with fp32 accumulation in TMEM; kind::tf32 for the bias columns) and the whole chain of a tile stays on chip:
//
//   shared memory (A operand, chunk-major) --tcgen05.mma--> TMEM accumulator --tcgen05.ld--> registers
//        ^                                                                          |
//        +---- activation / LayerNorm / gating, 1 / 2 / 4 threads per pixel row  <--+
//
// A tile is 128 pixels = 2 "units" of 64 tokens (grid branch: the 64 cells of one in-cell offset;
// block branch: one 8x8 block; merge / head: 64 consecutive pixels).  Thread (row = tid % 128, part = tid / 128)
// owns one part (1 / TPR) of the channels of pixel row `row`; TMEM lane == row, so GELU, gating and softmax are
// thread-local and LayerNorm needs one (sum, sum of squares) exchange between the parts of a row through shared
// memory.  Stage 1 runs one thread per row in five independent tile groups per CTA (BranchCfg).
//
// What the epilogues do NOT do: biases ride in the GEMM (one extra K = 8 MMA whose A operand is a
// constant [1 1 0 ...] column block and whose B rows hold the bias split into tf32 hi + lo parts), and
// the LayerNorm affine parameters that feed a Linear layer are folded into that layer's weights and bias
// when the weights are packed (W' = W diag(gamma), b' = b + W beta).  GELU is the exact erf form,
// evaluated as relu(v) - |v| * 0.5 erfc(|v| / sqrt 2) with erfc through exp2 of a degree-5 fit (|err| < 3.7e-6,
// scripts/fit_gelu.py).
//
// The 64x64 token mixing runs as M = 64 MMAs (A = mixing matrix, B = the tile's activations in the A-operand layout,
// read as an MN-major operand, see issue_mix_t); the accumulators of the two units interleave in the two 16-lane
// halves of every 32-lane TMEM quadrant, which fixes the lane <-> pixel mapping of the branch kernels:
//        unit g = (lane % 32) / 16,   token = (lane / 32) * 16 + lane % 16.
// Weights are pre-packed into the exact shared-memory image of the B operands and brought in by TMA
// bulk copies (cp.async.bulk + mbarrier) -- once per CTA when the whole set fits next to the operand
// region (stages 1-3), otherwise through a 2-3 slot ring that runs ahead of the MMAs.  Tensors that cross HBM between
// the kernels of a stage are fp16 wherever their consumer rounds them to fp16 anyway (u', v', r, the pooled level
// inputs); DESIGN.md section 3.
// This file is the body of two translation units (compile time): detector_tc.cu (BALF_TC_MAIN: weight packing, the single-rounded
// instantiations, the entry points) and detector_tc_x3.cu (the split-precision instantiations).
#pragma once
#include <cuda_fp16.h>
#include "detector.cuh"
#include "umma.cuh"

namespace balf {
using namespace umma;

constexpr int kMerge32Ctas = 3;         // CTAs per SM of the single-rounded stage-1 merge kernel (MergeBulkCfg::min_ctas)
constexpr int kRc16MinC = 32;           // conv1 / conv2 of the merge kernels run on fp16 operands for C > this
constexpr int TM = 128;                 // pixel rows per tile
constexpr int NT2 = 256;                // threads per CTA (two per row)
constexpr int kMaxSlot = 4;              // ring slots: per kernel family (G::nslot), sized from the shared-memory budget
constexpr int kMaxGemm = 6;

struct TcGemm {
    uint32_t goff;        // float offset of the first block inside the tc blob
    uint16_t nblk;        // K blocks
    uint16_t rows;        // rows of the packed operand (N of a Linear layer, 64 for a mixing matrix)
    uint16_t kb;          // K columns per block
    uint16_t bias;        // 1: the last block carries 8 extra K columns (bias hi, bias lo, 0 ...)
    uint16_t h16;         // 1: the K columns are fp16 (kind::f16 MMAs, 8 per 16-byte chunk); the bias columns stay tf32
                          // 2: split precision ("f16x3"): every block holds its kb columns twice, fp16 hi then fp16 lo = fp16(w - hi)
};
// bytes per K element of a packed operand
__host__ __device__ constexpr uint32_t tc_eb(int h16) { return h16 == 1 ? 2u : 4u; }
struct TcPlan {
    const float* base;
    TcGemm g[kMaxGemm];
    int ngemm;
    int resident;         // all blocks stay in shared memory for the life of the CTA
    uint32_t bytes;       // total bytes of all blocks (resident footprint)
    uint32_t slot_bytes;  // ring slot size (largest block, 128-byte multiple)
    uint32_t nslot;       // ring slots
    uint32_t ebias_off;   // float offset (inside the tc blob) of the [gemm][row][hi, lo, 0, 0] bias vectors the epilogues add (MergeG::ebias), or 0
    long long* trace;     // development hook (balf_debug_set_trace): clock stamps of CTA 0, or null
};
#ifdef BALF_TC_MAIN
long long* g_tc_trace = nullptr;
int g_tc_trace_sel = 0;           // which kernel family records (debug key 2): 0 = branch kernels, 1 = merge kernels
#else
extern long long* g_tc_trace;
extern int g_tc_trace_sel;
#endif
constexpr int kTracePoints = 16, kTraceTiles = 16;
// stamp `pt` of tile iteration `it` for thread 0 (slot 0: the MMA issuer) and the last thread (slot 1: pure epilogue)
#ifdef BALF_TC_TRACE          // development builds only (NVCC_FLAGS=-DBALF_TC_TRACE python balf_b200/build.py --force): the stamps cost
                             // ~5 % of the epilogue instructions (predicate + clock read per point)
#define TC_TRACE(plan, it, pt)                                                                                     \
    do {                                                                                                           \
        if ((plan).trace && blockIdx.x == 0 && (it) < kTraceTiles && (threadIdx.x == 0 || threadIdx.x == NT2 - 1)) \
            (plan).trace[(((it) * kTracePoints + (pt)) << 1) + (threadIdx.x ? 1 : 0)] = clock64();                 \
    } while (0)
#else
#define TC_TRACE(plan, it, pt) do { (void)(it); } while (0)
#endif

enum { BG_CONV0 = 0, BG_PD1, BG_D1A, BG_D1B, BG_WM, BG_D2, BG_COUNT };
enum { MG_CONV0 = 0, MG_PD2A, MG_PD2B, MG_RC1, MG_RC2, MG_COUNT };
enum { HG_C2 = 0, HG_DENSE, HG_COUNT };
constexpr int kHeadN = 80;              // 65 logits padded to a legal UMMA N (multiple of 16)

__host__ __device__ constexpr int tc_kin(int cin) { return cin < 8 ? 8 : cin; }
// K columns per streamed block: the largest power-of-two divisor of K (>= 8) whose block is <= cap bytes
__host__ __device__ constexpr int tc_kb(int rows, int K, int cap = 32768, int eb = 4) {
    int kb = K;
    while (kb > 32 / eb && (kb * rows * eb > cap || K % kb != 0)) kb /= 2;
    return kb;
}
__host__ __device__ constexpr int tc_cols(int need) { return need <= 32 ? 32 : need <= 64 ? 64 : need <= 128 ? 128 : need <= 256 ? 256 : 512; }
__host__ __device__ inline uint32_t gemm_block_bytes(const TcGemm& g, uint32_t b) {
    return (uint32_t)g.rows * (g.kb * tc_eb(g.h16) + ((g.bias && b + 1 == g.nblk) ? 32u : 0u));
}
__host__ __device__ inline uint32_t gemm_bytes(const TcGemm& g) {
    return (uint32_t)g.rows * ((uint32_t)g.kb * g.nblk * tc_eb(g.h16) + (g.bias ? 32u : 0u));
}

// ------------------------------------------------------------------------------------------ weight ring (thread 0)
struct Ring {
    uint32_t wsm;          // shared address of the weight area
    uint64_t* full;        // [nslot]
    uint64_t* empty;       // [nslot]
    uint32_t pidx, nsched; // producer cursor into the block schedule / its length
    const uint2* sched;    // [nsched] (float offset inside the tc blob, bytes) of every block of the plan, in issue order
    uint32_t pcnt, ccnt;   // blocks loaded / consumed so far
    uint32_t pslot, puse;  // producer slot / how many times it has been filled before
    uint32_t cslot, cpar;  // consumer slot / its full-barrier parity
    uint32_t to_load;      // blocks still to be requested over the life of the CTA
};

__device__ __forceinline__ void bulk_load(uint32_t dst, const float* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// The block schedule is tabulated once per CTA (ring_build_schedule): walking the plan structure for every block put
// ~1500 cycles of serial single-thread code (local-memory struct reads, 64-bit address arithmetic) on the critical
// path of every GEMM phase of the streamed stages.
__device__ __forceinline__ void ring_build_schedule(uint2* sched, const TcPlan& p, uint32_t* count) {
    uint32_t n = 0;
    for (int gi = 0; gi < p.ngemm; ++gi) {
        const TcGemm g = p.g[gi];
        for (uint32_t b = 0; b < g.nblk; ++b)
            sched[n++] = make_uint2(g.goff + b * (uint32_t)g.rows * g.kb / (g.h16 == 1 ? 2u : 1u), gemm_block_bytes(g, b));
    }
    *count = n;
}
template <int NS>
__device__ __forceinline__ void ring_load_one(Ring& r, const TcPlan& p) {
    const uint2 e = r.sched[r.pidx];
    const uint32_t slot = r.pslot;
    if (r.puse > 0) mbar_wait(&r.empty[slot], (r.puse - 1) & 1);
    mbar_expect_tx(&r.full[slot], e.y);
    bulk_load(r.wsm + slot * p.slot_bytes, p.base + e.x, e.y, &r.full[slot]);
    ++r.pcnt;
    --r.to_load;
    if (++r.pslot == NS) { r.pslot = 0; ++r.puse; }
    if (++r.pidx == r.nsched) r.pidx = 0;
}
// Called at the top of every block AND right after a phase's MMAs have completed (wait_done_ring): at that point every
// slot is free, so the next phase's first blocks stream in under the epilogue instead of under the next issue.
template <int NS>
__device__ __forceinline__ void ring_top_up(Ring& r, const TcPlan& p) {
    while (r.to_load > 0 && r.pcnt < r.ccnt + NS) ring_load_one<NS>(r, p);
}
template <int NS>
__device__ __forceinline__ void ring_consumed(Ring& r) {
    ++r.ccnt;
    if (++r.cslot == NS) { r.cslot = 0; r.cpar ^= 1; }
}
// resident mode: every gemm, once
__device__ __forceinline__ void ring_load_all(Ring& r, const TcPlan& p) {
    mbar_expect_tx(&r.full[0], p.bytes);
    uint32_t off = 0;
    for (int gi = 0; gi < p.ngemm; ++gi) {
        const uint32_t bytes = gemm_bytes(p.g[gi]);
        bulk_load(r.wsm + off, p.base + p.g[gi].goff, bytes, &r.full[0]);
        off += bytes;
    }
}
// ---- compile-time plans.  Every GEMM of a kernel is fixed by its template parameters, so thread 0's issue path is
// straight-line code: descriptors are a per-kernel base plus immediates instead of per-MMA address arithmetic
// (the serial issue path sits on the critical path of every phase of every tile).  Must mirror tc_build_plans.
// PX = 1: the split-precision plans ("f16x3"): every operand is an fp16 hi + fp16 lo pair and every product runs as
// hi*hi + lo*hi + hi*lo on the tensor core (fp32-class results, 3x the MMAs, 2x the operand bytes); see issue_linear_t.
template <int CIN, int C, int PX = 0> struct BranchG {
    static constexpr int count = BG_COUNT;
    static constexpr bool x3 = PX != 0;
    static constexpr bool resident = PX ? C <= 64 : C <= 128;   // fp16 weights: 60 KB at C = 64 (shared by two tile groups), 172 KB at C = 128
    static constexpr int cap = 32768;
    static constexpr int nslot = PX ? (C == 256 ? 2 : 3) : (C == 256 ? 3 : 2);
    __host__ __device__ static constexpr int rows(int gi) { return gi == BG_WM ? 64 : C; }
    __host__ __device__ static constexpr int K(int gi) { return gi == BG_CONV0 ? tc_kin(CIN) : gi == BG_WM ? 64 : C; }
    __host__ __device__ static constexpr bool bias(int gi) { return gi != BG_WM; }
    // every GEMM runs on fp16 operands (kind::f16): the same 11-bit significand as tf32, half the weight bytes to stream / keep
    // resident, half the operand bytes and MMAs.  (The network-input stage computes conv.0, K = 3, on the CUDA cores.)
    __host__ __device__ static constexpr bool h16(int gi) { return gi != BG_CONV0 || CIN >= 8; }
};
template <int CIN, int C, int PX = 0> struct MergeG {
    static constexpr int count = MG_COUNT;
    static constexpr bool x3 = PX != 0;
    // C = 64: 64 KB of weights (dense2 in fp16) next to the 128 KB of tile regions.  C = 128 (single-rounded operands): the five
    // fp16 weight matrices (144 KB) stay resident next to a 64 KB operand region -- the streamed version was bound by the bytes
    // the ring keeps in flight (the issuing lane waited 2-6 k cycles per GEMM for weights, scripts/tc_trace.py) -- which leaves no
    // room for the bias blocks: the epilogues add the biases (`ebias`, from the plan's fp32 bias vectors) instead of an MMA.
    static constexpr bool ebias = C == 128 && PX == 0;
    static constexpr bool resident = PX ? C <= 32 : C <= 128;
    static constexpr int cap = 32768;
    static constexpr int nslot = PX ? (C == 64 ? 3 : 2) : (C == 256 ? 2 : 3);
    __host__ __device__ static constexpr int rows(int) { return C; }
    __host__ __device__ static constexpr int K(int gi) { return gi == MG_CONV0 ? tc_kin(CIN) : C; }
    __host__ __device__ static constexpr bool bias(int gi) { return !ebias && gi != MG_PD2A; }
    // stages 1-2: u' / v' cross HBM as fp16 tiles (same 11-bit significand as the tf32 operands they replace, half the
    // bytes of the HBM-bound merge kernels), so dense2 runs as kind::f16 on fp16 weights
    // conv1 / conv2 (A operands written by the epilogues) run on fp16 operands at every stage
    // and dense2 as well: u' / v' arrive as fp16 tiles (C <= 128) or are converted by the loader (C = 256)
    __host__ __device__ static constexpr bool h16(int gi) {
        return gi == MG_PD2A || gi == MG_PD2B || (gi == MG_CONV0 && CIN >= 8) || ((gi == MG_RC1 || gi == MG_RC2) && (PX || C > kRc16MinC));
    }
};
template <int C, int PX = 0> struct HeadG {
    static constexpr int count = HG_COUNT;
    static constexpr bool x3 = PX != 0;
    static constexpr bool resident = false;
    static constexpr int cap = 32768;
    static constexpr int nslot = 2;
    __host__ __device__ static constexpr int rows(int gi) { return gi == HG_DENSE ? kHeadN : C; }
    __host__ __device__ static constexpr int K(int) { return C; }
    __host__ __device__ static constexpr bool bias(int) { return true; }
    __host__ __device__ static constexpr bool h16(int) { return true; }
};
// packing mode of GEMM gi (TcGemm::h16) and its bytes per K element
template <typename G> __host__ __device__ constexpr int g_mode(int gi) { return G::h16(gi) ? (G::x3 ? 2 : 1) : 0; }
template <typename G> __host__ __device__ constexpr uint32_t g_bytes(int gi) {
    return (uint32_t)G::rows(gi) * (G::K(gi) * tc_eb(g_mode<G>(gi)) + (G::bias(gi) ? 32u : 0u));
}
template <typename G> __host__ __device__ constexpr uint32_t g_off(int gi) { uint32_t o = 0; for (int i = 0; i < gi; ++i) o += g_bytes<G>(i); return o; }

// high word of a SWIZZLE_NONE descriptor (SBO = 128, version 1) -- the low word is (LBO >> 4) << 16 | addr >> 4
constexpr uint32_t kDescHi = (128u >> 4) | (1u << 14);
__device__ __forceinline__ uint64_t desc_of(uint32_t addr, uint32_t lbo) {
    return ((uint64_t)kDescHi << 32) | (uint64_t)(((lbo >> 4) << 16) | ((addr >> 4) & 0x3FFFu));
}

// kind::f16 with fp16 operands (A, B format 0 = F16, D = F32), K = 16 per instruction; probed: scripts/umma_probe_f16.cu
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) { return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24); }
__device__ __forceinline__ void mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, bool accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"((uint32_t)accumulate) : "memory");
}
// Thread 0: D[128 x N] (+)= A[128 x K] * W^T (+ bias) for GEMM GI of plan G (see issue_linear).
// high word of a K-major SWIZZLE_128B descriptor (SBO = 1024: 8 rows x 128 B, version 1, layout type 2); LBO is ignored
// by the hardware for swizzled K-major operands (encoded 1).  Probed: profiles/r01_umma_probe.txt "Kmaj SW128".
constexpr uint32_t kDescHiSw = (1024u >> 4) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint64_t desc_sw_of(uint32_t addr) {
    return ((uint64_t)kDescHiSw << 32) | (uint64_t)((1u << 16) | ((addr >> 4) & 0x3FFFu));
}
// ASW: the A operand is a [128 rows x K] tile in the swizzled panel layout (sw_off below) instead of chunk-major
template <typename G, int GI, bool ASW = false>
__device__ __forceinline__ void issue_linear_t(Ring& r, const TcPlan& p, uint32_t a_addr, uint32_t ones_addr, uint32_t d_tmem, bool first) {
    constexpr int ROWS = G::rows(GI), K = G::K(GI);
    constexpr bool BIAS = G::bias(GI), H16 = G::h16(GI);        // H16: A and B are fp16 chunk-major (8 halves per 16-byte chunk)
    // X3 (split precision): the A region holds K / 8 hi chunks followed by K / 8 lo chunks, a weight block its KB / 8 hi chunks
    // followed by KB / 8 lo chunks; D += A_hi W_hi + A_lo W_hi + A_hi W_lo (the lo * lo term is below fp32 resolution)
    constexpr bool X3 = H16 && G::x3;
    static_assert(!(H16 && ASW), "fp16 operands use the chunk-major layout");
    constexpr int KB = tc_kb(ROWS, K, G::cap, (int)tc_eb(g_mode<G>(GI))), NBLK = K / KB;
    constexpr uint32_t idesc = H16 ? make_idesc_f16(128, ROWS) : make_idesc_tf32(128, ROWS);
    constexpr uint32_t a_lbo = TM * 16u, b_lbo = (uint32_t)ROWS * 16u;
    constexpr int KSTEP = H16 ? 16 : 8, EPC = H16 ? 8 : 4;      // K per MMA, elements per 16-byte chunk
    const uint64_t a_desc = ASW ? desc_sw_of(a_addr) : desc_of(a_addr, a_lbo);
#pragma unroll
    for (int b = 0; b < NBLK; ++b) {
        uint32_t w_addr, slot = 0;
        if (G::resident) {
            w_addr = r.wsm + g_off<G>(GI) + (uint32_t)b * ROWS * KB * tc_eb(g_mode<G>(GI));
        } else {
            ring_top_up<G::nslot>(r, p);
            slot = r.cslot;
            mbar_wait(&r.full[slot], r.cpar);
            w_addr = r.wsm + slot * p.slot_bytes;
        }
        const uint64_t b_desc = desc_of(w_addr, b_lbo);
        fence_after_sync();
#pragma unroll
        for (int ks = 0; ks < KB / KSTEP; ++ks) {
            const uint32_t kchunk = (uint32_t)(b * KB) / EPC + (uint32_t)ks * 2u;
            // swizzled panels: 32 K columns (128 B) per panel of TM rows, 32 B per MMA inside a panel
            const uint32_t a_off = ASW ? (kchunk / 8u) * (TM * 128u) + (kchunk % 8u) * 16u : kchunk * a_lbo;
            if (H16) mma_f16(d_tmem, a_desc + (a_off >> 4), b_desc + (((uint32_t)ks * 2u * b_lbo) >> 4), idesc, !(first && b == 0 && ks == 0));
            else mma_tf32(d_tmem, a_desc + (a_off >> 4), b_desc + (((uint32_t)ks * 2u * b_lbo) >> 4), idesc, !(first && b == 0 && ks == 0));
            if constexpr (X3) {
                mma_f16(d_tmem, a_desc + ((a_off + (uint32_t)(K / 8) * a_lbo) >> 4), b_desc + (((uint32_t)ks * 2u * b_lbo) >> 4), idesc, true);
                mma_f16(d_tmem, a_desc + (a_off >> 4), b_desc + ((((uint32_t)KB / 8u + (uint32_t)ks * 2u) * b_lbo) >> 4), idesc, true);
            }
        }
        if (BIAS && b + 1 == NBLK)      // the bias columns (tf32: bias hi, bias lo, 0 ...) follow the block's KB / EPC chunks (twice that: X3)
            mma_tf32(d_tmem, desc_of(ones_addr, TM * 16u), b_desc + ((((uint32_t)KB / EPC) * (X3 ? 2u : 1u) * b_lbo) >> 4), make_idesc_tf32(128, ROWS), true);
        if (!G::resident) { commit(&r.empty[slot]); ring_consumed<G::nslot>(r); }
    }
}

// Thread 0: token mixing of both units, GEMM GI = the 64 x 64 mixing matrix (A operand, K-major).  B = the tile's LayerNorm'ed
// activations exactly as row_to_a16 wrote them -- [channel / 8][tile row][8 halves], i.e. an MN-major operand (instruction
// descriptor bit 16): 16 bytes = 8 channels of one token, tile rows (tokens) 16 bytes apart, channel chunks TM * 16 bytes apart;
// for an MN-major SWIZZLE_NONE operand LBO is the K-direction stride between 8-row core matrices (128) and SBO the MN-direction
// stride between chunk planes (probed: scripts/umma_probe_mn.cu, profiles/r02_umma_probe_mn.txt).  Tokens 16 g .. 16 g + 15 of
// unit u are tile rows 32 g + 16 u .. + 15 (TMEM lane = tile row), so K step g of unit u starts (32 g + 16 u) * 16 bytes in.
// (The first version stored a transposed [channel][token] copy with one 2-byte shared-memory store per value.)
constexpr uint32_t kDescHiMn = ((uint32_t)(TM * 16u) >> 4) | (1u << 14);
__device__ __forceinline__ uint64_t desc_mn_of(uint32_t addr) {
    return ((uint64_t)kDescHiMn << 32) | (uint64_t)(((128u >> 4) << 16) | ((addr >> 4) & 0x3FFFu));
}
template <typename G, int GI, int C>
__device__ __forceinline__ void issue_mix_t(Ring& r, const TcPlan& p, uint32_t y_addr, uint32_t d_tmem) {
    uint32_t w_addr, slot = 0;
    if (G::resident) {
        w_addr = r.wsm + g_off<G>(GI);
    } else {
        ring_top_up<G::nslot>(r, p);
        slot = r.cslot;
        mbar_wait(&r.full[slot], r.cpar);
        w_addr = r.wsm + slot * p.slot_bytes;
    }
    fence_after_sync();
    constexpr uint32_t idesc = make_idesc_f16(64, C) | (1u << 16);          // B MN-major
    constexpr uint32_t lo_off = (uint32_t)(C / 8) * TM * 16u;                // split precision: the lo chunk planes follow the hi ones
    const uint64_t w_desc = desc_of(w_addr, 1024u);
    const uint64_t y_desc = desc_mn_of(y_addr);
#pragma unroll
    for (uint32_t u = 0; u < 2; ++u) {
#pragma unroll
        for (uint32_t ks = 0; ks < 4; ++ks) {
            const uint32_t yo = (32u * ks + 16u * u) * 16u;
            mma_f16(d_tmem + ((u * 16u) << 16), w_desc + ((ks * 2u * 1024u) >> 4), y_desc + (yo >> 4), idesc, ks > 0);
            if constexpr (G::x3) {      // lo copies: the mixing matrix 8 KB (64 x 64 halves) further
                mma_f16(d_tmem + ((u * 16u) << 16), w_desc + ((ks * 2u * 1024u) >> 4), y_desc + ((lo_off + yo) >> 4), idesc, true);
                mma_f16(d_tmem + ((u * 16u) << 16), w_desc + ((8192u + ks * 2u * 1024u) >> 4), y_desc + (yo >> 4), idesc, true);
            }
        }
    }
    if (!G::resident) { commit(&r.empty[slot]); ring_consumed<G::nslot>(r); }
}

// ------------------------------------------------------------------------------------------ epilogue pieces
// exact-erf GELU: gelu(v) = max(v, 0) - a * e,  a = |v|,  e = 0.5 erfc(a / sqrt(2)) = exp2(R(a)) with R a degree-5
// polynomial (R(0) = -1; scripts/fit_gelu.py, |err| < 3.7e-6 absolute).  a is clamped to 4 sqrt(2), where e < 1e-8.
// Evaluated on pairs of values, see gelu_erf2.
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// ---- packed fp32x2 arithmetic (FFMA2 / FADD2 / FMUL2 on sm_100): one issue slot for two lanes-worth of work.  The
// epilogues are issue-bound (ncu: ~50 % issue utilisation at 24 warps/SM, a third of it FFMA), so the GELU polynomial,
// LayerNorm statistics / normalisation and the gating products run on register pairs.
__device__ __forceinline__ unsigned long long pk2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk2(unsigned long long r, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(r)); }
__device__ __forceinline__ unsigned long long fma2(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ unsigned long long add2(unsigned long long a, unsigned long long b) {
    unsigned long long d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ unsigned long long mul2(unsigned long long a, unsigned long long b) {
    unsigned long long d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
// two GELUs: the polynomial is evaluated in t = -a (alternating coefficient signs) so that the last step is one FFMA2
// relu(v) + t * e.  12 instructions per pair (4 FMNMX, 6 FFMA2, 2 MUFU) instead of 20.
__device__ __forceinline__ void gelu_erf2(float& v0, float& v1) {
    const float t0 = fmaxf(-fabsf(v0), -5.6568542494923806f), t1 = fmaxf(-fabsf(v1), -5.6568542494923806f);
    const unsigned long long t = pk2(t0, t1);
    // degree-5 fit (scripts/fit_gelu.py): |err| < 3.7e-6 absolute, 20x below the tf32 rounding of the value it feeds;
    // the degree-6 fit (3e-7) measured the same score-map error and keypoint agreement, one FFMA2 more per pair
    unsigned long long p = fma2(pk2(3.586947569e-04f, 3.586947569e-04f), t, pk2(6.316647399e-03f, 6.316647399e-03f));
    p = fma2(p, t, pk2(5.013782158e-02f, 5.013782158e-02f));
    p = fma2(p, t, pk2(-4.613807201e-01f, -4.613807201e-01f));
    p = fma2(p, t, pk2(1.150490999e+00f, 1.150490999e+00f));
    p = fma2(p, t, pk2(-1.0f, -1.0f));
    float p0, p1;
    upk2(p, p0, p1);
    const unsigned long long r = fma2(t, pk2(ex2_approx(p0), ex2_approx(p1)), pk2(fmaxf(v0, 0.0f), fmaxf(v1, 0.0f)));
    upk2(r, v0, v1);
}
// v[i] = gelu(v[i]) over an even-length register array; optionally accumulates sum and sum of squares
template <int N, bool STATS>
__device__ __forceinline__ void gelu_row(float (&v)[N], float& sum, float& sq) {
    unsigned long long s2 = pk2(0.f, 0.f), q2 = pk2(0.f, 0.f);
#pragma unroll
    for (int i = 0; i < N; i += 2) {
        gelu_erf2(v[i], v[i + 1]);
        if (STATS) { const unsigned long long x = pk2(v[i], v[i + 1]); s2 = add2(s2, x); q2 = fma2(x, x, q2); }
    }
    if (STATS) { float a, b; upk2(s2, a, b); sum = a + b; upk2(q2, a, b); sq = a + b; }
}
// v[i] = v[i] * rstd + shift
template <int N>
__device__ __forceinline__ void norm_row(float (&v)[N], float rstd, float shift) {
    const unsigned long long r2 = pk2(rstd, rstd), h2 = pk2(shift, shift);
#pragma unroll
    for (int i = 0; i < N; i += 2) { const unsigned long long x = fma2(pk2(v[i], v[i + 1]), r2, h2); upk2(x, v[i], v[i + 1]); }
}
__device__ __forceinline__ float lrelu02(float v) { return v > 0.0f ? v : 0.2f * v; }

// CH consecutive accumulator columns of this thread's row -> registers (tcgen05.ld is warp-collective)
template <int CH>
__device__ __forceinline__ void ld_row(uint32_t taddr, float (&v)[CH]) {
    if constexpr (CH == 16) {
        tmem_ld16(taddr, v);
    } else {
#pragma unroll
        for (int c0 = 0; c0 < CH; c0 += 32) tmem_ld32(taddr + c0, *reinterpret_cast<float (*)[32]>(&v[c0]));
    }
    tmem_ld_wait();
}
template <int CH>
__device__ __forceinline__ void st_row(uint32_t taddr, const float (&v)[CH]) {
    if constexpr (CH == 16) {
        asm volatile(
            "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
            :: "r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
               "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
               "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
               "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
            : "memory");
    } else {
#pragma unroll
        for (int c0 = 0; c0 < CH; c0 += 32) tmem_st32(taddr + c0, *reinterpret_cast<const float (*)[32]>(&v[c0]));
    }
    tmem_st_wait();
}

// this thread's CH values -> A operand (chunk-major, 128 rows), columns [col0, col0 + CH), tf32-rounded
template <int CH>
__device__ __forceinline__ void row_to_a(const float (&v)[CH], float* region, int row, int col0) {
#pragma unroll
    for (int j = 0; j < CH / 4; ++j)
        *reinterpret_cast<float4*>(region + ((size_t)(col0 / 4 + j) * TM + row) * 4) =
            to_tf32(make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
}

// the same as fp16 (kind::f16 operand): 8 channels per 16-byte chunk, round to nearest, saturating at the fp16 range
// (a, b) -> packed fp16 pair hi = (fp16(a), fp16(b)) and the packed fp16 pair of the rounding residuals lo = (fp16(a - hi.a), ...):
// hi + lo carries ~22 significant bits of the value (fp16 subnormals keep |lo| down to 6e-8 absolute)
__device__ __forceinline__ void split_h2(float a, float b, uint32_t& hi, uint32_t& lo) {
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&hi));
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(b - f.y), "f"(a - f.x));
}
// LOC > 0 (split precision): the lo chunks follow LOC chunks (= K / 8) after the hi chunks
template <int CH, int LOC = 0>
__device__ __forceinline__ void row_to_a16(const float (&v)[CH], float* region, int row, int col0) {
#pragma unroll
    for (int j = 0; j < CH / 8; ++j) {
        uint32_t h[4], l[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            if constexpr (LOC > 0) split_h2(v[8 * j + 2 * e], v[8 * j + 2 * e + 1], h[e], l[e]);
            else asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h[e]) : "f"(v[8 * j + 2 * e + 1]), "f"(v[8 * j + 2 * e]));
        }
        *reinterpret_cast<uint4*>(region + ((size_t)(col0 / 8 + j) * TM + row) * 4) = make_uint4(h[0], h[1], h[2], h[3]);
        if constexpr (LOC > 0) *reinterpret_cast<uint4*>(region + ((size_t)(LOC + col0 / 8 + j) * TM + row) * 4) = make_uint4(l[0], l[1], l[2], l[3]);
    }
}

// ---- "swizzled panel" layout of a [128 rows x C] tile (the K-major SWIZZLE_128B operand layout of tcgen05): panels of 32
// channels (128 B per row), rows 128 B apart inside a panel, the eight 16-byte chunks of a row XOR-permuted by (row % 8).
// A tile stored this way in GLOBAL memory (u', v', r, q of the network-input stage) moves to / from shared memory with one
// plain bulk copy (cp.async.bulk, 16 KB per panel, perfectly coalesced, no thread instructions), is a valid MMA operand as
// it lands, and is written by the epilogue threads without bank conflicts (eight consecutive rows hit eight different
// 16-byte bank groups).  Float offset of chunk `chunk` (4 channels) of row `row`:
__host__ __device__ __forceinline__ int sw_off(int row, int chunk) { return (chunk >> 3) * (TM * 32) + row * 32 + (((chunk & 7) ^ (row & 7)) << 2); }
template <int CH, bool ROUND>
__device__ __forceinline__ void row_to_sw(const float (&v)[CH], float* region, int row, int col0) {
#pragma unroll
    for (int j = 0; j < CH / 4; ++j) {
        float4 o = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        if (ROUND) o = to_tf32(o);
        *reinterpret_cast<float4*>(region + sw_off(row, col0 / 4 + j)) = o;
    }
}
// bulk copies shared <-> global (async proxy) and their bookkeeping
__device__ __forceinline__ void bulk_store(const float* gdst, uint32_t ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" :: "l"(gdst), "r"(ssrc), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---- tile groups.  A CTA is NG independent groups of 256 threads (NG = 1 everywhere except the branch kernels of the
// network-input stage): each group walks its own tiles with its own operand region, TMEM columns, completion barrier and
// hardware named barrier (id 1 + group), and all groups share one resident copy of the weights.  This is how four tiles are
// in flight per SM at C = 32 -- four separate CTAs would each need the 39 KB of weights.
template <int NG, int NTG = NT2>
__device__ __forceinline__ void group_sync(int grp) {
    if constexpr (NG == 1) __syncthreads();
    else asm volatile("bar.sync %0, %1;" :: "r"(grp + 1), "n"(NTG) : "memory");
}

// LayerNorm statistics of a row whose TPR parts live in TPR threads: exchange (sum, sum of squares).  TPR = 1: the thread
// owns the whole row, no exchange and no barrier.  TPR = 4: every thread adds the four partials in part order, so all
// threads of a row normalise with bit-identical statistics.
template <int NG = 1, int TPR = 2>
__device__ __forceinline__ void row_stats(float sum, float sq, float2* xch, int row, int half, int C, float& rstd, float& shift, int grp = 0) {
    if constexpr (TPR == 2) {
        xch[half * TM + row] = make_float2(sum, sq);
        group_sync<NG, TM * TPR>(grp);
        const float2 o = xch[(half ^ 1) * TM + row];
        sum += o.x; sq += o.y;
    } else if constexpr (TPR > 2) {
        xch[half * TM + row] = make_float2(sum, sq);
        group_sync<NG, TM * TPR>(grp);
        sum = 0.f; sq = 0.f;
#pragma unroll
        for (int p = 0; p < TPR; ++p) { const float2 o = xch[p * TM + row]; sum += o.x; sq += o.y; }
    }
    const float inv_c = C == 32 ? 1.0f / 32 : C == 64 ? 1.0f / 64 : C == 128 ? 1.0f / 128 : 1.0f / 256;   // C is a literal at every call
    const float mean = sum * inv_c;
    const float var = fmaxf(sq * inv_c - mean * mean, 0.f);
    rstd = rsqrtf(var + 1e-5f);                        // MUFU.RSQ, 2 ulp: far inside the tf32 operand rounding that follows
    shift = -mean * rstd;                              // normalised value = v * rstd + shift
}

// ------------------------------------------------------------------------------------------ shared memory carve-up
struct TcShared {
    float* region;         // operand region
    uint32_t wsm;          // weight area (shared address)
    float* ones;           // [2 chunks][128 rows][4]: (1 1 0 0), (0 0 0 0)
    float2* xch;           // [2 buffers][2 halves][128 rows]
    float* vec;            // small per-kernel vectors (gating LayerNorm affine)
    uint2* sched;          // weight-block schedule of the ring (kSchedEntries entries) + its length
    uint64_t* full;
    uint64_t* empty;
    uint64_t* done;
    uint64_t* aux;         // kernel-specific barrier (bulk-loaded tiles of tc_merge_bulk_kernel)
    uint32_t* tmem_slot;
    uint64_t* gdone;       // [kMaxGroups] completion barriers of tile groups 1.. (group 0 uses `done`)
};
constexpr int kMaxGroups = 8;
constexpr uint32_t kSchedEntries = 62;
constexpr uint32_t kOnesBytes = 2 * TM * 16, kXchBytes = 2 * 2 * TM * 8, kVecBytes = (2 * 256 + 64) * 4, kSchedBytes = (kSchedEntries + 2) * 8, kTcTail = 256;
__host__ __device__ inline uint32_t tc_weight_bytes(const TcPlan& p) {
    return p.resident ? (p.bytes + 127u) / 128u * 128u : p.nslot * p.slot_bytes;
}
__host__ __device__ inline uint32_t tc_smem_bytes(uint32_t region, const TcPlan& p, uint32_t groups = 1, uint32_t xchb = kXchBytes) {
    return groups * (region + xchb) + tc_weight_bytes(p) + kOnesBytes + kVecBytes + kSchedBytes + kTcTail;
}
// region / xch point at group 0's copy; group g's follow at g * region_bytes / g * kXchBytes
__device__ __forceinline__ TcShared carve(unsigned char* smem, uint32_t region_bytes, const TcPlan& p, uint32_t groups = 1, uint32_t xchb = kXchBytes) {
    TcShared s;
    unsigned char* q = smem;
    s.region = reinterpret_cast<float*>(q); q += groups * region_bytes;
    s.wsm = smem_u32(q); q += tc_weight_bytes(p);
    s.ones = reinterpret_cast<float*>(q); q += kOnesBytes;
    s.xch = reinterpret_cast<float2*>(q); q += groups * xchb;
    s.vec = reinterpret_cast<float*>(q); q += kVecBytes;
    s.sched = reinterpret_cast<uint2*>(q); q += kSchedBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(q);
    s.full = bars;
    s.empty = bars + kMaxSlot;
    s.done = bars + 2 * kMaxSlot;
    s.aux = bars + 2 * kMaxSlot + 1;
    s.tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kMaxSlot + 2);
    s.gdone = bars + 2 * kMaxSlot + 3;
    return s;
}

template <int NS>
__device__ __forceinline__ void tc_prologue(const TcShared& s, uint32_t ncols, Ring& ring, const TcPlan& plan, uint32_t my_tiles, bool w0) {
    if (threadIdx.x < 32) tmem_alloc(s.tmem_slot, ncols);
    if (threadIdx.x == 0) {
        for (int i = 0; i < kMaxSlot; ++i) { mbar_init(&s.full[i], 1); mbar_init(&s.empty[i], 1); }
        mbar_init(s.done, 1);
        mbar_init(s.aux, 1);
        for (int i = 0; i < kMaxGroups; ++i) mbar_init(&s.gdone[i], 1);
        mbar_fence_init();
    }
    for (int i = threadIdx.x; i < 2 * TM; i += blockDim.x)
        reinterpret_cast<float4*>(s.ones)[i] = i < TM ? make_float4(1.f, 1.f, 0.f, 0.f) : make_float4(0.f, 0.f, 0.f, 0.f);
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    ring.wsm = s.wsm; ring.full = s.full; ring.empty = s.empty; ring.sched = s.sched;
    ring.pidx = ring.pcnt = ring.ccnt = 0;
    ring.pslot = ring.puse = ring.cslot = ring.cpar = 0;
    uint32_t nb = 0;
    for (int i = 0; i < plan.ngemm; ++i) nb += plan.g[i].nblk;
    ring.nsched = nb;
    ring.to_load = nb * my_tiles;
    if (w0 && elect_one()) {      // the elected lane of warp 0 owns the ring state and issues every MMA
        if (plan.resident) { ring_load_all(ring, plan); mbar_wait(&s.full[0], 0); }
        else {
            uint32_t cnt;
            ring_build_schedule(s.sched, plan, &cnt);
            ring_top_up<NS>(ring, plan);
        }
    }
}
__device__ __forceinline__ void tc_finish(uint32_t tm, uint32_t ncols) {
    fence_before_sync();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc(tm, ncols);
}
// all threads: operand region written -> visible to the tensor core, TMEM reads retired
template <int NG = 1, int NTG = NT2>
__device__ __forceinline__ void sync_for_mma(int grp = 0) {
    fence_async_smem();
    fence_before_sync();
    group_sync<NG, NTG>(grp);
    fence_after_sync();
}
// One thread polls the mbarrier; everybody else parks on the (hardware-blocking) CTA barrier instead of
// spinning -- 255 spinning threads per CTA took ~40 % of the SM's issue slots away from co-resident CTAs.
__device__ __forceinline__ void wait_done(uint64_t* done, uint32_t& phase) {
    if (threadIdx.x == 0) mbar_wait(done, phase & 1);
    __syncthreads();
    ++phase;
    fence_after_sync();
}
// same, and the issuing lane refills the (now entirely free) weight ring before joining the barrier
template <typename G, int NG = 1, int NTG = NT2>
__device__ __forceinline__ void wait_done_ring(uint64_t* done, uint32_t& phase, Ring& r, const TcPlan& p, bool w0, int grp = 0) {
    if (w0 && elect_one()) {
        mbar_wait(done, phase & 1);
        if (!G::resident) ring_top_up<G::nslot>(r, p);
    }
    group_sync<NG, NTG>(grp);
    ++phase;
    fence_after_sync();
}

struct UnitGeom {
    int h, w, fh, fw;       // level size, grid-cell extent
    int upi;                // units (64 tokens) per image
    int total_units;        // over the batch chunk
    float inv_upi, inv_fw, inv_bw;   // reciprocals for fast_div (bw = w / 8)
};
// n / d for 0 <= n < 2^23, d >= 1: float-reciprocal estimate (off by at most one) + exact fix-up; ~8 instructions instead of
// the ~25 of the integer division sequence (coords() ran it three times per tile on every thread)
__device__ __forceinline__ int fast_div(int n, int d, float inv_d) {
    int q = __float2int_rz(__int2float_rn(n) * inv_d);
    const int r = n - q * d;
    q += (r >= d) ? 1 : 0;
    q -= (r < 0) ? 1 : 0;
    return q;
}

// pixel index (inside its image) of token `tok` of unit `u`
template <int KIND>   // 0 grid, 1 block, 2 linear
__device__ __forceinline__ int unit_pixel(const UnitGeom& g, int u, int tok) {
    if (KIND == 0) { const int fy = fast_div(u, g.fw, g.inv_fw), fx = u - fy * g.fw; return ((tok >> 3) * g.fh + fy) * g.w + (tok & 7) * g.fw + fx; }
    if (KIND == 1) { const int bw = g.w >> 3, by = fast_div(u, bw, g.inv_bw), bx = u - by * bw; return (by * 8 + (tok >> 3)) * g.w + bx * 8 + (tok & 7); }
    return u * 64 + tok;
}

// ---- full-sector global accesses.  A lane owns one pixel row and moves it in 16-byte chunks, so "chunk j of 32 rows"
// is a warp instruction over 32 half-used 32-byte sectors, which the LSU serialises.  Lanes 2i / 2i+1 instead access the
// two halves of ONE sector of row 2i, then of row 2i+1, and swap every other chunk by shuffle: 16 full sectors per
// instruction.  (Both lanes of a pair always belong to the same unit, so `valid` is pair-uniform.)
__device__ __forceinline__ float4 shfl_xor1(float4 v) {
    return make_float4(__shfl_xor_sync(0xffffffffu, v.x, 1), __shfl_xor_sync(0xffffffffu, v.y, 1),
                       __shfl_xor_sync(0xffffffffu, v.z, 1), __shfl_xor_sync(0xffffffffu, v.w, 1));
}
// raw pair-layout load of N chunks: v[2k] = row 2i chunk 2k + odd, v[2k+1] = row 2i+1 chunk 2k + odd
template <int N>
__device__ __forceinline__ void pair_load(const float4* own, bool valid, float4 (&v)[N]) {
    static_assert(N % 2 == 0, "pairs of chunks");
    const bool odd = (threadIdx.x & 1) != 0;
    const float4* oth = reinterpret_cast<const float4*>(__shfl_xor_sync(0xffffffffu, (unsigned long long)own, 1));
    const float4* a = (odd ? oth : own) + (odd ? 1 : 0);
    const float4* b = (odd ? own : oth) + (odd ? 1 : 0);
#pragma unroll
    for (int k = 0; k < N; k += 2) {
        v[k] = valid ? __ldg(a + k) : make_float4(0.f, 0.f, 0.f, 0.f);
        v[k + 1] = valid ? __ldg(b + k) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
}
// store this lane's N consecutive chunks, taken from v[4 * j ..], at out + own_off (floats) with full sectors
template <int N>
__device__ __forceinline__ void pair_store(float* __restrict__ out, size_t own_off, const float* v, bool valid) {
    static_assert(N % 2 == 0, "pairs of chunks");
    const bool odd = (threadIdx.x & 1) != 0;
    const size_t oth_off = __shfl_xor_sync(0xffffffffu, (unsigned long long)own_off, 1);
    const size_t off_a = (odd ? oth_off : own_off) + (odd ? 4 : 0), off_b = (odd ? own_off : oth_off) + (odd ? 4 : 0);
#pragma unroll
    for (int j = 0; j < N; j += 2) {
        const float4 c0 = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        const float4 c1 = make_float4(v[4 * j + 4], v[4 * j + 5], v[4 * j + 6], v[4 * j + 7]);
        const float4 recv = shfl_xor1(odd ? c0 : c1);
        if (valid) {
            *reinterpret_cast<float4*>(out + off_a + 4 * j) = odd ? recv : c0;      // row 2i,     chunk j + odd
            *reinterpret_cast<float4*>(out + off_b + 4 * j) = odd ? c1 : recv;      // row 2i + 1, chunk j + odd
        }
    }
}
// ---- full-LINE global accesses.  The pair layout above still touches 16 different 128-byte lines per warp instruction, and the
// L1 processes one line per ~2 cycles (the stage 3-4 kernels, whose rows are 512-1024 bytes apart, spent a quarter to a half of
// their time queued there while every ncu pipe looked idle).  Groups of 8 lanes (8 consecutive rows) transpose 8 x 8 blocks of
// 16-byte chunks by shuffle so that each group writes 128 contiguous bytes of ONE row per instruction: 4 lines per instruction.
__device__ __forceinline__ float4 shfl_xor_f4(float4 v, int m) {
    return make_float4(__shfl_xor_sync(0xffffffffu, v.x, m), __shfl_xor_sync(0xffffffffu, v.y, m),
                       __shfl_xor_sync(0xffffffffu, v.z, m), __shfl_xor_sync(0xffffffffu, v.w, m));
}
// a[k] on lane j (of its group of 8) <-> a[j] on lane k
__device__ __forceinline__ void transpose8(float4 (&a)[8]) {
    const int j = threadIdx.x & 7;
#pragma unroll
    for (int s = 4; s >= 1; s >>= 1) {
        const bool up = (j & s) != 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if ((k & s) != 0) continue;
            const float4 recv = shfl_xor_f4(up ? a[k] : a[k | s], s);
            if (up) a[k] = recv; else a[k | s] = recv;
        }
    }
}
// store this lane's N consecutive chunks (v[4 * c ..]) of its row at out + own_off (floats); the rows of a group of 8 lanes are
// `stride` floats apart (consecutive pixels of a channels-last tensor) and share `valid`
template <int N>
__device__ __forceinline__ void oct_store(float* __restrict__ out, size_t own_off, int stride, const float* v, bool valid) {
    static_assert(N % 8 == 0, "blocks of 8 chunks");
    const int j = threadIdx.x & 7;
    float* const base = out + own_off - (size_t)j * stride + 4 * j;      // row 0 of the group, this lane's chunk column
#pragma unroll
    for (int c0 = 0; c0 < N; c0 += 8) {
        float4 a[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) a[c] = make_float4(v[4 * (c0 + c)], v[4 * (c0 + c) + 1], v[4 * (c0 + c) + 2], v[4 * (c0 + c) + 3]);
        transpose8(a);                                                     // a[k] = chunk c0 + j of row k
        if (valid) {
#pragma unroll
            for (int k = 0; k < 8; ++k) *reinterpret_cast<float4*>(base + (size_t)k * stride + 4 * c0) = a[k];
        }
    }
}
// the mirror image: N consecutive chunks of this lane's row, loaded as full lines and transposed back
template <int N>
__device__ __forceinline__ void oct_load(const float* __restrict__ in, size_t own_off, int stride, bool valid, float4 (&v)[N]) {
    static_assert(N % 8 == 0, "blocks of 8 chunks");
    const int j = threadIdx.x & 7;
    const float* const base = in + own_off - (size_t)j * stride + 4 * j;
#pragma unroll
    for (int c0 = 0; c0 < N; c0 += 8) {
        float4 a[8];
#pragma unroll
        for (int k = 0; k < 8; ++k)
            a[k] = valid ? __ldg(reinterpret_cast<const float4*>(base + (size_t)k * stride + 4 * c0)) : make_float4(0.f, 0.f, 0.f, 0.f);
        transpose8(a);
#pragma unroll
        for (int c = 0; c < 8; ++c) v[c0 + c] = a[c];
    }
}
// pair layout -> this lane's own chunks k, k+1 (call with the same k on every lane)
__device__ __forceinline__ void pair_unswap(float4& c0, float4& c1) {
    const bool odd = (threadIdx.x & 1) != 0;
    const float4 recv = shfl_xor1(odd ? c0 : c1);
    if (odd) c0 = recv; else c1 = recv;
}

// this thread's part (1 / TPR) of a pixel row of the level input -> A operand (chunk-major, 128 rows), K padded to >= 8
// H16: 1 = the operand is fp16 (two 4-channel chunks -> one 16-byte chunk of 8 halves), 2 = fp16 hi + lo (lo chunks CIN / 8 further)
// ostride > 0: the rows of a group of 8 lanes are `ostride` floats apart -> full-line loads (oct_load) instead of the pair layout
template <int CIN, int TPR = 2, int H16 = 0>
__device__ __forceinline__ void load_input_row(const float* __restrict__ xin, size_t npix, size_t img, int pix, bool valid,
                                               float* dst, int row, int half, int ostride = 0) {
    if constexpr (CIN < 8) {                       // NCHW network input: part 0 gathers the planes, part 1 zero-fills
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
        if (half == 0 && valid) {
            float v[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int c = 0; c < CIN; ++c) v[c] = __ldg(xin + (img * CIN + c) * npix + pix);
            o = to_tf32(make_float4(v[0], v[1], v[2], v[3]));
        }
        if (half < 2) *reinterpret_cast<float4*>(dst + ((size_t)half * TM + row) * 4) = o;
    } else if constexpr (H16 == 3) {
        // the level input is already fp16, channels-last [pixel][CIN halves] (written by pool_kernel for this path): its 16-byte
        // chunks ARE operand chunks -- half the bytes of the fp32 tensor, no conversion (every consumer rounded it to fp16 anyway)
        constexpr int N16 = CIN / (8 * TPR);
        const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(xin) + (img * npix + pix) * CIN) + half * N16;
        uint4 v[N16];
#pragma unroll
        for (int j = 0; j < N16; ++j) v[j] = valid ? __ldg(src + j) : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
        for (int j = 0; j < N16; ++j) *reinterpret_cast<uint4*>(dst + ((size_t)(half * N16 + j) * TM + row) * 4) = v[j];
    } else {
        constexpr int N = CIN / (4 * TPR), NB = N > 8 ? 8 : N;          // batches of 8 chunks bound the registers in flight
        const float4* src = reinterpret_cast<const float4*>(xin + (img * npix + pix) * CIN) + half * N;
#pragma unroll 1
        for (int j0 = 0; j0 < N; j0 += NB) {
            float4 v[NB];
            const bool oct = NB % 8 == 0 && ostride > 0;        // (uniform)
            if constexpr (NB % 8 == 0) {
                if (oct) oct_load<NB>(xin, (img * npix + pix) * CIN + (size_t)(half * N + j0) * 4, ostride, valid, v);
                else pair_load<NB>(src + j0, valid, v);
            } else {
                pair_load<NB>(src + j0, valid, v);
            }
#pragma unroll
            for (int j = 0; j < NB; j += 2) {
                if (!oct) pair_unswap(v[j], v[j + 1]);
                if constexpr (H16 != 0) {
                    const float e[8] = {v[j].x, v[j].y, v[j].z, v[j].w, v[j + 1].x, v[j + 1].y, v[j + 1].z, v[j + 1].w};
                    uint32_t h[4], l[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        if constexpr (H16 == 2) split_h2(e[2 * q], e[2 * q + 1], h[q], l[q]);
                        else asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h[q]) : "f"(e[2 * q + 1]), "f"(e[2 * q]));
                    }
                    *reinterpret_cast<uint4*>(dst + ((size_t)((half * N + j0 + j) / 2) * TM + row) * 4) = make_uint4(h[0], h[1], h[2], h[3]);
                    if constexpr (H16 == 2)
                        *reinterpret_cast<uint4*>(dst + ((size_t)(CIN / 8 + (half * N + j0 + j) / 2) * TM + row) * 4) = make_uint4(l[0], l[1], l[2], l[3]);
                } else {
                    *reinterpret_cast<float4*>(dst + ((size_t)(half * N + j0 + j) * TM + row) * 4) = to_tf32(v[j]);
                    *reinterpret_cast<float4*>(dst + ((size_t)(half * N + j0 + j + 1) * TM + row) * 4) = to_tf32(v[j + 1]);
                }
            }
        }
    }
}

// Software prefetch of the level input (CIN <= 64: at most 8 float4 per thread): the next tile's rows are requested
// right after the current tile's operand is stored, so the ~2000-cycle global-load latency at the top of every tile
// (scripts/tc_trace.py) hides under the tile's six GEMM phases.
template <int CIN, int TPR = 2> struct InputPf {
    static constexpr int N = CIN < 8 ? 1 : CIN / (4 * TPR);
    static constexpr bool enabled = CIN <= 64;
    float4 v[N];
};
template <int CIN, bool PAIR = true, int TPR = 2, bool XH = false>      // XH: fp16 level input (see load_input_row, mode 3)
__device__ __forceinline__ void fetch_input_row(const float* __restrict__ xin, size_t npix, size_t img, int pix, bool valid, int half,
                                                InputPf<CIN, TPR>& pf) {
    if constexpr (XH && CIN >= 8) {
        constexpr int N16 = CIN / (8 * TPR);
        const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(xin) + (img * npix + pix) * CIN) + half * N16;
#pragma unroll
        for (int j = 0; j < N16; ++j) {
            const uint4 u = valid ? __ldg(src + j) : make_uint4(0u, 0u, 0u, 0u);
            pf.v[j] = make_float4(__uint_as_float(u.x), __uint_as_float(u.y), __uint_as_float(u.z), __uint_as_float(u.w));
        }
        return;
    }
    if constexpr (CIN < 8) {                       // conv.0 runs on the CUDA cores: every part of the row needs the pixel
        float v[4] = {0.f, 0.f, 0.f, 0.f};
        if (valid) {
#pragma unroll
            for (int c = 0; c < CIN; ++c) v[c] = __ldg(xin + (img * CIN + c) * npix + pix);
        }
        pf.v[0] = make_float4(v[0], v[1], v[2], v[3]);
    } else {
        constexpr int N = InputPf<CIN, TPR>::N;
        const float4* src = reinterpret_cast<const float4*>(xin + (img * npix + pix) * CIN) + half * N;
        if constexpr (PAIR) {
            pair_load<N>(src, valid, pf.v);           // pair layout; un-swapped when stored (store_input_row)
        } else {
#pragma unroll
            for (int j = 0; j < N; ++j) pf.v[j] = valid ? __ldg(src + j) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
}
template <int CIN, bool PAIR = true, int TPR = 2, int H16 = 0>
__device__ __forceinline__ void store_input_row(const InputPf<CIN, TPR>& pf, float* dst, int row, int half) {
    if constexpr (H16 == 3 && CIN >= 8) {
        constexpr int N16 = CIN / (8 * TPR);
#pragma unroll
        for (int j = 0; j < N16; ++j) *reinterpret_cast<float4*>(dst + ((size_t)(half * N16 + j) * TM + row) * 4) = pf.v[j];
        return;
    }
    if constexpr (CIN < 8) {
        if (half < 2) *reinterpret_cast<float4*>(dst + ((size_t)half * TM + row) * 4) = to_tf32(pf.v[0]);
    } else {
        constexpr int N = InputPf<CIN, TPR>::N;
#pragma unroll
        for (int j = 0; j < N; j += 2) {
            float4 c0 = pf.v[j], c1 = pf.v[j + 1];
            if constexpr (PAIR) pair_unswap(c0, c1);
            if constexpr (H16 != 0) {            // two 4-channel chunks -> one 16-byte chunk of 8 halves
                const float e[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
                uint32_t h[4], l[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    if constexpr (H16 == 2) split_h2(e[2 * q], e[2 * q + 1], h[q], l[q]);
                    else asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h[q]) : "f"(e[2 * q + 1]), "f"(e[2 * q]));
                }
                *reinterpret_cast<uint4*>(dst + ((size_t)((half * N + j) / 2) * TM + row) * 4) = make_uint4(h[0], h[1], h[2], h[3]);
                if constexpr (H16 == 2)
                    *reinterpret_cast<uint4*>(dst + ((size_t)(CIN / 8 + (half * N + j) / 2) * TM + row) * 4) = make_uint4(l[0], l[1], l[2], l[3]);
            } else {
                *reinterpret_cast<float4*>(dst + ((size_t)(half * N + j) * TM + row) * 4) = to_tf32(c0);
                *reinterpret_cast<float4*>(dst + ((size_t)(half * N + j + 1) * TM + row) * 4) = to_tf32(c1);
            }
        }
    }
}


// ---- network input stage (CIN < 8): conv.0 has K = 3, so x0 = ReLU(conv.0(x)) is 3 FMAs per channel on the CUDA cores
// (exact fp32) instead of a whole MMA phase (operand store, two barriers, commit / wait round trip, tcgen05.ld).
// Weights sit in shared memory as cw[k][C] (k < CIN) followed by the bias [C]  (vec + kConv0Off).
constexpr int kConv0Off = 64;
template <int CIN, int C>
__device__ __forceinline__ void conv0_stage_weights(const DownW& w, float* vec) {
    for (int i = threadIdx.x; i < CIN * C; i += NT2) vec[kConv0Off + i] = __ldg(w.conv0_w + i);
    for (int i = threadIdx.x; i < C; i += NT2) vec[kConv0Off + CIN * C + i] = __ldg(w.conv0_b + i);
}
template <int CIN, int C, int CH>
__device__ __forceinline__ void conv0_row(const float4 x, const float* vec, int col0, float (&v)[CH]) {
    const float xs[4] = {x.x, x.y, x.z, x.w};
    const float* cw = vec + kConv0Off + col0;
#pragma unroll
    for (int i = 0; i < CH; i += 4) {
        const float4 b = *reinterpret_cast<const float4*>(cw + CIN * C + i);
        unsigned long long a01 = pk2(b.x, b.y), a23 = pk2(b.z, b.w);
#pragma unroll
        for (int k = 0; k < CIN; ++k) {
            const float4 wv = *reinterpret_cast<const float4*>(cw + k * C + i);
            const unsigned long long xk = pk2(xs[k], xs[k]);
            a01 = fma2(pk2(wv.x, wv.y), xk, a01);
            a23 = fma2(pk2(wv.z, wv.w), xk, a23);
        }
        upk2(a01, v[i], v[i + 1]);
        upk2(a23, v[i + 2], v[i + 3]);
#pragma unroll
        for (int j = 0; j < 4; ++j) v[i + j] = fmaxf(v[i + j], 0.f);
    }
}

// ------------------------------------------------------------------------------------------ branch kernel
// One configuration per stage.  TPR = threads per pixel row (each owns C / TPR channels), groups = tile groups per CTA:
//   C = 32:       one thread per row, five tile groups: half the per-row overhead instructions (address arithmetic, barriers,
//                 LayerNorm exchanges) of a kernel that is bound by instruction issue -- -30 % instructions, -13 % time
//                 against two threads per row
//   C = 64, 128:  two threads per row (two tile groups at C = 64); four threads per row measured no gain
//   C = 256:      four threads per row: 16 epilogue warps instead of 8 on an SM whose epilogues are latency-bound, -10 %
// PX = 1: split precision (fp16 hi + lo operands, see BranchG).
template <int C, int PX> struct BranchCfg {
    static constexpr int TPR = C == 32 ? 1 : C == 256 ? 4 : 2;
    static constexpr int groups = C == 32 ? 5 : C == 64 ? 2 : 1;   // tile groups per CTA (shared resident weights)
    static constexpr int NTG = TM * TPR;                           // threads per tile group
    static constexpr int CH = C / TPR;
    // operand region of a group: the [128 x C] A operand (hi chunks, then lo chunks: PX); the token mixing reads the same layout
    static constexpr uint32_t region = (uint32_t)TM * C * (PX ? 4u : 2u);
    static constexpr bool park_u = C <= 128;                       // u stays in TMEM (else it round-trips through `out`)
    static constexpr bool h16_out = C <= 128;                      // u' / v' leave as fp16 tiles [C / 8 chunks][128 pixels][8 halves]: the operand
                                                                   // layout of the merge kernel's kind::f16 dense2, half the HBM bytes
    static constexpr int col_u = 0;
    static constexpr int col_y = park_u ? C : 0;
    static constexpr int ncols = groups * tc_cols(col_y + 2 * C) > 512 ? col_y + 2 * C : tc_cols(col_y + 2 * C);   // TMEM columns per group
    static constexpr uint32_t xch = TPR == 1 ? 0u : 2u * TPR * TM * 8u;   // LayerNorm exchange buffers per group
    static constexpr int SC = TPR == 1 ? 16 : TPR == 4 ? (CH < 32 ? CH : 32) : (CH > 64 ? 64 : CH);   // sub-chunks bound the live registers
};

template <int CIN, int C, int BR, int PX>
__device__ __forceinline__ void tc_branch_body(const float* __restrict__ xin, const DownW& w, const TcPlan& plan, const UnitGeom& geo,
                                               float* __restrict__ out, float* __restrict__ scratch, unsigned char* smem) {
    using Cfg = BranchCfg<C, PX>;
    using G = BranchG<CIN, C, PX>;
    constexpr int CH = Cfg::CH, NG = Cfg::groups, TPR = Cfg::TPR, NTG = Cfg::NTG, SC = Cfg::SC;
    constexpr bool X3 = PX != 0;
    constexpr int LOC = X3 ? C / 8 : 0;                                   // lo chunks of an A operand follow its C / 8 hi chunks
    constexpr bool XH = !X3 && CIN >= 8;                                  // the level input arrives as fp16 (pool_kernel, single-rounded path)
    // stage 4, single-rounded path: u' / v' leave as fp16 channels-last rows (the merge kernel's loaders take their 16-byte chunks as
    // operand chunks, like the pooled level inputs); the fp32 residual u then round-trips through `scratch`, not through `out`
    constexpr bool CL16 = !Cfg::h16_out && !X3;
    float* const rt = CL16 ? scratch : out;
    constexpr int XM = XH ? 3 : X3 ? 2 : 1;
    static_assert(NG == 1 || G::resident, "tile groups share resident weights (no ring state per group)");
    static_assert(CH % SC == 0 && SC % 16 == 0, "sub-chunking");
    TcShared s = carve(smem, Cfg::region, plan, NG, Cfg::xch);
    const int grp = NG == 1 ? 0 : (int)(threadIdx.x / NTG);               // tile group (warp-uniform)
    const int tid = threadIdx.x - grp * NTG, row = tid & (TM - 1), half = tid >> 7;   // half = which part of the row
    const int vblock = (int)blockIdx.x * NG + grp, vgrid = (int)gridDim.x * NG;   // this group as a virtual CTA
    const int ntiles = (geo.total_units + 1) / 2;
    const uint32_t my_tiles = vblock < ntiles ? (ntiles - 1 - vblock) / vgrid + 1 : 0;
    const DownW::Branch& br = w.br[BR];
    if (grp == 0) {
        for (int i = tid; i < C; i += NTG) { s.vec[i] = __ldg(br.gn_w + i); s.vec[256 + i] = __ldg(br.gn_b + i); }
        for (int i = tid; i < 64; i += NTG) s.vec[512 + i] = __ldg(br.gd_b + i) + 1.0f;
        if constexpr (CIN < 8) {
            for (int i = tid; i < CIN * C; i += NTG) s.vec[kConv0Off + i] = __ldg(w.conv0_w + i);
            for (int i = tid; i < C; i += NTG) s.vec[kConv0Off + CIN * C + i] = __ldg(w.conv0_b + i);
        }
    }
    Ring ring;
    const bool w0 = __shfl_sync(0xffffffffu, tid >> 5, 0) == 0;           // first warp of the group: issues its MMAs
    tc_prologue<G::nslot>(s, tc_cols(Cfg::ncols * NG), ring, plan, my_tiles, w0 && grp == 0);
    if (NG > 1) {
        if (grp > 0 && w0 && elect_one()) mbar_wait(&s.full[0], 0);       // the resident weights (loaded by group 0) have landed
        s.region += (size_t)grp * (Cfg::region / 4);
        s.xch += (size_t)grp * (Cfg::xch / 8);
        if (grp > 0) s.done = &s.gdone[grp];
    }
    const uint32_t tm = *s.tmem_slot + (uint32_t)(grp * Cfg::ncols);
    const uint32_t lane_base = tm + ((uint32_t)(row & ~31) << 16);        // this warp's 32-lane window
    const uint32_t region_addr = smem_u32(s.region), ones_addr = smem_u32(s.ones);
    const int ug = (row & 31) >> 4, tok = (row >> 5) * 16 + (row & 15);   // unit / token of this lane
    const int col0 = half * CH;                                           // this thread's channel range
    // mixing bias + 1 of this lane's token, from shared memory (vec[512 + tok]): as a register the compiler re-loaded it from
    // global memory in every tile (7 % of the stage-2 kernel's stall samples on that one load)
    const float* const mix_b1p = s.vec + 512 + tok;
    // float distance between the rows of 8 consecutive lanes (8 consecutive tokens: a block row, or 8 grid cells fw pixels apart)
    const int ostride = (BR == 0 ? geo.fw : 1) * C;
    const size_t npix = (size_t)geo.h * geo.w;
    uint32_t phase = 0, xb = 0;
    int it = 0;
    InputPf<CIN, TPR> pf;
    auto coords = [&](int tt, bool& vld, int& im, int& px) {
        const int un = 2 * tt + ug;
        vld = un < geo.total_units;
        im = vld ? fast_div(un, geo.upi, geo.inv_upi) : 0;
        px = unit_pixel<BR>(geo, vld ? un - im * geo.upi : 0, tok);
    };
    auto stats_of = [&](const float (&v)[CH], float& sum, float& sq) {
        unsigned long long s2 = pk2(0.f, 0.f), q2 = pk2(0.f, 0.f);
#pragma unroll
        for (int i = 0; i < CH; i += 2) {
            const unsigned long long x = pk2(v[i], v[i + 1]);
            s2 = add2(s2, x); q2 = fma2(x, x, q2);
        }
        float a, b;
        upk2(s2, a, b); sum = a + b;
        upk2(q2, a, b); sq = a + b;
    };
    // (the coordinates of the prefetched tile are carried into its iteration: the unit -> pixel arithmetic ran twice per tile)
    bool nvld = false; int nim = 0, npx = 0;
    if (InputPf<CIN, TPR>::enabled && vblock < ntiles) {
        coords(vblock, nvld, nim, npx);
        fetch_input_row<CIN, true, TPR, XH>(xin, npix, (size_t)nim, npx, nvld, half, pf);
    }
    for (int t = vblock; t < ntiles; t += vgrid, ++it) {
        TC_TRACE(plan, it, 0);
        bool valid; int img, pix;
        if (InputPf<CIN, TPR>::enabled && (TPR > 1 || !X3)) { valid = nvld; img = nim; pix = npx; }   // (split precision at one thread per row: no registers to spare)
        else coords(t, valid, img, pix);
        float* orow = rt + ((size_t)img * npix + pix) * C + col0;
        float v[CH], rstd, shift;
        // ---- x -> conv.0 -> ReLU -> LayerNorm (affine folded into dense1)
        if constexpr (CIN < 8) {
            const float4 xv = pf.v[0];
            if (t + vgrid < ntiles) {
                coords(t + vgrid, nvld, nim, npx);
                fetch_input_row<CIN, true, TPR, XH>(xin, npix, (size_t)nim, npx, nvld, half, pf);
            }
            conv0_row<CIN, C, CH>(xv, s.vec, col0, v);
        } else {
            if (InputPf<CIN, TPR>::enabled) {
                store_input_row<CIN, true, TPR, XM>(pf, s.region, row, half);
                if (t + vgrid < ntiles) {
                    coords(t + vgrid, nvld, nim, npx);
                    fetch_input_row<CIN, true, TPR, XH>(xin, npix, (size_t)nim, npx, nvld, half, pf);
                }
            } else {
                load_input_row<CIN, TPR, XM>(xin, npix, (size_t)img, pix, valid, s.region, row, half);
            }
            TC_TRACE(plan, it, 1);
            sync_for_mma<NG, NTG>(grp);
            if (w0 && elect_one()) { issue_linear_t<G, BG_CONV0>(ring, plan, region_addr, ones_addr, tm + Cfg::col_y, true); commit(s.done); }
            TC_TRACE(plan, it, 2);
            wait_done_ring<G, NG, NTG>(s.done, phase, ring, plan, w0, grp);
            TC_TRACE(plan, it, 3);
            ld_row<CH>(lane_base + Cfg::col_y + col0, v);
#pragma unroll
            for (int i = 0; i < CH; ++i) v[i] = fmaxf(v[i], 0.f);
        }
        {
            float sum, sq;
            stats_of(v, sum, sq);
            row_stats<NG, TPR>(sum, sq, s.xch + (xb++ & 1) * TPR * TM, row, half, C, rstd, shift, grp);
            norm_row<CH>(v, rstd, shift);
            row_to_a16<CH, LOC>(v, s.region, row, col0);
        }
        TC_TRACE(plan, it, 4);
        sync_for_mma<NG, NTG>(grp);
        // ---- this branch's half of dense1 -> GELU = u (residual, parked) -> LayerNorm (affine folded into gMLP dense1)
        if (w0 && elect_one()) { issue_linear_t<G, BG_PD1>(ring, plan, region_addr, ones_addr, tm + Cfg::col_u, true); commit(s.done); }
        TC_TRACE(plan, it, 5);
        wait_done_ring<G, NG, NTG>(s.done, phase, ring, plan, w0, grp);
        TC_TRACE(plan, it, 6);
        {
            ld_row<CH>(lane_base + Cfg::col_u + col0, v);
            float sum = 0.f, sq = 0.f;
            gelu_row<CH, true>(v, sum, sq);
            if (Cfg::park_u) st_row<CH>(lane_base + Cfg::col_u + col0, v);
            else if constexpr (CH % 32 == 0 && !X3) oct_store<CH / 4>(rt, ((size_t)img * npix + pix) * C + col0, ostride, v, valid);
            else pair_store<CH / 4>(rt, ((size_t)img * npix + pix) * C + col0, v, valid);
            row_stats<NG, TPR>(sum, sq, s.xch + (xb++ & 1) * TPR * TM, row, half, C, rstd, shift, grp);
            norm_row<CH>(v, rstd, shift);
            row_to_a16<CH, LOC>(v, s.region, row, col0);
        }
        TC_TRACE(plan, it, 7);
        sync_for_mma<NG, NTG>(grp);
        // ---- gMLP dense1 (two halves) -> GELU; y1 parked, y2 -> LayerNorm -> [channel][token] operand
        if (w0 && elect_one()) {
            issue_linear_t<G, BG_D1A>(ring, plan, region_addr, ones_addr, tm + Cfg::col_y, true);
            issue_linear_t<G, BG_D1B>(ring, plan, region_addr, ones_addr, tm + Cfg::col_y + C, true);
            commit(s.done);
        }
        TC_TRACE(plan, it, 8);
        wait_done_ring<G, NG, NTG>(s.done, phase, ring, plan, w0, grp);
        TC_TRACE(plan, it, 9);
        {
            ld_row<CH>(lane_base + Cfg::col_y + col0, v);
            { float d0, d1; gelu_row<CH, false>(v, d0, d1); }
            st_row<CH>(lane_base + Cfg::col_y + col0, v);
            ld_row<CH>(lane_base + Cfg::col_y + C + col0, v);
            float sum = 0.f, sq = 0.f;
            gelu_row<CH, true>(v, sum, sq);
            row_stats<NG, TPR>(sum, sq, s.xch + (xb++ & 1) * TPR * TM, row, half, C, rstd, shift, grp);
            norm_row<CH>(v, rstd, shift);
#pragma unroll
            for (int i = 0; i < CH; i += 4) {
                const float4 gw = *reinterpret_cast<const float4*>(s.vec + col0 + i), gb = *reinterpret_cast<const float4*>(s.vec + 256 + col0 + i);
                upk2(fma2(pk2(v[i], v[i + 1]), pk2(gw.x, gw.y), pk2(gb.x, gb.y)), v[i], v[i + 1]);
                upk2(fma2(pk2(v[i + 2], v[i + 3]), pk2(gw.z, gw.w), pk2(gb.z, gb.w)), v[i + 2], v[i + 3]);
            }
            row_to_a16<CH, LOC>(v, s.region, row, col0);          // the mixing MMA reads it as an MN-major B operand (issue_mix_t)
        }
        TC_TRACE(plan, it, 10);
        sync_for_mma<NG, NTG>(grp);
        // ---- token mixing, gating y1 * (y2' + 1)
        if (w0 && elect_one()) { issue_mix_t<G, BG_WM, C>(ring, plan, region_addr, tm + Cfg::col_y + C); commit(s.done); }
        TC_TRACE(plan, it, 11);
        wait_done_ring<G, NG, NTG>(s.done, phase, ring, plan, w0, grp);
        TC_TRACE(plan, it, 12);
        {
#pragma unroll 1
            for (int c = 0; c < CH; c += SC) {
                float y1[SC], y2[SC];
                ld_row<SC>(lane_base + Cfg::col_y + col0 + c, y1);
                ld_row<SC>(lane_base + Cfg::col_y + C + col0 + c, y2);
                const float mix_b1 = *mix_b1p;
                const unsigned long long b2 = pk2(mix_b1, mix_b1);
#pragma unroll
                for (int i = 0; i < SC; i += 2) upk2(mul2(pk2(y1[i], y1[i + 1]), add2(pk2(y2[i], y2[i + 1]), b2)), y2[i], y2[i + 1]);
                row_to_a16<SC, LOC>(y2, s.region, row, col0 + c);
            }
        }
        TC_TRACE(plan, it, 13);
        sync_for_mma<NG, NTG>(grp);
        // ---- dense2 + residual u -> out
        if (w0 && elect_one()) { issue_linear_t<G, BG_D2>(ring, plan, region_addr, ones_addr, tm + Cfg::col_y, true); commit(s.done); }
        TC_TRACE(plan, it, 14);
        wait_done_ring<G, NG, NTG>(s.done, phase, ring, plan, w0, grp);
        TC_TRACE(plan, it, 15);
        {
            // Full-sector stores: a lane's row chunks are 16 bytes, so a warp store of "chunk j of 32 rows" touches 32
            // half-used sectors and the LSU serialises them (removing these stores bought 0.3-0.6 ms per kernel per 64
            // images).  Lanes 2i / 2i+1 therefore swap every other chunk: both lanes write the two halves of one 32-byte
            // sector of row 2i, then of row 2i+1 -- 16 full sectors per instruction.
            const bool odd = (threadIdx.x & 1) != 0;
            // (own_base counts elements of the tile format: halves of an fp16 tile -- twice as many per tile in split precision)
            const size_t own_base = Cfg::h16_out ? ((size_t)img * npix + (pix & ~(TM - 1))) * C * (X3 ? 2 : 1)
                                                 : ((size_t)img * npix + pix) * C;
            const size_t oth_base = __shfl_xor_sync(0xffffffffu, (unsigned long long)own_base, 1);
            const size_t base_a = odd ? oth_base : own_base, base_b = odd ? own_base : oth_base;   // rows 2i, 2i+1
            if constexpr (CL16 && CH % 64 == 0) {
                float hv[CH / 2];                                   // this thread's CH output channels as packed halves
#pragma unroll
                for (int c = 0; c < CH; c += SC) {
                    float a[SC];
                    ld_row<SC>(lane_base + Cfg::col_y + col0 + c, a);
#pragma unroll
                    for (int j0 = 0; j0 < SC / 4; j0 += 8) {
                        float4 t8[8];
                        pair_load<8>(reinterpret_cast<const float4*>(orow + c) + j0, valid, t8);
#pragma unroll
                        for (int j = 0; j < 8; j += 2) {
                            pair_unswap(t8[j], t8[j + 1]);
#pragma unroll
                            for (int u2 = 0; u2 < 2; ++u2) {
                                const float4 rr = t8[j + u2];
                                const int i = 4 * (j0 + j + u2);
                                uint32_t h0, h1;
                                asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h0) : "f"(a[i + 1] + rr.y), "f"(a[i] + rr.x));
                                asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h1) : "f"(a[i + 3] + rr.w), "f"(a[i + 2] + rr.z));
                                hv[(c + i) / 2] = __uint_as_float(h0);
                                hv[(c + i) / 2 + 1] = __uint_as_float(h1);
                            }
                        }
                    }
                }
                oct_store<CH / 8>(out, (((size_t)img * npix + pix) * C + col0) / 2, ostride / 2, hv, valid);
            } else
#pragma unroll 1
            for (int c = 0; c < CH; c += SC) {
                float a[SC], r[SC];
                ld_row<SC>(lane_base + Cfg::col_y + col0 + c, a);
                if (Cfg::park_u) ld_row<SC>(lane_base + Cfg::col_u + col0 + c, r);
                if constexpr (Cfg::h16_out) {
                    // fp16 tile of the merge kernel: chunk j (8 channels) of pixel row p sits at halves j * 1024 + p * 8 of the
                    // tile; a lane stores 16 bytes per chunk -- neighbouring pixels (the other unit of the tile in the grid
                    // branch, the same block row in the block branch) complete the 32-byte sectors.  fp16 has the 11-bit
                    // significand of the tf32 operand this value would otherwise be rounded to; satfinite guards the range.
                    __half* tile = reinterpret_cast<__half*>(out) + own_base + (size_t)(pix & (TM - 1)) * 8;
#pragma unroll
                    for (int j = 0; j < SC / 8; ++j) {
                        uint32_t h[4], l[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            float lo, hi;
                            upk2(add2(pk2(a[8 * j + 2 * e], a[8 * j + 2 * e + 1]), pk2(r[8 * j + 2 * e], r[8 * j + 2 * e + 1])), lo, hi);
                            if constexpr (X3) split_h2(lo, hi, h[e], l[e]);
                            else asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h[e]) : "f"(hi), "f"(lo));
                        }
                        if (valid) {
                            *reinterpret_cast<uint4*>(tile + (size_t)((col0 + c) / 8 + j) * (TM * 8)) = make_uint4(h[0], h[1], h[2], h[3]);
                            if constexpr (X3)      // split precision: the tile is the merge kernel's [hi chunks | lo chunks] A operand
                                *reinterpret_cast<uint4*>(tile + (size_t)(C / 8 + (col0 + c) / 8 + j) * (TM * 8)) = make_uint4(l[0], l[1], l[2], l[3]);
                        }
                    }
                    continue;
                }
                float4 o[SC / 4];
                if constexpr (!Cfg::park_u) {                // the residual u comes back from `out` (full-sector pair loads)
                    float4* rq = reinterpret_cast<float4*>(r);
#pragma unroll
                    for (int j0 = 0; j0 < SC / 4; j0 += 8) {
                        float4 t8[8];
                        pair_load<8>(reinterpret_cast<const float4*>(orow + c) + j0, valid, t8);
#pragma unroll
                        for (int j = 0; j < 8; j += 2) { pair_unswap(t8[j], t8[j + 1]); rq[j0 + j] = t8[j]; rq[j0 + j + 1] = t8[j + 1]; }
                    }
                }
#pragma unroll
                for (int j = 0; j < SC / 4; ++j) {
                    float4 res;
                    res = make_float4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
                    o[j] = make_float4(a[4 * j] + res.x, a[4 * j + 1] + res.y, a[4 * j + 2] + res.z, a[4 * j + 3] + res.w);
                    // u' / v' feed nothing but the merge GEMM: rounding them here (RN, as every operand) lets the merge
                    // kernel stream them into its operand regions asynchronously, no register pass.  Low bits cleared:
                    // the C >= 128 merge kernels round again when they load, which must be a no-op
                    if (BR == 1 && !X3) o[j] = to_tf32_clean(o[j]);
                }
                if constexpr (SC % 32 == 0 && !X3) {      // full-line stores (see oct_store)
                    oct_store<SC / 4>(out, ((size_t)img * npix + pix) * C + col0 + c, ostride, reinterpret_cast<const float*>(o), valid);
                    continue;
                }
#pragma unroll
                for (int j = 0; j < SC / 4; j += 2) {
                    const float4 send = odd ? o[j] : o[j + 1];
                    float4 recv;
                    recv.x = __shfl_xor_sync(0xffffffffu, send.x, 1); recv.y = __shfl_xor_sync(0xffffffffu, send.y, 1);
                    recv.z = __shfl_xor_sync(0xffffffffu, send.z, 1); recv.w = __shfl_xor_sync(0xffffffffu, send.w, 1);
                    const float4 to_a = odd ? recv : o[j], to_b = odd ? o[j + 1] : recv;     // (row 2i, row 2i+1), chunk j + odd
                    const int chunk = (col0 + c) / 4 + j + (odd ? 1 : 0);
                    if (valid) {        // both lanes of a pair belong to the same unit
                        *reinterpret_cast<float4*>(out + base_a + 4 * chunk) = to_a;
                        *reinterpret_cast<float4*>(out + base_b + 4 * chunk) = to_b;
                    }
                }
            }
        }
        // the next tile's input load overwrites the region: every MMA reading it has completed (wait_done)
    }
    tc_finish(*s.tmem_slot, tc_cols(Cfg::ncols * NG));
}

template <int CIN, int C, int BR, int PX>
__global__ void __launch_bounds__(BranchCfg<C, PX>::NTG * BranchCfg<C, PX>::groups, 1)
tc_branch_kernel(const float* __restrict__ xin, DownW w, TcPlan plan, UnitGeom geo, float* __restrict__ out, float* __restrict__ scratch) {
    extern __shared__ __align__(1024) unsigned char smem[];
    tc_branch_body<CIN, C, BR, PX>(xin, w, plan, geo, out, scratch, smem);
}


// Channel sums of each unit (64 rows) of an exact-fp32 [128 x C] tile staged chunk-major in `reg` (squeeze input of the
// channel attention).  Every thread takes part: a group of TPP lanes owns one (unit, 4-channel chunk) pair, each lane adds
// 64 / TPP rows with float4 loads, then an xor butterfly inside the group -- a fixed order, so the result is bit-identical
// run to run.  (The first version used 2C threads x 64 dependent scalar loads: ~2000 cycles of exposed latency per tile.)
template <int C, int NTH = NT2>
__device__ __forceinline__ void unit_channel_sums(const float* reg, int t, int total_units, float* __restrict__ partial) {
    constexpr int CQ = C / 4, PAIRS = 2 * CQ, TPP = NTH / PAIRS, RPT = 64 / TPP;
    static_assert(TPP >= 2 && TPP <= 16, "group must fit in a warp");
    const int tid = threadIdx.x, pair = tid / TPP, sub = tid % TPP;
    const int uu = pair / CQ, ch = pair % CQ;
    const float4* src = reinterpret_cast<const float4*>(reg) + (size_t)ch * TM + uu * 64 + sub;
    float4 acc = src[0];
#pragma unroll
    for (int i = 1; i < RPT; ++i) {
        const float4 x = src[i * TPP];
        acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
    }
#pragma unroll
    for (int o = TPP / 2; o >= 1; o >>= 1) {
        acc.x += __shfl_xor_sync(0xffffffffu, acc.x, o);
        acc.y += __shfl_xor_sync(0xffffffffu, acc.y, o);
        acc.z += __shfl_xor_sync(0xffffffffu, acc.z, o);
        acc.w += __shfl_xor_sync(0xffffffffu, acc.w, o);
    }
    const int un = 2 * t + uu;
    if (sub == 0 && un < total_units) *reinterpret_cast<float4*>(partial + (size_t)un * C + ch * 4) = acc;
}

// ------------------------------------------------------------------------------------------ merge kernel
__device__ __forceinline__ int col0_of(int tid, int ch) { return (tid >> 7) * ch; }
template <int C, int PX = 0> struct MergeCfg {
    // threads per pixel row.  scripts/tc_trace.py at C = 128: the two epilogues that also store q / r take 5.6 k + 7.1 k of a
    // tile's 22 k cycles; four threads per row (16 warps) did not shorten them (0.85 -> 0.88 ms) -- the 16-byte-per-row global
    // stores touch 16 different 128-byte lines per warp instruction and queue in the L1 (one line per cycle), not in the issue slots
    static constexpr int TPR = 2;
    static constexpr int NT = TM * TPR;
    static constexpr uint32_t xch = 2u * TPR * TM * 8u;
    static constexpr int CH = C / TPR;
    // C = 128: u' and v' (swizzled panel tiles, tf32-rounded by the branch kernels) arrive by bulk copy -- u' into a second
    // region a tile ahead, v' into the first as soon as conv.0 has released it -- and conv.0 shares its phase with dense2(u')
    static constexpr bool bulk_uv = C == 128;
    static constexpr uint32_t uv_bytes = (uint32_t)TM * C * (PX ? 4u : 2u);                 // an fp16 u' / v' tile (hi + lo: PX)
    // compact layout (C = 128, single-rounded operands, resident weights): the u' tile lands in the second half of the fp32-sized
    // region, which the exact-fp32 staging of r (channel sums) overwrites at the end of the tile -- so the next u' is requested
    // after the sums and arrives under the next tile's input store and conv.0
    static constexpr bool two = C == 128 && PX == 0;
    static constexpr uint32_t r2_off = two ? (uint32_t)TM * C * 2 : (uint32_t)TM * C * 4;
    static constexpr uint32_t region = two ? (uint32_t)TM * C * 4 : (uint32_t)TM * C * 4 + (bulk_uv ? uv_bytes : 0u);   // + the u' tile
    static constexpr int col_x0 = 0, col_acc = C;
    static constexpr int ncols = tc_cols(2 * C);
    static constexpr int min_ctas = C <= 32 ? 3 : C <= 64 ? 2 : 1;
};

template <int CIN, int C, int PX = 0>
__global__ void __launch_bounds__(MergeCfg<C, PX>::NT, MergeCfg<C, PX>::min_ctas)
tc_merge_kernel(const float* __restrict__ xin, TcPlan plan, UnitGeom geo, const float* __restrict__ uin,
                const float* __restrict__ vin, float* __restrict__ rout, float* __restrict__ qout, float* __restrict__ partial, int r16) {
    extern __shared__ __align__(1024) unsigned char smem[];
    using Cfg = MergeCfg<C, PX>;
    using G = MergeG<CIN, C, PX>;
    constexpr int CH = Cfg::CH, TPR = Cfg::TPR, NTK = Cfg::NT;
    constexpr int HM = PX ? 2 : 1, LOC = PX ? C / 8 : 0;      // operand mode of the loaders, lo-chunk offset of a K = C operand
    constexpr bool XH = PX == 0 && CIN >= 8;                  // fp16 level input (pool_kernel, single-rounded path)
    constexpr int XM = XH ? 3 : HM;
    const TcShared s = carve(smem, Cfg::region, plan, 1, Cfg::xch);
    const int tid = threadIdx.x, row = tid & (TM - 1), half = tid >> 7;
    const int ntiles = (geo.total_units + 1) / 2;
    const uint32_t my_tiles = blockIdx.x < (unsigned)ntiles ? (ntiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;
    Ring ring;
    const bool w0 = warp0_uniform();
    tc_prologue<G::nslot>(s, Cfg::ncols, ring, plan, my_tiles, w0);
    const uint32_t tm = *s.tmem_slot;
    if constexpr (G::ebias) {             // fp32 biases of conv.0, dense2, conv1, conv2 -> vec[g * C + c] (first read after the next barrier)
        for (int i = tid; i < 4 * C; i += NTK) {
            const float2 e = __ldg(reinterpret_cast<const float2*>(plan.base + plan.ebias_off + (size_t)i * 4));
            s.vec[i] = e.x + e.y;
        }
    }
    const float* const eb = s.vec + col0_of(tid, CH);
    const uint32_t lane_base = tm + ((uint32_t)(row & ~31) << 16);
    const uint32_t region_addr = smem_u32(s.region), ones_addr = smem_u32(s.ones);
    const uint32_t r2_addr = region_addr + Cfg::r2_off;                     // bulk_uv: u' tiles land here
    uint64_t* const ld_u = s.aux;
    uint64_t* const ld_v = &s.gdone[1];
    constexpr uint32_t kTileBytes = Cfg::uv_bytes;                         // u' / v' tiles are fp16 (chunk-major; hi then lo chunks: PX)
    const size_t tile_floats = (size_t)kTileBytes / 4;                     // ... i.e. that many floats apart
    uint32_t ld_phase = 0;
    const int ug = row >> 6, tok = row & 63;
    const int col0 = half * CH;
    const size_t npix = (size_t)geo.h * geo.w;
    uint32_t phase = 0, xb = 0;
    int it = 0;
    InputPf<CIN, TPR> pf;                  // next tile's level input
    InputPf<C> pfu;                        // this tile's u' / v' rows, requested one phase ahead (C <= 32)
    auto coords = [&](int tt, bool& vld, int& im, int& px) {
        const int un = 2 * tt + ug;
        vld = un < geo.total_units;
        im = vld ? fast_div(un, geo.upi, geo.inv_upi) : 0;
        px = (vld ? un - im * geo.upi : 0) * 64 + tok;
    };
    if (InputPf<CIN, TPR>::enabled && (int)blockIdx.x < ntiles) {
        bool vld; int im, px;
        coords(blockIdx.x, vld, im, px);
        fetch_input_row<CIN, true, TPR, XH>(xin, npix, (size_t)im, px, vld, half, pf);
    }
    if (Cfg::bulk_uv && (int)blockIdx.x < ntiles && w0 && elect_one()) {
        mbar_expect_tx(ld_u, kTileBytes);
        bulk_load(r2_addr, uin + (size_t)blockIdx.x * tile_floats, kTileBytes, ld_u);
    }
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++it) {
        TC_TRACE(plan, it, 0);
        bool valid; int img, pix;
        coords(t, valid, img, pix);
        const size_t row_off = ((size_t)img * npix + pix) * C + col0;
        float v[CH];
        // ---- x0 = ReLU(conv.0(x)), parked
        if (InputPf<CIN, TPR>::enabled) {
            store_input_row<CIN, true, TPR, XM>(pf, s.region, row, half);
            if (t + (int)gridDim.x < ntiles) {
                bool vld; int im, px;
                coords(t + gridDim.x, vld, im, px);
                fetch_input_row<CIN, true, TPR, XH>(xin, npix, (size_t)im, px, vld, half, pf);
            }
        } else {
            load_input_row<CIN, TPR, XM>(xin, npix, (size_t)img, pix, valid, s.region, row, half, PX ? 0 : CIN);
        }
        if (InputPf<C>::enabled) fetch_input_row<C>(uin, npix, (size_t)img, pix, valid, half, pfu);
        TC_TRACE(plan, it, 1);
        sync_for_mma();
        if constexpr (Cfg::bulk_uv) {
            // ---- phase 1: conv.0(x) | dense2(u') (u' landed a tile ago); then v' -> region, next tile's u' -> second region
            if (w0 && elect_one()) {
                issue_linear_t<G, MG_CONV0>(ring, plan, region_addr, ones_addr, tm + Cfg::col_x0, true);
                mbar_wait(ld_u, ld_phase & 1);
                fence_after_sync();
                issue_linear_t<G, MG_PD2A>(ring, plan, r2_addr, ones_addr, tm + Cfg::col_acc, true);
                commit(s.done);
            }
            wait_done_ring<G>(s.done, phase, ring, plan, w0);
            if (w0 && elect_one()) {
                mbar_expect_tx(ld_v, kTileBytes);
                bulk_load(region_addr, vin + (size_t)t * tile_floats, kTileBytes, ld_v);
                if (!Cfg::two && t + (int)gridDim.x < ntiles) {
                    mbar_expect_tx(ld_u, kTileBytes);
                    bulk_load(r2_addr, uin + (size_t)(t + gridDim.x) * tile_floats, kTileBytes, ld_u);
                }
            }
            ld_row<CH>(lane_base + Cfg::col_x0 + col0, v);
#pragma unroll
            for (int i = 0; i < CH; ++i) v[i] = fmaxf(G::ebias ? v[i] + eb[i] : v[i], 0.f);
            st_row<CH>(lane_base + Cfg::col_x0 + col0, v);
            // ---- phase 2: dense2(v') accumulates (no thread wrote an operand: the elected lane issues as soon as v' is in)
            if (w0 && elect_one()) {
                mbar_wait(ld_v, ld_phase & 1);
                fence_after_sync();
                issue_linear_t<G, MG_PD2B>(ring, plan, region_addr, ones_addr, tm + Cfg::col_acc, false);
                commit(s.done);
            }
            ++ld_phase;
            wait_done_ring<G>(s.done, phase, ring, plan, w0);
        } else {
        if (w0 && elect_one()) { issue_linear_t<G, MG_CONV0>(ring, plan, region_addr, ones_addr, tm + Cfg::col_x0, true); commit(s.done); }
        TC_TRACE(plan, it, 2);
        wait_done_ring<G>(s.done, phase, ring, plan, w0);
        TC_TRACE(plan, it, 3);
        ld_row<CH>(lane_base + Cfg::col_x0 + col0, v);
#pragma unroll
        for (int i = 0; i < CH; ++i) v[i] = fmaxf(v[i], 0.f);
        st_row<CH>(lane_base + Cfg::col_x0 + col0, v);
        // ---- dense2([u', v']) accumulated over the two K halves (the region is reloaded in between)
        if (InputPf<C>::enabled) {
            store_input_row<C, true, 2, HM>(pfu, s.region, row, half);
            fetch_input_row<C>(vin, npix, (size_t)img, pix, valid, half, pfu);
        } else {
            load_input_row<C, TPR, PX ? HM : 3>(uin, npix, (size_t)img, pix, valid, s.region, row, half, 0);
        }
        TC_TRACE(plan, it, 4);
        sync_for_mma();
        if (w0 && elect_one()) { issue_linear_t<G, MG_PD2A>(ring, plan, region_addr, ones_addr, tm + Cfg::col_acc, true); commit(s.done); }
        TC_TRACE(plan, it, 5);
        wait_done_ring<G>(s.done, phase, ring, plan, w0);
        TC_TRACE(plan, it, 6);
        if (InputPf<C>::enabled) store_input_row<C, true, 2, HM>(pfu, s.region, row, half);
        else load_input_row<C, TPR, PX ? HM : 3>(vin, npix, (size_t)img, pix, valid, s.region, row, half, 0);
        TC_TRACE(plan, it, 7);
        sync_for_mma();
        if (w0 && elect_one()) { issue_linear_t<G, MG_PD2B>(ring, plan, region_addr, ones_addr, tm + Cfg::col_acc, false); commit(s.done); }
        TC_TRACE(plan, it, 8);
        wait_done_ring<G>(s.done, phase, ring, plan, w0);
        }
        TC_TRACE(plan, it, 9);
        // x1 = acc + x0; q = x1 + x0 -> global; LayerNorm(x1) (affine folded into conv1) -> region
        {
            float rstd, shift;
            ld_row<CH>(lane_base + Cfg::col_acc + col0, v);
            float sum = 0.f, sq = 0.f;
            constexpr int SC = CH > 64 ? 64 : CH;
            unsigned long long s2 = pk2(0.f, 0.f), q2 = pk2(0.f, 0.f);
#pragma unroll
            for (int c = 0; c < CH; c += SC) {
                float x0[SC];
                ld_row<SC>(lane_base + Cfg::col_x0 + col0 + c, x0);
#pragma unroll
                for (int i = 0; i < SC; i += 2) {
                    const unsigned long long xz = pk2(x0[i], x0[i + 1]);
                    unsigned long long x1 = add2(pk2(v[c + i], v[c + i + 1]), xz);
                    if constexpr (G::ebias) x1 = add2(x1, pk2(eb[C + c + i], eb[C + c + i + 1]));
                    s2 = add2(s2, x1);
                    q2 = fma2(x1, x1, q2);
                    upk2(x1, v[c + i], v[c + i + 1]);
                    upk2(add2(x1, xz), x0[i], x0[i + 1]);
                }
                if constexpr (SC % 32 == 0 && PX == 0) oct_store<SC / 4>(qout, row_off + c, C, x0, valid); else pair_store<SC / 4>(qout, row_off + c, x0, valid);
            }
            { float a, b; upk2(s2, a, b); sum = a + b; upk2(q2, a, b); sq = a + b; }
            row_stats<1, TPR>(sum, sq, s.xch + (xb++ & 1) * TPR * TM, row, half, C, rstd, shift);
            norm_row<CH>(v, rstd, shift);
            row_to_a16<CH, LOC>(v, s.region, row, col0);
        }
        TC_TRACE(plan, it, 10);
        sync_for_mma();
        // ---- conv1 -> LeakyReLU(0.2)
        if (w0 && elect_one()) { issue_linear_t<G, MG_RC1>(ring, plan, region_addr, ones_addr, tm + Cfg::col_acc, true); commit(s.done); }
        TC_TRACE(plan, it, 11);
        wait_done_ring<G>(s.done, phase, ring, plan, w0);
        TC_TRACE(plan, it, 12);
        ld_row<CH>(lane_base + Cfg::col_acc + col0, v);
#pragma unroll
        for (int i = 0; i < CH; i += 2) {          // LeakyReLU(0.2) = max(v, 0.2 v)
            if constexpr (G::ebias) { v[i] += eb[2 * C + i]; v[i + 1] += eb[2 * C + i + 1]; }
            float l0, l1;
            upk2(mul2(pk2(v[i], v[i + 1]), pk2(0.2f, 0.2f)), l0, l1);
            v[i] = fmaxf(v[i], l0); v[i + 1] = fmaxf(v[i + 1], l1);
        }
        row_to_a16<CH, LOC>(v, s.region, row, col0);
        TC_TRACE(plan, it, 13);
        sync_for_mma();
        // ---- conv2 = r -> global, and staged (exact fp32) in the region for the per-unit channel sums (squeeze)
        if (w0 && elect_one()) { issue_linear_t<G, MG_RC2>(ring, plan, region_addr, ones_addr, tm + Cfg::col_acc, true); commit(s.done); }
        TC_TRACE(plan, it, 14);
        wait_done_ring<G>(s.done, phase, ring, plan, w0);
        TC_TRACE(plan, it, 15);
        ld_row<CH>(lane_base + Cfg::col_acc + col0, v);
        if constexpr (G::ebias) {
#pragma unroll
            for (int i = 0; i < CH; ++i) v[i] += eb[3 * C + i];
        }
#pragma unroll
        for (int j = 0; j < CH / 4; ++j) {
            const float4 o = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            *reinterpret_cast<float4*>(s.region + ((size_t)(col0 / 4 + j) * TM + row) * 4) = o;
        }
        static_assert(PX != 0 || C < 128 || CH % 64 == 0, "the fp16 r store (r16, decided by the host) assumes two threads per row");
        if constexpr (CH % 64 == 0 && PX == 0) {
            if (r16) {
                // r leaves as fp16 (channels-last halves): it only enters r * s + q, which its consumer (pool_kernel / the head
                // kernel) rounds to fp16 next -- as at stages 1-2; half the bytes and half the chunk transposes of the store
                float hv[CH / 2];
#pragma unroll
                for (int i = 0; i < CH / 2; ++i) {
                    uint32_t h;
                    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h) : "f"(v[2 * i + 1]), "f"(v[2 * i]));
                    hv[i] = __uint_as_float(h);
                }
                oct_store<CH / 8>(rout, row_off / 2, C / 2, hv, valid);
            } else {
                oct_store<CH / 4>(rout, row_off, C, v, valid);
            }
        } else if constexpr (CH % 32 == 0 && PX == 0) {
            oct_store<CH / 4>(rout, row_off, C, v, valid);
        } else {
            pair_store<CH / 4>(rout, row_off, v, valid);
        }
        __syncthreads();
        unit_channel_sums<C, NTK>(s.region, t, geo.total_units, partial);
        if constexpr (Cfg::two) fence_async_smem();                   // generic reads of the staging tile before the async write below
        __syncthreads();
        if constexpr (Cfg::two) {
            if (t + (int)gridDim.x < ntiles && w0 && elect_one()) {
                mbar_expect_tx(ld_u, kTileBytes);
                bulk_load(r2_addr, uin + (size_t)(t + gridDim.x) * tile_floats, kTileBytes, ld_u);
            }
        }
    }
    tc_finish(tm, Cfg::ncols);
}


// ------------------------------------------------------------------------------------------ merge kernel with bulk-copied tiles (C <= 64)
// The first two stages hold 64x / 16x the pixel rows of the last one and their merge kernels are the largest of the detector.
// A first 3-phase version with per-thread loads / stores measured 4.2 ms per 64 images at C = 32 of which 1.5 ms was compute:
// its 16-byte global accesses neither overlapped the phases nor coalesced (32 sectors per warp instruction).  Here every
// tile-sized transfer is ONE bulk copy issued by the elected lane: u' and v' arrive from the branch kernels already
// tf32-rounded in the swizzled panel layout, land in shared memory as valid SWIZZLE_128B operands (no thread touches
// them) a tile ahead of their use, and q / r leave through swizzled staging tiles with bulk stores that drain under the
// following phases.  At C = 32 (CIN = 3) x0 = ReLU(conv.0(x)) runs on the CUDA cores while the dense2 MMAs execute; at
// C = 64 conv.0 is a third MMA of phase 1 on a register-prefetched x tile.  Consumers of r / q (pool_kernel) un-permute.
// Regions: U | V (operands of dense2) | W (conv1 / conv2 input, then r staging) | Q (q staging) | X (conv.0 operand).
template <int CIN, int C, int PX = 0> struct MergeBulkCfg {
    static constexpr int CH = C / 2;
    static constexpr bool cc0 = CIN < 8;
    static constexpr uint32_t tile_bytes = (uint32_t)TM * C * 4;      // W / Q staging tiles (fp32)
    static constexpr uint32_t uv_bytes = (uint32_t)TM * C * (PX ? 4u : 2u);   // u' / v' tiles (fp16, chunk-major; hi then lo chunks: PX)
    // r leaves as an fp16 tile staged in the first half of Q (q's own store was issued two phases earlier and has been waited
    // for); split precision stores the fp32 staging tile W instead.  No region of its own: 3 CTAs per SM fit at C = 32.
    static constexpr uint32_t r16_bytes = 0u;
    static constexpr uint32_t xbytes = cc0 ? 0u : (uint32_t)TM * tc_kin(CIN) * 4;
    static constexpr uint32_t region = 2 * uv_bytes + r16_bytes + 2 * tile_bytes + xbytes;   // U, V (fp16) | W, Q (fp32) | X
    static constexpr uint32_t xch = 2u * TM * 8u;                    // one LayerNorm exchange per tile: a single buffer
    static constexpr int col_acc = 0, col_x0 = C;
    static constexpr int ncols = tc_cols(cc0 ? C : 2 * C);
    static constexpr int min_ctas = C <= 32 ? (PX ? 2 : kMerge32Ctas) : 1;
};

template <int CIN, int C, int PX = 0>
__global__ void __launch_bounds__(NT2, MergeBulkCfg<CIN, C, PX>::min_ctas)
tc_merge_bulk_kernel(const float* __restrict__ xin, DownW w, TcPlan plan, UnitGeom geo, const float* __restrict__ uin,
                     const float* __restrict__ vin, float* __restrict__ rout, float* __restrict__ qout, float* __restrict__ partial) {
    extern __shared__ __align__(1024) unsigned char smem[];
    using Cfg = MergeBulkCfg<CIN, C, PX>;
    constexpr int CH = Cfg::CH;
    using G = MergeG<CIN, C, PX>;
    constexpr int HM = PX ? 2 : 1, LOC = PX ? C / 8 : 0;
    constexpr bool XH = PX == 0 && CIN >= 8;                  // fp16 level input (pool_kernel, single-rounded path)
    constexpr int XM = XH ? 3 : HM;
    const TcShared s = carve(smem, Cfg::region, plan, 1, Cfg::xch);
    float* const regU = s.region;                                    // fp16 tile: TM * C / 2 floats
    float* const regV = regU + Cfg::uv_bytes / 4;
    float* const regW = regV + Cfg::uv_bytes / 4;
    float* const regQ = regW + (size_t)TM * C;
    float* const regR = regQ;                                        // r as an fp16 tile (chunk-major) for its bulk store (not PX): over Q
    float* const regX = regQ + (size_t)TM * C;
    uint64_t* const ld_bar = s.aux;
    const int tid = threadIdx.x, row = tid & (TM - 1), half = tid >> 7;
    const int ntiles = geo.total_units / 2;                 // host guarantees an even unit count: whole tiles only
    const uint32_t my_tiles = blockIdx.x < (unsigned)ntiles ? (ntiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;
    if constexpr (Cfg::cc0) conv0_stage_weights<CIN, C>(w, s.vec);
    Ring ring;
    const bool w0 = warp0_uniform();
    tc_prologue<G::nslot>(s, Cfg::ncols, ring, plan, my_tiles, w0);
    const uint32_t tm = *s.tmem_slot;
    const uint32_t lane_base = tm + ((uint32_t)(row & ~31) << 16);
    const uint32_t u_addr = smem_u32(regU), v_addr = smem_u32(regV), w_addr = smem_u32(regW), q_addr = smem_u32(regQ);
    const uint32_t x_addr = smem_u32(regX), ones_addr = smem_u32(s.ones);
    const int col0 = half * CH;
    const size_t npix = (size_t)geo.h * geo.w;
    const size_t tile_floats = (size_t)TM * C;              // tile t of the batch chunk starts at float t * tile_floats in u', v', r, q
    uint32_t phase = 0, ld_phase = 0;
    auto coords = [&](int tt, int& im, int& px) {
        const int un = 2 * tt + (row >> 6);
        im = fast_div(un, geo.upi, geo.inv_upi);
        px = (un - im * geo.upi) * 64 + (row & 63);
    };
    auto load_tile = [&](int tt) {                          // elected lane: next tile's u' and v' (fp16 tiles) -> U, V
        mbar_expect_tx(ld_bar, 2 * Cfg::uv_bytes);
        bulk_load(u_addr, uin + (size_t)tt * (Cfg::uv_bytes / 4), Cfg::uv_bytes, ld_bar);
        bulk_load(v_addr, vin + (size_t)tt * (Cfg::uv_bytes / 4), Cfg::uv_bytes, ld_bar);
    };
    InputPf<CIN> pfx;
    if ((int)blockIdx.x < ntiles) {
        int im, px;
        coords(blockIdx.x, im, px);
        fetch_input_row<CIN, false, 2, XH>(xin, npix, (size_t)im, px, true, half, pfx);
        if (w0 && elect_one()) load_tile(blockIdx.x);
    }
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int nt = t + (int)gridDim.x;
        float v[CH], x0[CH];
        // ---- phase 1: acc = dense2([u', v']) (+ conv.0(x) at CIN >= 8) on the tensor core | x0 on the CUDA cores at CIN < 8
        if constexpr (!Cfg::cc0) {
            store_input_row<CIN, false, 2, XM>(pfx, regX, row, half);     // X was released by the previous tile's phase 1
            sync_for_mma();
        }
        if (w0 && elect_one()) {
            if constexpr (!Cfg::cc0) issue_linear_t<G, MG_CONV0>(ring, plan, x_addr, ones_addr, tm + Cfg::col_x0, true);
            mbar_wait(ld_bar, ld_phase & 1);
            fence_after_sync();
            issue_linear_t<G, MG_PD2A>(ring, plan, u_addr, ones_addr, tm + Cfg::col_acc, true);      // kind::f16 on the fp16 tiles
            issue_linear_t<G, MG_PD2B>(ring, plan, v_addr, ones_addr, tm + Cfg::col_acc, false);
            commit(s.done);
            bulk_wait_read();                               // the previous tile's q / r stores have left W and Q
        }
        ++ld_phase;
        if constexpr (Cfg::cc0) conv0_row<CIN, C, CH>(pfx.v[0], s.vec, col0, x0);
        if (nt < ntiles) {
            int im, px;
            coords(nt, im, px);
            fetch_input_row<CIN, false, 2, XH>(xin, npix, (size_t)im, px, true, half, pfx);
        }
        wait_done_ring<G>(s.done, phase, ring, plan, w0);
        // x1 = acc + x0; q = x1 + x0 -> Q (staging); LayerNorm(x1) (affine folded into conv1) -> W
        {
            float rstd, shift;
            ld_row<CH>(lane_base + Cfg::col_acc + col0, v);
            if constexpr (!Cfg::cc0) {
                ld_row<CH>(lane_base + Cfg::col_x0 + col0, x0);
#pragma unroll
                for (int i = 0; i < CH; ++i) x0[i] = fmaxf(x0[i], 0.f);
            }
            unsigned long long s2 = pk2(0.f, 0.f), q2 = pk2(0.f, 0.f);
#pragma unroll
            for (int i = 0; i < CH; i += 2) {
                const unsigned long long xz = pk2(x0[i], x0[i + 1]);
                const unsigned long long x1 = add2(pk2(v[i], v[i + 1]), xz);
                s2 = add2(s2, x1);
                q2 = fma2(x1, x1, q2);
                upk2(x1, v[i], v[i + 1]);
                upk2(add2(x1, xz), x0[i], x0[i + 1]);
            }
            if constexpr (PX == 0) {
                // q crosses HBM as 24 bits per value -- the top 16 bits of the fp32 pattern (rounded to 16 mantissa bits, RN on
                // the bit pattern) in a [C / 8][128][8 x u16] plane and the next 8 bits in a [C / 16][128][16 x u8] plane: its only
                // consumer (pool_kernel) rounds max(r s + q) to fp16, 2^-17 on q is noise there; 96 instead of 128 bytes per pixel
                // at C = 32 on the two HBM-bound kernels of the stage.  (fp16 q was measured at +15 % score-map error.)
                uint32_t bq[CH];
#pragma unroll
                for (int i = 0; i < CH; ++i) bq[i] = __float_as_uint(x0[i]) + 0x80u;
                unsigned char* const qb = reinterpret_cast<unsigned char*>(regQ);
#pragma unroll
                for (int j = 0; j < CH / 8; ++j) {          // top halves: bytes 2, 3 of each value
                    uint4 o;
                    o.x = __byte_perm(bq[8 * j], bq[8 * j + 1], 0x7632); o.y = __byte_perm(bq[8 * j + 2], bq[8 * j + 3], 0x7632);
                    o.z = __byte_perm(bq[8 * j + 4], bq[8 * j + 5], 0x7632); o.w = __byte_perm(bq[8 * j + 6], bq[8 * j + 7], 0x7632);
                    *reinterpret_cast<uint4*>(qb + ((size_t)(col0 / 8 + j) * TM + row) * 16) = o;
                }
#pragma unroll
                for (int j = 0; j < CH / 16; ++j) {         // middle bytes: byte 1 of each value
                    uint32_t w4[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const uint32_t lo = __byte_perm(bq[16 * j + 4 * e], bq[16 * j + 4 * e + 1], 0x0051);
                        const uint32_t hi = __byte_perm(bq[16 * j + 4 * e + 2], bq[16 * j + 4 * e + 3], 0x0051);
                        w4[e] = __byte_perm(lo, hi, 0x5410);
                    }
                    *reinterpret_cast<uint4*>(qb + (size_t)TM * C * 2 + ((size_t)(col0 / 16 + j) * TM + row) * 16) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
                }
            } else {
                row_to_sw<CH, false>(x0, regQ, row, col0);
            }
            float sum, sq;
            { float a, b; upk2(s2, a, b); sum = a + b; upk2(q2, a, b); sq = a + b; }
            row_stats(sum, sq, s.xch, row, half, C, rstd, shift);
            norm_row<CH>(v, rstd, shift);
            if constexpr (G::h16(MG_RC1)) row_to_a16<CH, LOC>(v, regW, row, col0); else row_to_sw<CH, true>(v, regW, row, col0);
        }
        sync_for_mma();
        // ---- phase 2: conv1 -> LeakyReLU(0.2); q leaves, the next tile's u' / v' arrive (phase 1 released U and V)
        if (w0 && elect_one()) {
            issue_linear_t<G, MG_RC1, !G::h16(MG_RC1)>(ring, plan, w_addr, ones_addr, tm + Cfg::col_acc, true);
            commit(s.done);
            if constexpr (PX == 0) bulk_store(qout + (size_t)t * (tile_floats * 3 / 4), q_addr, Cfg::tile_bytes / 4 * 3);   // 24-bit planes
            else bulk_store(qout + (size_t)t * tile_floats, q_addr, Cfg::tile_bytes);
            bulk_commit();
            if (nt < ntiles) load_tile(nt);
        }
        wait_done_ring<G>(s.done, phase, ring, plan, w0);
        ld_row<CH>(lane_base + Cfg::col_acc + col0, v);
#pragma unroll
        for (int i = 0; i < CH; i += 2) {          // LeakyReLU(0.2) = max(v, 0.2 v)
            float l0, l1;
            upk2(mul2(pk2(v[i], v[i + 1]), pk2(0.2f, 0.2f)), l0, l1);
            v[i] = fmaxf(v[i], l0); v[i + 1] = fmaxf(v[i + 1], l1);
        }
        if constexpr (G::h16(MG_RC1)) row_to_a16<CH, LOC>(v, regW, row, col0); else row_to_sw<CH, true>(v, regW, row, col0);
        sync_for_mma();
        // ---- phase 3: conv2 = r (exact fp32) -> W (staging) -> global, and the per-unit channel sums (squeeze)
        if (w0 && elect_one()) {
            issue_linear_t<G, MG_RC2, !G::h16(MG_RC2)>(ring, plan, w_addr, ones_addr, tm + Cfg::col_acc, true);
            commit(s.done);
            if constexpr (!PX) bulk_wait_read();            // q's store (issued in phase 2) has read Q: its first half becomes the r tile
        }
        wait_done_ring<G>(s.done, phase, ring, plan, w0);
        ld_row<CH>(lane_base + Cfg::col_acc + col0, v);
        row_to_sw<CH, false>(v, regW, row, col0);              // exact fp32: the squeeze sums below
        if constexpr (!PX) {
            // r crosses HBM as an fp16 tile [C / 8 chunks][128 pixels][8 halves] (pool_kernel reads it back): r only enters
            // r * s + q with s in (0, 1) next to the fp32 q, and the sum is rounded to an 11-bit significand by its consumer --
            // measured effect on the score map: mean relative error 1.017e-4 -> 1.022e-4 (emulation, DESIGN.md)
            __half* rt = reinterpret_cast<__half*>(regR) + (size_t)row * 8;
#pragma unroll
            for (int j = 0; j < CH / 8; ++j) {
                uint32_t h[4];
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h[e]) : "f"(v[8 * j + 2 * e + 1]), "f"(v[8 * j + 2 * e]));
                *reinterpret_cast<uint4*>(rt + (size_t)(col0 / 8 + j) * (TM * 8)) = make_uint4(h[0], h[1], h[2], h[3]);
            }
        }
        sync_for_mma();
        if (w0 && elect_one()) {
            // split precision: r leaves as the exact fp32 staging tile (swizzled panel layout, like q)
            if constexpr (PX) bulk_store(rout + (size_t)t * tile_floats, w_addr, Cfg::tile_bytes);
            else bulk_store(rout + (size_t)t * (tile_floats / 2), smem_u32(regR), Cfg::uv_bytes);
            bulk_commit();
        }
        {   // channel sums of each unit from the swizzled staging tile (see unit_channel_sums; same fixed order)
            constexpr int CQ = C / 4, TPP = NT2 / (2 * CQ), RPT = 64 / TPP;
            const int pair = tid / TPP, sub = tid % TPP;
            const int uu = pair / CQ, ch = pair % CQ;
            float4 acc = *reinterpret_cast<const float4*>(regW + sw_off(uu * 64 + sub, ch));
#pragma unroll
            for (int i = 1; i < RPT; ++i) {
                const float4 x = *reinterpret_cast<const float4*>(regW + sw_off(uu * 64 + sub + i * TPP, ch));
                acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
            }
#pragma unroll
            for (int o = TPP / 2; o >= 1; o >>= 1) {
                acc.x += __shfl_xor_sync(0xffffffffu, acc.x, o);
                acc.y += __shfl_xor_sync(0xffffffffu, acc.y, o);
                acc.z += __shfl_xor_sync(0xffffffffu, acc.z, o);
                acc.w += __shfl_xor_sync(0xffffffffu, acc.w, o);
            }
            if (sub == 0) *reinterpret_cast<float4*>(partial + (size_t)(2 * t + uu) * C + ch * 4) = acc;
        }
        // W is next written by the following tile's phase-1 epilogue, i.e. after its wait_done barrier: every thread has
        // finished the sums by then, and the elected lane has waited for the r store to have read W (bulk_wait_read)
    }
    if (w0 && elect_one()) bulk_wait_all();
    tc_finish(tm, Cfg::ncols);
}

// ------------------------------------------------------------------------------------------ head kernel (last stage)
// t = r * s + q -> conv2 (C -> C) -> ReLU -> dense (C -> 65, BatchNorm folded into weights and bias) = logits ->
// softmax -> drop the dustbin -> depth-to-space.  The half-0 thread of a row finishes its 8x8 cell.
template <int C, int PX = 0>
__global__ void __launch_bounds__(NT2, 1) tc_head_kernel(const float* __restrict__ r, const float* __restrict__ q,
                                                         const float* __restrict__ scale, TcPlan plan, UnitGeom geo, int cell,
                                                         float* __restrict__ logits, float* __restrict__ prob, int r16) {
    extern __shared__ __align__(1024) unsigned char smem[];
    using G = HeadG<C, PX>;
    constexpr int LOC = PX ? C / 8 : 0;
    constexpr uint32_t region_bytes = (uint32_t)TM * C * 4;
    constexpr int ncols = tc_cols(C + 96);
    constexpr int CH = C / 2;
    const TcShared s = carve(smem, region_bytes, plan);
    const int tid = threadIdx.x, row = tid & (TM - 1), half = tid >> 7;
    const int ntiles = (geo.total_units + 1) / 2;
    const uint32_t my_tiles = blockIdx.x < (unsigned)ntiles ? (ntiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;
    Ring ring;
    const bool w0 = warp0_uniform();
    tc_prologue<G::nslot>(s, ncols, ring, plan, my_tiles, w0);
    const uint32_t tm = *s.tmem_slot;
    const uint32_t lane_base = tm + ((uint32_t)(row & ~31) << 16);
    const uint32_t region_addr = smem_u32(s.region), ones_addr = smem_u32(s.ones);
    const int ug = row >> 6, tok = row & 63;
    const int col0 = half * CH;
    const size_t npix = (size_t)geo.h * geo.w;
    const int nlog = cell * cell + 1;
    uint32_t phase = 0;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int unit = 2 * t + ug;
        const bool valid = unit < geo.total_units;
        const int img = valid ? fast_div(unit, geo.upi, geo.inv_upi) : 0, u = valid ? unit - img * geo.upi : 0;
        const int pix = u * 64 + tok;
        const size_t row_off = ((size_t)img * npix + pix) * C + col0;
#pragma unroll 1
        for (int j0 = 0; j0 < CH / 4; j0 += 8) {            // full-sector pair loads of r and q, 8 chunks at a time
            float4 rv[8], qv[8];
            if constexpr (PX == 0) {              // full-line loads (see oct_load)
                if (r16) {                         // r as fp16 channels-last (tc_merge_kernel): 4 chunks of 8 halves
                    const uint4* rh = reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(r) + row_off) + j0 / 2;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint4 h = valid ? __ldg(rh + k) : make_uint4(0u, 0u, 0u, 0u);
                        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&h.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&h.y));
                        const float2 c2 = __half22float2(*reinterpret_cast<const __half2*>(&h.z)), d = __half22float2(*reinterpret_cast<const __half2*>(&h.w));
                        rv[2 * k] = make_float4(a.x, a.y, b.x, b.y);
                        rv[2 * k + 1] = make_float4(c2.x, c2.y, d.x, d.y);
                    }
                } else {
                    oct_load<8>(r, row_off + (size_t)j0 * 4, C, valid, rv);
                }
                oct_load<8>(q, row_off + (size_t)j0 * 4, C, valid, qv);
            } else {
                pair_load<8>(reinterpret_cast<const float4*>(r + row_off) + j0, valid, rv);
                pair_load<8>(reinterpret_cast<const float4*>(q + row_off) + j0, valid, qv);
#pragma unroll
                for (int j = 0; j < 8; j += 2) { pair_unswap(rv[j], rv[j + 1]); pair_unswap(qv[j], qv[j + 1]); }
            }
#pragma unroll
            for (int j = 0; j < 8; j += 2) {                  // two 4-channel chunks -> one fp16 chunk of 8 channels
                float e[8];
#pragma unroll
                for (int u2 = 0; u2 < 2; ++u2) {
                    const float4 sv = __ldg(reinterpret_cast<const float4*>(scale + (size_t)img * C + col0) + j0 + j + u2);
                    e[4 * u2] = rv[j + u2].x * sv.x + qv[j + u2].x; e[4 * u2 + 1] = rv[j + u2].y * sv.y + qv[j + u2].y;
                    e[4 * u2 + 2] = rv[j + u2].z * sv.z + qv[j + u2].z; e[4 * u2 + 3] = rv[j + u2].w * sv.w + qv[j + u2].w;
                }
                uint32_t h[4], l[4];
#pragma unroll
                for (int w2 = 0; w2 < 4; ++w2) {
                    if constexpr (PX) split_h2(e[2 * w2], e[2 * w2 + 1], h[w2], l[w2]);
                    else asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h[w2]) : "f"(e[2 * w2 + 1]), "f"(e[2 * w2]));
                }
                *reinterpret_cast<uint4*>(s.region + ((size_t)((col0 / 4 + j0 + j) / 2) * TM + row) * 4) = make_uint4(h[0], h[1], h[2], h[3]);
                if constexpr (PX)
                    *reinterpret_cast<uint4*>(s.region + ((size_t)(LOC + (col0 / 4 + j0 + j) / 2) * TM + row) * 4) = make_uint4(l[0], l[1], l[2], l[3]);
            }
        }
        sync_for_mma();
        if (w0 && elect_one()) { issue_linear_t<G, HG_C2>(ring, plan, region_addr, ones_addr, tm, true); commit(s.done); }
        wait_done_ring<G>(s.done, phase, ring, plan, w0);
        {
            float v[CH];
            ld_row<CH>(lane_base + col0, v);
#pragma unroll
            for (int i = 0; i < CH; ++i) v[i] = fmaxf(v[i], 0.f);
            row_to_a16<CH, LOC>(v, s.region, row, col0);
        }
        sync_for_mma();
        if (w0 && elect_one()) { issue_linear_t<G, HG_DENSE>(ring, plan, region_addr, ones_addr, tm + C, true); commit(s.done); }
        wait_done_ring<G>(s.done, phase, ring, plan, w0);
        // logits = columns C .. C+64 of the row.  tcgen05.ld is warp-collective and `half` is warp-uniform, so the
        // branch below is convergent per warp.
        if (half == 0) {
            float z[96];
            ld_row<96>(lane_base + C, z);                           // columns >= 80 hold stale data (never read below)
            float mx = kNegInf;
#pragma unroll
            for (int n = 0; n < 65; ++n) mx = fmaxf(mx, z[n]);
            float den = 0.f;
#pragma unroll
            for (int n = 0; n < 65; ++n) den += expf(z[n] - mx);
            if (valid) {
                const int cy = pix / geo.w, cx = pix - cy * geo.w;
                const int Wp = geo.w * cell, Hp = geo.h * cell;
                if (logits) {
#pragma unroll
                    for (int n = 0; n < 65; ++n) logits[((size_t)img * nlog + n) * npix + pix] = z[n];
                }
                const float inv = 1.0f / den;
                if (cell == 8) {                 // 8 x 8 cell: two 16-byte stores per output row (a quarter of the store instructions)
#pragma unroll
                    for (int n = 0; n < 64; n += 4) {
                        const int yy = cy * 8 + (n >> 3), xx = cx * 8 + (n & 7);
                        *reinterpret_cast<float4*>(prob + ((size_t)img * Hp + yy) * Wp + xx) =
                            make_float4(expf(z[n] - mx) * inv, expf(z[n + 1] - mx) * inv, expf(z[n + 2] - mx) * inv, expf(z[n + 3] - mx) * inv);
                    }
                } else {
#pragma unroll
                for (int n = 0; n < 64; ++n) {
                    const int yy = cy * cell + (n >> 3), xx = cx * cell + (n & 7);
                    prob[((size_t)img * Hp + yy) * Wp + xx] = expf(z[n] - mx) * inv;
                }
                }
            }
        }
    }
    tc_finish(tm, ncols);
}

#ifdef BALF_TC_MAIN
// ------------------------------------------------------------------------------------------ weight packing (tc blob)
// wT [K][ld] (the fp32 path's transposed weight) -> blocks of [rows x kb] chunk-major, rows n0..n0+rows.
// Optional folds: gamma[k] (LayerNorm weight of the layer's input), alpha[n] (per-output scale).
__global__ void tc_pack_kernel(const float* __restrict__ wT, int ld, int n0, int rows, int k_real, int k_pad, int kb,
                               const float* __restrict__ gamma, const float* __restrict__ alpha, float* __restrict__ dst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * k_pad) return;
    const int k = i / rows, n = i - k * rows;
    const int b = k / kb, kk = k - b * kb;
    float v = 0.f;
    if (k < k_real) {
        v = wT[(size_t)k * ld + n0 + n];
        if (gamma) v *= gamma[k];
        if (alpha) v *= alpha[n0 + n];
    }
    dst[(size_t)b * rows * kb + (size_t)(kk >> 2) * rows * 4 + n * 4 + (kk & 3)] = to_tf32_exact(v);
}
// the same for fp16 GEMMs (TcGemm::h16): blocks of [rows x kb] halves, chunk-major with 8 halves per 16-byte chunk
__global__ void tc_pack_h16_kernel(const float* __restrict__ wT, int ld, int n0, int rows, int k_real, int k_pad, int kb,
                                   const float* __restrict__ gamma, const float* __restrict__ alpha, __half* __restrict__ dst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * k_pad) return;
    const int k = i / rows, n = i - k * rows;
    const int b = k / kb, kk = k - b * kb;
    float v = 0.f;
    if (k < k_real) {
        v = wT[(size_t)k * ld + n0 + n];
        if (gamma) v *= gamma[k];
        if (alpha) v *= alpha[n0 + n];
    }
    dst[(size_t)b * rows * kb + (size_t)(kk >> 3) * rows * 8 + n * 8 + (kk & 7)] = __float2half_rn(v);
}
// split precision (TcGemm::h16 == 2): every block holds its kb columns as fp16 hi chunks followed by the fp16 lo chunks
__global__ void tc_pack_x3_kernel(const float* __restrict__ wT, int ld, int n0, int rows, int k_real, int k_pad, int kb,
                                  const float* __restrict__ gamma, const float* __restrict__ alpha, __half* __restrict__ dst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * k_pad) return;
    const int k = i / rows, n = i - k * rows;
    const int b = k / kb, kk = k - b * kb;
    float v = 0.f;
    if (k < k_real) {
        v = wT[(size_t)k * ld + n0 + n];
        if (gamma) v *= gamma[k];
        if (alpha) v *= alpha[n0 + n];
    }
    const __half hi = __float2half_rn(v);
    const size_t at = (size_t)b * rows * kb * 2 + (size_t)(kk >> 3) * rows * 8 + n * 8 + (kk & 7);
    dst[at] = hi;
    dst[at + (size_t)rows * kb] = __float2half_rn(v - __half2float(hi));
}
// bias columns of the last block: b' = (bias[n] + sum_k W[n][k] beta[k]) * alpha[n] + add[n], split into tf32 hi + lo
__global__ void tc_pack_bias_kernel(const float* __restrict__ wT, int ld, int n0, int rows, int k_real,
                                    const float* __restrict__ bias, const float* __restrict__ beta,
                                    const float* __restrict__ alpha, const float* __restrict__ add, float* __restrict__ dst) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= rows) return;
    float acc = bias ? bias[n0 + n] : 0.f;
    if (beta) {
        float comp = 0.f;                                           // compensated: the fold must not cost precision
        for (int k = 0; k < k_real; ++k) {
            const float y = wT[(size_t)k * ld + n0 + n] * beta[k] - comp, t = acc + y;
            comp = (t - acc) - y;
            acc = t;
        }
    }
    if (alpha) acc *= alpha[n0 + n];
    if (add) acc += add[n0 + n];
    const float hi = to_tf32_exact(acc), lo = to_tf32_exact(acc - hi);
    dst[n * 4 + 0] = hi;
    dst[n * 4 + 1] = lo;
    dst[n * 4 + 2] = 0.f;
    dst[n * 4 + 3] = 0.f;
}

#endif  // BALF_TC_MAIN

struct TcPlans {
    TcPlan branch[4][2], merge[4], head;
    size_t floats;
};

static void tc_add(TcPlan& p, int gi, size_t& off, int rows, int K, bool bias, int cap = 32768, int h16 = 0) {
    const int kb = tc_kb(rows, K, cap, (int)tc_eb(h16));
    TcGemm& g = p.g[gi];
    g.goff = (uint32_t)off;
    g.nblk = (uint16_t)(K / kb);
    g.rows = (uint16_t)rows;
    g.kb = (uint16_t)kb;
    g.bias = bias ? 1 : 0;
    g.h16 = (uint16_t)h16;
    off += gemm_bytes(g) / 4;
    p.bytes += gemm_bytes(g);
    const uint32_t big = (gemm_block_bytes(g, g.nblk - 1) + 127u) / 128u * 128u;
    if (big > p.slot_bytes) p.slot_bytes = big;
}

template <typename G>
static bool plan_matches(const TcPlan& p) {
    if (p.ngemm != G::count || (p.resident != 0) != G::resident || (int)p.nslot != G::nslot) return false;
    uint32_t off = 0;
    bool ok = true;
    for (int gi = 0; gi < G::count; ++gi) {
        const TcGemm& g = p.g[gi];
        ok = ok && g.rows == G::rows(gi) && g.kb == tc_kb(G::rows(gi), G::K(gi), G::cap, (int)tc_eb(g_mode<G>(gi))) && g.nblk * g.kb == G::K(gi) &&
             (g.bias != 0) == G::bias(gi) && (int)g.h16 == g_mode<G>(gi) && gemm_bytes(g) == g_bytes<G>(gi) &&
             (g.goff - p.g[0].goff) * 4u == off;
        off += gemm_bytes(g);
    }
    return ok;
}

// px = 1: the split-precision plans (they follow the px = 0 plans in the blob); `off` runs over both
static void tc_build_plans_px(const balf_detector_arch& a, const float* base, TcPlans* out, int px, size_t& off) {
    TcPlans P;
    const int hm = px ? 2 : 1;
    for (int l = 0; l < 4; ++l) {
        const int cin = tc_kin(a.dims[l]), c = a.dims[l + 1];
        for (int b = 0; b < 2; ++b) {
            TcPlan& p = P.branch[l][b];
            p = TcPlan{};
            p.base = base; p.ngemm = BG_COUNT;
            p.resident = px ? c <= 64 : c <= 128;                      // mirrors BranchG::resident
            p.nslot = px ? (c == 256 ? 2 : 3) : (c == 256 ? 3 : 2);    // mirrors BranchG::nslot (checked by plan_matches)
            tc_add(p, BG_CONV0, off, c, cin, true, 32768, a.dims[l] >= 8 ? hm : 0);
            tc_add(p, BG_PD1, off, c, c, true, 32768, hm);             // mirrors BranchG::h16
            tc_add(p, BG_D1A, off, c, c, true, 32768, hm);
            tc_add(p, BG_D1B, off, c, c, true, 32768, hm);
            tc_add(p, BG_WM, off, 64, 64, false, 32768, hm);
            tc_add(p, BG_D2, off, c, c, true, 32768, hm);
        }
        TcPlan& m = P.merge[l];
        m = TcPlan{};
        m.base = base; m.ngemm = MG_COUNT;
        m.resident = px ? c <= 32 : c <= 128;                          // mirrors MergeG::resident
        m.nslot = px ? (c == 64 ? 3 : 2) : (c == 256 ? 2 : 3);         // mirrors MergeG::nslot / MergeG::cap
        const int mcap = 32768;
        const bool ebias = c == 128 && !px;                            // mirrors MergeG::ebias: biases added by the epilogues
        tc_add(m, MG_CONV0, off, c, cin, !ebias, mcap, a.dims[l] >= 8 ? hm : 0);
        tc_add(m, MG_PD2A, off, c, c, false, mcap, hm);               // mirrors MergeG::h16
        tc_add(m, MG_PD2B, off, c, c, !ebias, mcap, hm);
        tc_add(m, MG_RC1, off, c, c, !ebias, mcap, (px || c > kRc16MinC) ? hm : 0);
        tc_add(m, MG_RC2, off, c, c, !ebias, mcap, (px || c > kRc16MinC) ? hm : 0);
        if (ebias) { m.ebias_off = (uint32_t)off; off += (size_t)4 * c * 4; }     // [conv.0, dense2, conv1, conv2][row][hi, lo, 0, 0]
    }
    TcPlan& h = P.head;
    h = TcPlan{};
    h.base = base; h.ngemm = HG_COUNT; h.resident = 0; h.nslot = 2;
    tc_add(h, HG_C2, off, a.dims[4], a.dims[4], true, 32768, hm);          // mirrors HeadG::h16
    tc_add(h, HG_DENSE, off, kHeadN, a.dims[4], true, 32768, hm);
    P.floats = off;
    for (int l = 0; l < 4; ++l) {
        P.branch[l][0].trace = P.branch[l][1].trace = g_tc_trace_sel == 0 ? g_tc_trace : nullptr;
        P.merge[l].trace = g_tc_trace_sel == 1 ? g_tc_trace : nullptr;
    }
    P.head.trace = nullptr;
    if (out) *out = P;
}
static void tc_build_plans(const balf_detector_arch& a, const float* base, TcPlans* out, int px = 0) {
    size_t off = 0;
    TcPlans P0;
    tc_build_plans_px(a, base, &P0, 0, off);
    if (px) tc_build_plans_px(a, base, out, 1, off);
    else if (out) *out = P0;
}

#ifdef BALF_TC_MAIN
size_t tc_blob_floats(const balf_detector_arch& a) {
    TcPlans P;
    tc_build_plans(a, nullptr, &P, 1);
    return P.floats;
}

struct Fold { const float* gamma; const float* beta; const float* alpha; const float* add; };

static void tc_pack_one(const TcPlan& p, int gi, const float* wT, int ld, int n0, int k_real, const float* bias, Fold f,
                        float* blob, cudaStream_t st) {
    const TcGemm& g = p.g[gi];
    const int k_pad = g.nblk * g.kb;
    if (g.h16 == 2)
        tc_pack_x3_kernel<<<cdiv(g.rows * k_pad, 256), 256, 0, st>>>(wT, ld, n0, g.rows, k_real, k_pad, g.kb, f.gamma, f.alpha,
                                                                     reinterpret_cast<__half*>(blob + g.goff));
    else if (g.h16)
        tc_pack_h16_kernel<<<cdiv(g.rows * k_pad, 256), 256, 0, st>>>(wT, ld, n0, g.rows, k_real, k_pad, g.kb, f.gamma, f.alpha,
                                                                      reinterpret_cast<__half*>(blob + g.goff));
    else
        tc_pack_kernel<<<cdiv(g.rows * k_pad, 256), 256, 0, st>>>(wT, ld, n0, g.rows, k_real, k_pad, g.kb, f.gamma, f.alpha, blob + g.goff);
    if (g.bias)   // two chunk planes after the last block's kb columns; the second stays zero (blob is memset)
        tc_pack_bias_kernel<<<cdiv(g.rows, 128), 128, 0, st>>>(wT, ld, n0, g.rows, k_real, bias, f.beta, f.alpha, f.add,
                                                               blob + g.goff + (size_t)g.rows * k_pad / (g.h16 == 1 ? 2 : 1));
    else if (p.ebias_off && bias) {   // biases added by the epilogues: the same folded (hi, lo) pairs, in the plan's bias-vector area
        const int slot = gi == MG_CONV0 ? 0 : gi == MG_PD2B ? 1 : gi == MG_RC1 ? 2 : 3;
        tc_pack_bias_kernel<<<cdiv(g.rows, 128), 128, 0, st>>>(wT, ld, n0, g.rows, k_real, bias, f.beta, f.alpha, f.add,
                                                               blob + p.ebias_off + (size_t)slot * g.rows * 4);
    }
}

// fp32-path packed weights (DetW) -> tc blob
int tc_pack_weights(const balf_detector_arch& a, const DetW& w, float* blob, cudaStream_t st) {
    BALF_CUDA_OK(cudaMemsetAsync(blob, 0, tc_blob_floats(a) * sizeof(float), st));
    const Fold none{nullptr, nullptr, nullptr, nullptr};
    for (int px = 0; px < 2; ++px) {
    TcPlans P;
    tc_build_plans(a, blob, &P, px);
    for (int l = 0; l < 4; ++l) {
        const int ci = a.dims[l], c = a.dims[l + 1];
        const DownW& d = w.down[l];
        for (int b = 0; b < 2; ++b) {
            const TcPlan& p = P.branch[l][b];
            const DownW::Branch& r = d.br[b];
            tc_pack_one(p, BG_CONV0, d.conv0_w, c, 0, ci, d.conv0_b, none, blob, st);
            tc_pack_one(p, BG_PD1, d.pd1_w, 2 * c, b * c, c, d.pd1_b, Fold{d.pn_w, d.pn_b, nullptr, nullptr}, blob, st);
            tc_pack_one(p, BG_D1A, r.d1_w, 2 * c, 0, c, r.d1_b, Fold{r.n_w, r.n_b, nullptr, nullptr}, blob, st);
            tc_pack_one(p, BG_D1B, r.d1_w, 2 * c, c, c, r.d1_b, Fold{r.n_w, r.n_b, nullptr, nullptr}, blob, st);
            tc_pack_one(p, BG_WM, r.gd_w, 64, 0, 64, nullptr, none, blob, st);
            tc_pack_one(p, BG_D2, r.d2_w, c, 0, c, r.d2_b, none, blob, st);
        }
        const TcPlan& m = P.merge[l];
        tc_pack_one(m, MG_CONV0, d.conv0_w, c, 0, ci, d.conv0_b, none, blob, st);
        tc_pack_one(m, MG_PD2A, d.pd2_w, c, 0, c, nullptr, none, blob, st);
        tc_pack_one(m, MG_PD2B, d.pd2_w + (size_t)c * c, c, 0, c, d.pd2_b, none, blob, st);
        tc_pack_one(m, MG_RC1, d.rc1_w, c, 0, c, d.rc1_b, Fold{d.rn_w, d.rn_b, nullptr, nullptr}, blob, st);
        tc_pack_one(m, MG_RC2, d.rc2_w, c, 0, c, d.rc2_b, none, blob, st);
    }
    tc_pack_one(P.head, HG_C2, w.down[3].c2_w, a.dims[4], 0, a.dims[4], w.down[3].c2_b, none, blob, st);
    // logits = (x W^T + b) * alpha + beta_bn  (eval BatchNorm folded, decoder.py:18-22)
    tc_pack_one(P.head, HG_DENSE, w.head.w, kHeadPad, 0, a.dims[4], w.head.b, Fold{nullptr, nullptr, w.head.alpha, w.head.beta}, blob, st);
    }
    BALF_LAUNCH_OK();
    return 0;
}

#endif  // BALF_TC_MAIN

// ------------------------------------------------------------------------------------------ host: one stage
static int g_num_sms = 0;
static int num_sms() {
    if (!g_num_sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
        if (g_num_sms <= 0) g_num_sms = 148;
    }
    return g_num_sms;
}

// persistent grid: one CTA per resident slot.  Resident CTAs per SM = min over shared memory (227 KB usable,
// 1 KB reserved per CTA), registers (64 K per SM) and TMEM columns (512 per SM).
template <typename K>
static int tc_launch_cfg(K kernel, size_t smem, int tmem_cols, int ntiles, int* grid, int groups = 1, int group_threads = NT2) {
    BALF_REQUIRE(smem <= 227 * 1024, "internal: tc kernel needs %zu bytes of shared memory", smem);
    BALF_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    BALF_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    cudaFuncAttributes fa;
    BALF_CUDA_OK(cudaFuncGetAttributes(&fa, kernel));
    const int regs_per_cta = ((fa.numRegs + 7) / 8 * 8) * group_threads * groups;
    ntiles = (ntiles + groups - 1) / groups;                // CTAs needed
    int per_sm = (int)((227 * 1024) / (smem + 1024));
    if (regs_per_cta > 0 && 65536 / regs_per_cta < per_sm) per_sm = 65536 / regs_per_cta;
    if (512 / tmem_cols < per_sm) per_sm = 512 / tmem_cols;
    if (per_sm < 1) per_sm = 1;
    const int cap = num_sms() * per_sm;
    *grid = ntiles < cap ? ntiles : cap;
    return 0;
}


template <int CIN, int C, int PX>
static int tc_launch_branches(const float* xin, const DownW& w, const TcPlans& P, int level, const UnitGeom& g, int ntiles,
                              float* u, float* v, float* su, float* sv, cudaStream_t st) {
    using Cfg = BranchCfg<C, PX>;
    constexpr int NG = Cfg::groups;
    int grid = 0;
    for (int b = 0; b < 2; ++b) {
        const TcPlan& p = P.branch[level][b];
        const size_t smem = tc_smem_bytes(Cfg::region, p, NG, Cfg::xch);
        if (b == 0) {
            if (int e = tc_launch_cfg(tc_branch_kernel<CIN, C, 0, PX>, smem, tc_cols(Cfg::ncols * NG), ntiles, &grid, NG, Cfg::NTG)) return e;
            ProfScope ps(C == 32 ? "det_branch_grid_c32" : C == 64 ? "det_branch_grid_c64" : C == 128 ? "det_branch_grid_c128" : "det_branch_grid_c256", st);
            tc_branch_kernel<CIN, C, 0, PX><<<grid, Cfg::NTG * NG, smem, st>>>(xin, w, p, g, u, su);
        } else {
            if (int e = tc_launch_cfg(tc_branch_kernel<CIN, C, 1, PX>, smem, tc_cols(Cfg::ncols * NG), ntiles, &grid, NG, Cfg::NTG)) return e;
            ProfScope ps(C == 32 ? "det_branch_block_c32" : C == 64 ? "det_branch_block_c64" : C == 128 ? "det_branch_block_c128" : "det_branch_block_c256", st);
            tc_branch_kernel<CIN, C, 1, PX><<<grid, Cfg::NTG * NG, smem, st>>>(xin, w, p, g, v, sv);
        }
    }
    return 0;
}

template <int CIN, int C, int PX>
static int tc_run_level(const float* xin, const DownW& w, const TcPlans& P, int level, int Bc, int h, int wd,
                        float* u, float* v, float* r, float* q, float* partial, cudaStream_t st, int r16) {
    UnitGeom g{h, wd, h / 8, wd / 8, h * wd / 64, Bc * (h * wd / 64), 1.0f / (float)(h * wd / 64), 1.0f / (float)(wd / 8), 1.0f / (float)(wd / 8)};
    BALF_REQUIRE(g.total_units < (1 << 23), "internal: %d units in one pass exceed the fast_div range", g.total_units);
    const int ntiles = (g.total_units + 1) / 2;
    int grid = 0;
    BALF_REQUIRE((plan_matches<BranchG<CIN, C, PX>>(P.branch[level][0]) && plan_matches<BranchG<CIN, C, PX>>(P.branch[level][1]) &&
                  plan_matches<MergeG<CIN, C, PX>>(P.merge[level])), "internal: compile-time and packed GEMM plans differ (level %d)", level);
    // (r and q are free until the merge kernel writes them: scratch of the stage-4 branch kernels' residual round trip)
    if (int e = tc_launch_branches<CIN, C, PX>(xin, w, P, level, g, ntiles, u, v, r, q, st)) return e;
    if constexpr (C <= 64) {
        const TcPlan& p = P.merge[level];
        BALF_REQUIRE(g.total_units % 2 == 0, "internal: odd unit count at stage %d", level);
        const size_t smem = tc_smem_bytes(MergeBulkCfg<CIN, C, PX>::region, p, 1, MergeBulkCfg<CIN, C, PX>::xch);
        if (int e = tc_launch_cfg(tc_merge_bulk_kernel<CIN, C, PX>, smem, MergeBulkCfg<CIN, C, PX>::ncols, ntiles, &grid)) return e;
        ProfScope ps(C == 32 ? "det_merge_c32" : "det_merge_c64", st);
        tc_merge_bulk_kernel<CIN, C, PX><<<grid, NT2, smem, st>>>(xin, w, p, g, u, v, r, q, partial);
    } else {
        const TcPlan& p = P.merge[level];
        BALF_REQUIRE((!MergeCfg<C, PX>::bulk_uv || g.total_units % 2 == 0), "internal: odd unit count at stage %d", level);
        const size_t smem = tc_smem_bytes(MergeCfg<C, PX>::region, p, 1, MergeCfg<C, PX>::xch);
        if (int e = tc_launch_cfg(tc_merge_kernel<CIN, C, PX>, smem, MergeCfg<C, PX>::ncols, ntiles, &grid, 1, MergeCfg<C, PX>::NT)) return e;
        ProfScope ps(C == 128 ? "det_merge_c128" : "det_merge_c256", st);
        tc_merge_kernel<CIN, C, PX><<<grid, MergeCfg<C, PX>::NT, smem, st>>>(xin, p, g, u, v, r, q, partial, r16);
    }
    BALF_COUNT_LAUNCH(3);
    BALF_LAUNCH_OK();
    return 0;
}

// one stage / the head in precision class PX (0 single-rounded, 1 split): instantiated in detector_tc.cu (PX = 0) and detector_tc_x3.cu
template <int PX>
int tc_level_px(int level, const float* xin, const DownW& w, const balf_detector_arch& a, const float* blob,
                int Bc, int h, int wd, float* u, float* v, float* r, float* q, float* partial, cudaStream_t st, int r16) {
    TcPlans P;
    tc_build_plans(a, blob, &P, PX);
    switch (level) {
        case 0: return tc_run_level<3, 32, PX>(xin, w, P, 0, Bc, h, wd, u, v, r, q, partial, st, r16);
        case 1: return tc_run_level<32, 64, PX>(xin, w, P, 1, Bc, h, wd, u, v, r, q, partial, st, r16);
        case 2: return tc_run_level<64, 128, PX>(xin, w, P, 2, Bc, h, wd, u, v, r, q, partial, st, r16);
        default: return tc_run_level<128, 256, PX>(xin, w, P, 3, Bc, h, wd, u, v, r, q, partial, st, r16);
    }
}
template <int PX>
int tc_head_px(const float* r, const float* q, const float* scale, const balf_detector_arch& a,
               const float* blob, int Bc, int hc, int wc, float* logits, float* prob, cudaStream_t st, int r16) {
    TcPlans P;
    tc_build_plans(a, blob, &P, PX);
    UnitGeom g{hc, wc, hc / 8, wc / 8, hc * wc / 64, Bc * (hc * wc / 64), 1.0f / (float)(hc * wc / 64), 1.0f / (float)(wc / 8), 1.0f / (float)(wc / 8)};
    BALF_REQUIRE(g.total_units < (1 << 23), "internal: %d units in one pass exceed the fast_div range", g.total_units);
    const int ntiles = (g.total_units + 1) / 2;
    const size_t smem = tc_smem_bytes((uint32_t)TM * 256 * 4, P.head);
    int grid = 0;
    BALF_REQUIRE((plan_matches<HeadG<256, PX>>(P.head)), "internal: compile-time and packed GEMM plans differ (head)");
    if (int e = tc_launch_cfg(tc_head_kernel<256, PX>, smem, 512, ntiles, &grid)) return e;
    {
        ProfScope ps("det_head", st);
        tc_head_kernel<256, PX><<<grid, NT2, smem, st>>>(r, q, scale, P.head, g, a.cell, logits, prob, PX ? 0 : r16);
    }
    BALF_COUNT_LAUNCH(1);
    BALF_LAUNCH_OK();
    return 0;
}

#ifdef BALF_TC_MAIN
extern template int tc_level_px<1>(int, const float*, const DownW&, const balf_detector_arch&, const float*, int, int, int, float*, float*,
                                   float*, float*, float*, cudaStream_t, int);
extern template int tc_head_px<1>(const float*, const float*, const float*, const balf_detector_arch&, const float*, int, int, int, float*,
                                  float*, cudaStream_t, int);

int tc_run_level_dispatch(int level, const float* xin, const DownW& w, const balf_detector_arch& a, const float* blob,
                          int Bc, int h, int wd, float* u, float* v, float* r, float* q, float* partial, cudaStream_t st, int px, int r16) {
    return px ? tc_level_px<1>(level, xin, w, a, blob, Bc, h, wd, u, v, r, q, partial, st, r16)
              : tc_level_px<0>(level, xin, w, a, blob, Bc, h, wd, u, v, r, q, partial, st, r16);
}

int tc_run_head(const float* r, const float* q, const float* scale, const balf_detector_arch& a,
                const float* blob, int Bc, int hc, int wc, float* logits, float* prob, cudaStream_t st, int px, int r16) {
    return px ? tc_head_px<1>(r, q, scale, a, blob, Bc, hc, wc, logits, prob, st, r16)
              : tc_head_px<0>(r, q, scale, a, blob, Bc, hc, wc, logits, prob, st, r16);
}
#endif  // BALF_TC_MAIN

}  // namespace balf

#ifdef BALF_TC_MAIN
extern "C" int balf_debug_set_trace(void* buf) {
    balf::g_tc_trace = static_cast<long long*>(buf);
    return 0;
}
#endif
