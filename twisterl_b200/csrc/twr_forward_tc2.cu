// twr_forward_tc2.cu -- K2, tensor-core variant for sm_100a: batched Policy::_raw_predict (rust/src/nn/policy.rs:79-100)
// as two chained tcgen05 GEMMs, run by CTA pairs (tcgen05 cta_group::2).
//
//   GEMM1 (embedding, layers.rs:56-86):     D1 = onehot(obs)[256 x K1] * Emb[K1 x E]
//   epilogue-1:                             h1 = relu(D1 + emb_bias) -> fp16 hi + lo, stored back into the same TMEM columns
//   GEMM2 (common Linear, layers.rs:31-37): D2 = h1[256 x E] * W1[E x H]   (A operand read from TMEM)
//   epilogue-2 (heads, policy.rs:89-97):    h2 = relu(D2 + b1); logits = Wa h2 + ba; value = wv.h2 + bv
//
// Every fp32 operand is split into two fp16 terms (x = hi + lo); which of the products are accumulated is the engine's
// precision (TERMS below).  E runs in chunks of 128 features and GEMM1 over PAIRS of chunks: an embedding of an odd
// number of chunks is zero-padded to the next pair in the operand image (zero table columns, bias and W1 rows), so the
// padded features give h1 = 0 and add exact zeros to D2.
//
// Two CTAs of a cluster cooperate on a 256-env tile:
// every tcgen05.mma is M=256 (rows 0..127 live in CTA 0's TMEM, 128..255 in CTA 1's) and the B operand
// (weights) is split along N between the two CTAs' shared memory -- each SM therefore streams only
// HALF of the operand bytes per env and issues M = 256 instructions (see DESIGN.md for what bounds it).
//
//   CTA 0 (leader): warp 1 issues all MMAs; its mbarriers collect the arrivals of both CTAs
//   CTA 1 (peer)  : its TMA loads credit the leader's `full` barrier (2-SM TMA); epilogue warps
//                   arrive remotely (mapa + mbarrier.arrive on the shared::cluster address) on the leader's barriers
//   both          : warp 0 streams this CTA's half tiles with 2-SM tensor-map TMA into its own 8-slot ring;
//                   warps 2..9 are the epilogue of this CTA's 128 envs (two warps per TMEM lane quarter: epilogue-1
//                   conversion, heads, and -- lower column half -- the fused collect step, upper half -- the one-hot
//                   operand of the next item); tcgen05.commit.cta_group::2 (multicast) publishes accumulators / frees
//                   ring slots in both CTAs.
//
// Per 256-env item: GEMM1 runs over PAIRS of 128-feature chunks as N = 256 MMAs (N = 128 issues at half rate), the
// last k-block finishing the two chunks one after the other; GEMM2 (3 split passes, A from TMEM) follows per chunk.
// A launch is persistent over up to 32 time steps of the tiles a pair owns (struct Sched balances left-over tiles
// along time between pairs); the fused collect step of an item is deferred behind the next item's first epilogue-1.
#include "twr_kernels.cuh"
#include "twr_tc_ptx.cuh"
#include "twr_step.cuh"

#include <atomic>
#include <cstdlib>
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>
#include <map>
#include <mutex>

extern std::atomic<long long> g_twr_launches;

namespace {

constexpr int TM = 128;               // envs per CTA (the pair covers 256)
constexpr int NTHREADS = 320;          // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue (two per TMEM lane quarter)
constexpr int NEPI = 256;
constexpr int TILE_BYTES = 16384;
constexpr int NSLOTS = 8;
constexpr int MAX_KB1 = 4;
constexpr int MAX_OBS = 32;

constexpr int SM_A1 = 0;
constexpr int SM_RING = SM_A1 + MAX_KB1 * TILE_BYTES;
// fp8 correction terms (TERMS bit 4): the first two ring slots hold the e5m2 copy of the one-hot operand (two k-blocks of
// 128 one-byte columns), the ring keeps the other six
constexpr int SM_A8 = SM_RING;
constexpr int A8_TILES = 2;
constexpr int SM_MISC = SM_RING + NSLOTS * TILE_BYTES;
constexpr int SM_HEADW = SM_MISC;
constexpr int SM_B1 = SM_HEADW + 8192;
constexpr int SM_EMBB = SM_B1 + 1024;
constexpr int SM_PART = SM_EMBB + 4096;                   // [2][128][8] float: head partial sums of the upper column half
constexpr int SM_PERM = SM_PART + 2 * TM * 8 * 4;         // [4][128] int8: twist index of the tiles in flight
constexpr int SM_OPERM = SM_PERM + 4 * TM;                // uint8 copy of the twist tables (obs_perms), up to OPERM_MAX entries
constexpr int OPERM_MAX = 2048;
constexpr int SM_BARS = SM_OPERM + OPERM_MAX;
constexpr int SM_TOTAL = SM_BARS + 512;
static_assert(SM_TOTAL <= 227 * 1024, "shared memory budget");

enum Bar { B_FULL0 = 0, B_EMPTY0 = NSLOTS, B_A1_FULL = 2 * NSLOTS, B_A1_EMPTY, B_D1_FULL0, B_D1_FULL1,
           B_A2_FULL0, B_A2_FULL1, B_D2_FULL, B_D2_EMPTY, B_COUNT };
static_assert(B_COUNT * 8 + 8 <= 384, "barrier area (the last 128 bytes hold the action twists)");

// ---- cluster / cta_group::2 PTX ----
// TMA tile load (tensor map over the packed operand image, one box = one 16 KB ring slot) whose completion
// bytes are credited to the LEADER CTA's mbarrier (peer bit of the barrier address cleared), the
// cta_group::2 form CUTLASS uses for 2-SM MMA (cute/arch/copy_sm100_tma.hpp, SM100_TMA_2SM_LOAD_2D).
__device__ __forceinline__ void tma_load_2sm(uint32_t dst, const CUtensorMap* tmap, int32_t c0, int32_t c1, uint32_t mbar) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(mbar & 0xFEFFFFFFu), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ uint32_t ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `local` (a shared::cta address) inside CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa(uint32_t local, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");   // default .release.cta like cutlass ClusterBarrier::arrive
}
// Waits on barriers that also collect remote arrivals.  Default (.acquire.cta) semantics like cutlass
// ClusterBarrier::wait: a cluster-scope acquire costs a CCTL.IVALL (L1 invalidate, ~400+ cycles) per wait, and no
// generic-proxy data crosses CTAs here -- operands travel through TMEM / the async proxy.
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    for (uint32_t spins = 0; !done; ++spins) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (!done && spins > (1u << 26)) __trap();
    }
}
__device__ __forceinline__ void mbar_wait_cluster_t(uint32_t bar, uint32_t parity, long long& acc, bool timed) {
    if (!timed) { mbar_wait_cluster(bar, parity); return; }
    const long long t0 = clock64();
    mbar_wait_cluster(bar, parity);
    acc += clock64() - t0;
}
__device__ __forceinline__ void tc2_commit(uint32_t bar) {   // arrives on `bar` in BOTH CTAs of the pair
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tc2_mma(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc2_mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// instruction descriptor (cute::UMMA::InstrDescriptor): c=F32 [4,6)=1, a=b=F16 (0), K-major both,
// N>>3 at [17,23), M>>4 at [24,29)
constexpr uint32_t IDESC_256x128 = (1u << 4) | ((128u >> 3) << 17) | ((256u >> 4) << 24);
constexpr uint32_t IDESC_256x256 = (1u << 4) | ((256u >> 3) << 17) | ((256u >> 4) << 24);
// kind::f8f6f4 (K = 32 per instruction): operand formats at [7,10) (A) and [10,13) (B), 0 = e4m3, 1 = e5m2
// (cute::UMMA::InstrDescriptor / MXF8F6F4Format)
__device__ __forceinline__ void tc2_mma8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc2_mma8_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
constexpr uint32_t idesc8(uint32_t n, uint32_t a_fmt, uint32_t b_fmt) {
    return (1u << 4) | (a_fmt << 7) | (b_fmt << 10) | ((n >> 3) << 17) | ((256u >> 4) << 24);
}
// The two correction terms as fp8 products (TWR_PREC_F16_F8C).  Each is ~2^-12 of its main term, so 2-3 mantissa bits are
// enough to keep the 1e-3 grade (tests/test_gpu_precision.py measures it), and an fp8 MMA covers K = 32 at the cost of an
// fp16 K = 16 one: half the instructions for these two terms.  This variant carries the hidden activations SCALED by
// S = 16 (table and embedding bias x 16, common-layer weight / 16: powers of two, nothing is rounded differently; fp16
// holds 16 h1 up to h1 = 4094 and the conversions saturate), which puts the fp16 residue of an activation where e5m2
// resolves it without a multiplication in epilogue-1 (-2.4 % on the collect):
//   GEMM1: one-hot value 2^-10 (e5m2 0x14)    x  e4m3((16 t - fp16(16 t)) * 2^10)        [t = table entry (+ folded bias)]
//   GEMM2: e5m2(16 h1 - fp16(16 h1))          x  e5m2(W / 16)                            [main term: fp16(16 h1) x fp16(W / 16)]
constexpr uint8_t  ONE8 = 0x14;          // 2^-10
constexpr float    H1_SCALE8 = 16.0f, TABLE8_SCALE = 1024.0f, W8_SCALE = 1.0f / 16.0f;
__host__ __device__ __forceinline__ uint32_t tile_off8(uint32_t row, uint32_t k) {       // [128 rows][128 one-byte k], 128B swizzle
    return (row >> 3) * 1024u + (row & 7u) * 128u + ((((k >> 4) ^ row) & 7u) << 4) + (k & 15u);
}

// cN > 0: GEMM1 runs over the COMPACT table of a GridWorld policy -- compact row k = cell (k / 4), value (k % 4) stands
// for table row (k / 4) * cN + (k % 4); the other obs_size - 4 * cN rows are unreachable (lib.rs:74-81: cell values 0..3)
// f8 = 1: the operand image of the fp8-correction variant (it follows the standard image in the same buffer, row0 = its
// first tensor-map row); NKB8 = k-blocks of 128 of the one-byte one-hot operand
struct Tc2Params { int NC, NKB1, E, H, cN, f8, NKB8, row0, fold; };
__host__ __device__ inline size_t slots_g1(const Tc2Params& t) { return t.f8 ? (size_t)(t.NC / 2) * (t.NKB1 + t.NKB8) : (size_t)t.NC * t.NKB1; }
__host__ __device__ inline size_t slots_g2(const Tc2Params& t) { return t.f8 ? (size_t)t.NC * (t.H == 256 ? 3 : 2) : (size_t)t.NC * (t.H == 256 ? 4 : 2); }
__host__ __device__ inline size_t slots_per_rank(const Tc2Params& t) { return slots_g1(t) + slots_g2(t); }
// fp8 variant, GEMM1 stream of one chunk pair: hi k-blocks in order, the one-byte k-block j (= hi k-blocks 2j, 2j+1) right
// after hi k-block 2j+1; the LAST hi and the LAST one-byte k-block close the sequence (they are issued chunk by chunk as
// N = 128 MMAs, see the kernel).  Unit u of NKB1 + NKB8 -> (is8, k-block, last).
__host__ __device__ inline void g1_unit8(int NKB1, int NKB8, int u, int& is8, int& kb, int& last) {
    int i = 0;
    for (int k = 0; k < NKB1 - 1; ++k) {
        if (i++ == u) { is8 = 0; kb = k; last = 0; return; }
        if ((k & 1) && (k >> 1) < NKB8 - 1) { if (i++ == u) { is8 = 1; kb = k >> 1; last = 0; return; } }
    }
    if (i++ == u) { is8 = 0; kb = NKB1 - 1; last = 1; return; }
    is8 = 1; kb = NKB8 - 1; last = 1;
}

// Operand image per CTA rank r (rank 0 image, then rank 1 image), in streaming order, 16 KB per ring slot:
//   G1 slot (s,kb,part) : [128 rows x 64 k] of the hi (part 0) or lo (part 1) table, rows n = feature (2s+r)*128 + (0..127),
//                         k = obs row kb*64 + kk -- GEMM1 runs as N = 256 MMAs over a PAIR of 128-feature chunks (both D1
//                         buffers at once; rank r's half of B is chunk 2s+r): N = 128 MMAs issue at half rate (DESIGN.md)
//   G2 slot (j,kb,part) : [128 rows x 64 k], rows n = output r*128 + (0..127), k = feature j*128 + kb*64 + kk      (H = 256)
//   G2 slot (j,part)    : two [64 rows x 64 k] sub-tiles (kb = 0, 1), rows n = output r*64 + (0..63)              (H = 128)
__global__ void __launch_bounds__(256) k_tc2_pack(PolicyDev p, Tc2Params t, __half* __restrict__ pack) {
    const size_t spr = slots_per_rank(t), n1 = slots_g1(t);
    const size_t total = 2 * spr * (TILE_BYTES / 2);
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const size_t gslot = idx / (TILE_BYTES / 2);
        const uint32_t within = (uint32_t)(idx % (TILE_BYTES / 2));
        const int r = (int)(gslot / spr);
        const size_t slot = gslot % spr;
        float x = 0.0f;
        int lo_part;
        uint32_t off;
        if (slot < n1) {
            const int sc = (int)(slot / (2 * t.NKB1)), kb = (int)((slot % (2 * t.NKB1)) / 2);
            lo_part = (int)(slot % 2);
            const uint32_t row = within >> 6, kk = within & 63u;
            // rows of rank r: chunk 2sc+r for the N = 256 MMAs; in the LAST k-block the two chunks are finished one after
            // the other with N = 128 MMAs (rows 0..63 = rank r's half of chunk 2sc, rows 64..127 = its half of chunk 2sc+1)
            const int f = kb == t.NKB1 - 1 ? (2 * sc + (int)(row >> 6)) * 128 + r * 64 + (int)(row & 63u) : (2 * sc + r) * 128 + (int)row;
            int k = kb * 64 + (int)kk;
            if (t.cN > 0) k = (k >> 2) < t.cN ? (k >> 2) * t.cN + (k & 3) : p.obs_size;
            if (k < p.obs_size && f < p.E) x = p.emb[(size_t)k * p.E + f];
            off = tile_off(row, kk);
        } else if (t.H == 256) {
            const size_t q = slot - n1;
            const int j = (int)(q / 4), kb = (int)((q % 4) / 2);
            lo_part = (int)(q % 2);
            const uint32_t row = within >> 6, kk = within & 63u;
            const int o = r * 128 + (int)row, f = j * 128 + kb * 64 + (int)kk;
            if (f < p.E) x = p.w1[(size_t)f * p.H + o];
            off = tile_off(row, kk);
        } else {
            const size_t q = slot - n1;
            const int j = (int)(q / 2);
            lo_part = (int)(q % 2);
            const uint32_t row = within >> 6, kk = within & 63u;
            const int kb = (int)(row >> 6);
            const int o = r * 64 + (int)(row & 63u), f = j * 128 + kb * 64 + (int)kk;
            if (f < p.E) x = p.w1[(size_t)f * p.H + o];
            off = (uint32_t)kb * 8192u + tile_off(row & 63u, kk);
        }
        const __half hi = __float2half_rn(x);
        const __half v = lo_part ? __float2half_rn(x - __half2float(hi)) : hi;
        *reinterpret_cast<__half*>(reinterpret_cast<unsigned char*>(pack) + gslot * TILE_BYTES + off) = v;
    }
}

// Operand image of the fp8-correction variant, per CTA rank, in streaming order:
//   per chunk pair sc: the units of g1_unit8 -- hi slots exactly as above (part 0), one-byte slots [128 rows x 128 k] of
//                      e4m3((table - hi) * 2^14), rows like the hi slot of the same kind (plain / last)
//   per chunk j      : H = 256: hi kb 0, hi kb 1 (as above), then [128 rows x 128 k] e5m2(W * 2^-6), rows n = output r*128 + ..
//                      H = 128: the hi slot (two sub-tiles), then [64 rows x 128 k] e5m2(W * 2^-6), rows n = output r*64 + ..
__global__ void __launch_bounds__(256) k_tc2_pack8(PolicyDev p, Tc2Params t, unsigned char* __restrict__ pack) {
    const size_t spr = slots_per_rank(t), n1 = slots_g1(t);
    const size_t total = 2 * spr * TILE_BYTES;                 // one thread per BYTE position (fp16 slots: even positions only)
    const int upc = t.NKB1 + t.NKB8;
    auto w1s = [&](int f, int o) { return f < p.E ? p.w1[(size_t)f * p.H + o] * W8_SCALE : 0.0f; };   // scaled W1, padding rows 0
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const size_t gslot = idx / TILE_BYTES;
        const uint32_t within = (uint32_t)(idx % TILE_BYTES);
        const int r = (int)(gslot / spr);
        const size_t slot = gslot % spr;
        unsigned char* dst = pack + gslot * TILE_BYTES;
        const uint32_t row = within >> 7;
        if (slot < n1) {
            const int sc = (int)(slot / upc);
            int is8, kb, last;
            g1_unit8(t.NKB1, t.NKB8, (int)(slot % upc), is8, kb, last);
            if (!is8 && (within & 1u)) continue;
            const uint32_t kk = is8 ? (within & 127u) : ((within & 127u) >> 1);
            const int f = last ? (2 * sc + (int)(row >> 6)) * 128 + r * 64 + (int)(row & 63u) : (2 * sc + r) * 128 + (int)row;
            int k = is8 ? kb * 128 + (int)kk : kb * 64 + (int)kk;
            if (t.cN > 0) k = (k >> 2) < t.cN ? (k >> 2) * t.cN + (k & 3) : p.obs_size;
            // PolicyDev::tc_fold: the embedding bias rides on the rows of block 0 (exactly one of them is in every observation)
            const float x = k < p.obs_size && f < p.E ? (p.emb[(size_t)k * p.E + f] + (k < t.fold ? p.emb_b[f] : 0.0f)) * H1_SCALE8 : 0.0f;
            const __half hi = __float2half_rn(x);
            if (is8) dst[tile_off8(row, kk)] = (unsigned char)__nv_cvt_float_to_fp8((x - __half2float(hi)) * TABLE8_SCALE, __NV_SATFINITE, __NV_E4M3);
            else *reinterpret_cast<__half*>(dst + tile_off(row, kk)) = hi;
        } else if (t.H == 256) {
            const size_t q = slot - n1;
            const int j = (int)(q / 3), u = (int)(q % 3);
            const int o = r * 128 + (int)row;
            if (u < 2) {
                if (within & 1u) continue;
                const uint32_t kk = (within & 127u) >> 1;
                *reinterpret_cast<__half*>(dst + tile_off(row, kk)) = __float2half_rn(w1s(j * 128 + u * 64 + (int)kk, o));
            } else {
                const uint32_t kk = within & 127u;
                dst[tile_off8(row, kk)] = (unsigned char)__nv_cvt_float_to_fp8(w1s(j * 128 + (int)kk, o), __NV_SATFINITE, __NV_E5M2);
            }
        } else {
            const size_t q = slot - n1;
            const int j = (int)(q / 2), u = (int)(q % 2);
            if (u == 0) {
                if (within & 1u) continue;
                const uint32_t kk = (within & 127u) >> 1;
                const int kb = (int)(row >> 6);
                const int o = r * 64 + (int)(row & 63u);
                *reinterpret_cast<__half*>(dst + (uint32_t)kb * 8192u + tile_off(row & 63u, kk)) = __float2half_rn(w1s(j * 128 + kb * 64 + (int)kk, o));
            } else {
                const uint32_t kk = within & 127u;
                const float w = row < 64 ? w1s(j * 128 + (int)kk, r * 64 + (int)row) : 0.0f;
                dst[tile_off8(row, kk)] = (unsigned char)__nv_cvt_float_to_fp8(w, __NV_SATFINITE, __NV_E5M2);
            }
        }
    }
}

// Item schedule of one CTA pair for a launch of T steps over G groups (256-env tiles pairs) on P pairs.
// Plain: the pair owns groups pair, pair+P, ... and walks them step-major.  Balanced (T >= 4, >= 2 own groups per
// pair, G % P != 0): the G % P left-over groups are cut along time into pieces of <= Lp steps; piece k of a group
// runs on the pair after the one that ran piece k-1, at item slots 2*step (+ bal_delta per hand-off), so no pair
// does more than floor(G/P)*T + Lp items instead of (floor(G/P)+1)*T.  scripts/sim_balance.py is the host model.
struct Sched {
    int n_items, lanes, T, P;
    int nA, nB, sA0, pA0, gA;   // dependent piece A = steps [sA0, sA0+nA) of extra group gA; head piece B = steps [0, nB) of gA+1
};
__device__ __forceinline__ Sched make_sched(int G, int P, int T, int pair, int delta) {
    Sched s;
    s.T = T; s.P = P; s.nA = 0; s.nB = 0; s.sA0 = 0; s.pA0 = 0; s.gA = 0;
    const int base = G / P, rem = G % P;
    if (delta > 0 && T >= 4 && base >= 2 && rem > 0) {
        s.lanes = base;
        const int X = rem * T;
        int Lp = (X + P - 1) / P;
        if (Lp < 4) Lp = 4;
        const int x0 = min(X, pair * Lp), x1 = min(X, x0 + Lp), nX = x1 - x0;
        if (nX > 0) {
            s.gA = x0 / T; s.sA0 = x0 % T;
            s.nA = min(nX, T - s.sA0); s.nB = nX - s.nA;
            int dA = s.sA0 > 0 ? delta * (pair - (s.gA * T) / Lp) : 0;
            // the piece must end inside this pair's sequence (base*T + nX items): with only two own groups the slack of
            // late hand-offs is clamped -- a shorter slack can make the consumer wait, never deadlock
            dA = max(0, min(dA, base * T + nX - 1 - 2 * (s.sA0 + s.nA - 1)));
            s.pA0 = 2 * s.sA0 + dA;
        }
        s.n_items = base * T + nX;
    } else {
        s.lanes = (G - pair + P - 1) / P;
        s.n_items = s.lanes * T;
    }
    return s;
}
// item i of `pair` -> (group, step); extra = 1 for piece A, 2 for piece B, 0 for an own group
__device__ __forceinline__ void sched_item(const Sched& s, int pair, int i, int& group, int& step, int& extra) {
    if (s.nA + s.nB == 0) { group = pair + (i % s.lanes) * s.P; step = i / s.lanes; extra = 0; return; }
    const int ja = i - s.pA0;
    if (!(i & 1) && (i >> 1) < s.nB) { group = s.lanes * s.P + s.gA + 1; step = i >> 1; extra = 2; return; }
    if (ja >= 0 && !(ja & 1) && (ja >> 1) < s.nA) { group = s.lanes * s.P + s.gA; step = s.sA0 + (ja >> 1); extra = 1; return; }
    const int before = min(s.nB, (i + 1) >> 1) + (ja > 0 ? min(s.nA, (ja + 1) >> 1) : 0);
    const int m = i - before;
    group = pair + (m % s.lanes) * s.P; step = m / s.lanes; extra = 0;
}
// one lane polls the hand-off counter of an extra group (acquire, gpu scope); the warp barrier orders the other lanes
__device__ __forceinline__ void wait_handoff(const int32_t* flag, int target) {
    if ((threadIdx.x & 31) == 0) {
        int v = 0;
        for (uint32_t spins = 0;; ++spins) {
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
            if (v >= target) break;
            if (spins > (1u << 26)) __trap();
            __nanosleep(100);
        }
    }
    __syncwarp();
}

// HT = common width (GEMM2 N): 256 or 128.  TERMS = the split-operand terms as a compile-time constant (7 = f16x2,
// 3 = f16x2w16) or -1 = taken from ForwardArgs::tc_terms at run time (precision ladder / debugging).  Both are template
// parameters because ONE thread issues every MMA: its loops must unroll to straight-line descriptor arithmetic, or the
// issue rate, not the tensor pipe, bounds the kernel (measured: runtime trip counts cost 13 % of the whole collect).
template <int HT, int TERMS, bool FOLD = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTHREADS, 1)
k_forward_tc2(PolicyDev p, ForwardArgs a, Tc2Params t, const __grid_constant__ CUtensorMap tmap) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t n = a.n_live_ptr ? (int64_t)*a.n_live_ptr : a.n;
    const int n_tiles = (int)((n + TM - 1) / TM);
    const int crank = (int)ctarank();
    const int pair_id = (int)blockIdx.x >> 1, n_pairs = (int)gridDim.x >> 1;
    const int n_groups = (n_tiles + 1) / 2;
    if (pair_id >= n_groups) return;                           // pair-uniform
    // Work items: (step, tile) pairs, all steps of this launch for all tiles owned by this pair, step-major.
    // With t_count > 1 the kernel is persistent over time: a tile's envs stay with this pair for the whole
    // chunk, finished envs idle, and the live list is re-compacted between launches.
    const int t_count = a.t_count > 0 ? a.t_count : 1;
    const Sched sch = make_sched(n_groups, n_pairs, t_count, pair_id, (a.fused && a.bal_flags) ? a.bal_delta : 0);
    const int my_tiles = sch.lanes;
    const int n_items = sch.n_items;

    const uint32_t sbase = smem_u32(smem);
    const uint32_t bars = sbase + SM_BARS;
    auto bar = [&](int i) { return bars + 8u * (uint32_t)i; };
    auto lbar = [&](int i) { return mapa(bars + 8u * (uint32_t)i, 0); };     // same barrier in the leader CTA
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SM_BARS + 8 * B_COUNT);
    float* headw = reinterpret_cast<float*>(smem + SM_HEADW);
    float* b1s = reinterpret_cast<float*>(smem + SM_B1);
    float* embb = reinterpret_cast<float*>(smem + SM_EMBB);
    float* part_s = reinterpret_cast<float*>(smem + SM_PART);
    int8_t* perm_s = reinterpret_cast<int8_t*>(smem + SM_PERM);
    uint8_t* operm_s = smem + SM_OPERM;
    // twist tables in shared memory when they fit (obs_size <= 256 makes every entry a byte): the one-hot build looks
    // up 16 of them per env and step
    const bool operm_smem = p.n_perms > 0 && p.obs_size <= 256 && p.n_perms * p.obs_size <= OPERM_MAX;
    const int NC = t.NC, NKB1 = t.NKB1;
    constexpr int H = HT;
    // Split-operand terms of this launch (ForwardArgs::tc_terms; 0 = all): GEMM1 always has one-hot x table_hi and GEMM2
    // h1_hi x W_hi; bit 0 adds one-hot x table_lo, bit 1 h1_lo x W_hi, bit 2 h1_hi x W_lo.  Skipped terms are neither
    // streamed nor issued.
    // TERMS = 16 | 3: the two correction terms of f16x2w16 as fp8 products (see ONE8 above) -- own operand image, own
    // one-hot copy, six ring slots.
    constexpr bool F8 = TERMS >= 16;
    static_assert(!F8 || TERMS == 19, "fp8 corrections replace exactly the terms of f16x2w16");
    constexpr int NS = F8 ? NSLOTS - A8_TILES : NSLOTS;                  // ring slots
    constexpr int RING = F8 ? SM_RING + A8_TILES * TILE_BYTES : SM_RING;
    const int terms = TERMS >= 0 ? (TERMS & 7) : (a.tc_terms ? (a.tc_terms & 7) : 7);
    const bool g1_lo = (terms & 1) != 0, g2_alo = (terms & 2) != 0, g2_wlo = (terms & 4) != 0;
    const int NKB8 = t.NKB8;
    constexpr uint32_t idesc2 = H == 256 ? IDESC_256x256 : IDESC_256x128;   // GEMM2: N = H
    constexpr int g2_units = H == 256 ? 4 : 2;                               // ring slots of one chunk's GEMM2 (see k_tc2_pack)

    if (threadIdx.x == 0) {
        for (int i = 0; i < NSLOTS; ++i) { mbar_init(bar(B_FULL0 + i), 1); mbar_init(bar(B_EMPTY0 + i), 1); }
        mbar_init(bar(B_A1_FULL), 2 * TM); mbar_init(bar(B_A1_EMPTY), 1);
        mbar_init(bar(B_D1_FULL0), 1); mbar_init(bar(B_D1_FULL1), 1);
        mbar_init(bar(B_A2_FULL0), 2 * NEPI); mbar_init(bar(B_A2_FULL1), 2 * NEPI);
        mbar_init(bar(B_D2_FULL), 1); mbar_init(bar(B_D2_EMPTY), 2 * NEPI);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = threadIdx.x; i < (MAX_KB1 + (F8 ? A8_TILES : 0)) * TILE_BYTES / 16; i += NTHREADS)   // A8 follows A1
        reinterpret_cast<uint4*>(smem + SM_A1)[i] = make_uint4(0, 0, 0, 0);
    // head weights as five rows [output][column] (4 actions, value): the heads read four columns of one output per load
    for (int i = threadIdx.x; i < H; i += NTHREADS) {
        for (int o = 0; o < 4; ++o) headw[o * H + i] = o < p.A ? p.wa[(size_t)i * p.A + o] : 0.0f;
        headw[4 * H + i] = p.wv[i];
        b1s[i] = p.b1[i];
    }
    // zero bias on the padding features; kept rolled, since the unrolled loop shifts ptxas' register allocation of the
    // whole kernel (spills in k_forward_tc2<128, 19>)
#pragma unroll 1
    for (int i = threadIdx.x; i < t.NC * 128; i += NTHREADS) embb[i] = i >= t.E ? 0.0f : F8 ? p.emb_b[i] * H1_SCALE8 : p.emb_b[i];
    if (operm_smem)
        for (int i = threadIdx.x; i < p.n_perms * p.obs_size; i += NTHREADS) operm_s[i] = (uint8_t)p.obs_perms[i];
    // action twists next to the barriers (the heads look one row up per item)
    uint8_t* aperm_s = smem + SM_BARS + 384;
    const bool aperm_smem = p.n_perms > 0 && p.n_perms * p.A <= 128;
    if (aperm_smem)
        for (int i = threadIdx.x; i < p.n_perms * p.A; i += NTHREADS) aperm_s[i] = (uint8_t)p.act_perms[i];
    if (warp == 1) {   // both CTAs, same warp id: allocates the same 512 columns in both SMs
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    cluster_sync();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t D2_COL = 0, D1_COL = 256;
    const bool timed = a.dbg != nullptr;
    // event trace of CTA 0 (first 8 items, 32 slots each) behind the per-CTA counters: clock64 stamps
    long long* trace = (timed && blockIdx.x == 0) ? a.dbg + TWR_DBG_TRACE : nullptr;
    auto stamp = [&](int item, int ev) { if (trace && item < 8) trace[item * 32 + ev] = clock64(); };

    if (warp == 0) {
        // =============================== TMA producer (both CTAs) ===================
        // Each CTA fetches ITS half of every operand tile into its own ring; both halves credit the
        // leader's `full` barrier, so the MMA issuer waits on one local barrier per ring slot.
        if (lane == 0) {
            const int img_row0 = t.row0 + crank * (int)slots_per_rank(t) * (TILE_BYTES / 128);   // tensor-map row of this rank's image
            const int g1_row0 = img_row0, g2_row0 = img_row0 + (int)slots_g1(t) * (TILE_BYTES / 128);
            uint32_t use = 0;
            long long w_empty = 0;
            auto push = [&](int row) {
                const uint32_t slot = use % NS, round = use / NS;
                mbar_wait_t(bar(B_EMPTY0 + slot), (round & 1u) ^ 1u, w_empty, timed);
                if (a.dbg_flags & 2) {                      // ablation: no operand traffic, the slot is "full" at once
                    if (crank == 0) mbar_arrive(bar(B_FULL0 + slot));
                } else {
                    if (crank == 0) mbar_expect_tx(bar(B_FULL0 + slot), 2 * TILE_BYTES);
                    tma_load_2sm(sbase + RING + slot * TILE_BYTES, &tmap, 0, row, bar(B_FULL0 + slot));
                }
                ++use;
            };
            auto push_g1 = [&](int sc) {
                for (int i = 0; i < 2 * NKB1; ++i)
                    if (!(i & 1) || g1_lo) push(g1_row0 + (sc * 2 * NKB1 + i) * (TILE_BYTES / 128));
            };
            auto push_g2 = [&](int j) {                     // unit u: part = u & 1 (H = 256: u = kb * 2 + part; H = 128: u = part)
                for (int u = 0; u < g2_units; ++u)
                    if (!(u & 1) || g2_wlo) push(g2_row0 + (j * g2_units + u) * (TILE_BYTES / 128));
            };
            if constexpr (F8) {
                // the image holds exactly the slots this variant streams, in order
                const int n1 = NKB1 + NKB8, n2 = 2 * (H == 256 ? 3 : 2);
                for (int it = 0; it < n_items; ++it)
                    for (int sc = 0; sc < NC / 2; ++sc) {
                        for (int u = 0; u < n1; ++u) push(g1_row0 + (sc * n1 + u) * (TILE_BYTES / 128));
                        for (int u = 0; u < n2; ++u) push(g2_row0 + (sc * n2 + u) * (TILE_BYTES / 128));
                    }
            } else {
                for (int it = 0; it < n_items; ++it)
                    for (int sc = 0; sc < NC / 2; ++sc) { push_g1(sc); push_g2(2 * sc); push_g2(2 * sc + 1); }
            }
            if (a.dbg) a.dbg[blockIdx.x * 16 + 8] = w_empty;
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0 && crank == 0) {
            // =========================== MMA issuer (leader CTA) ======================
            uint32_t use = 0, d1use = 0, a2use = 0;
            long long w_slot = 0, w_a1 = 0, w_a2 = 0, w_d2 = 0, w_slot_g1 = 0, w_slot_first = 0;
            const long long t_begin = clock64();
            auto wait_slot = [&]() -> uint32_t {
                const uint32_t slot = use % NS, round = use / NS;
                mbar_wait_cluster_t(bar(B_FULL0 + slot), round & 1u, w_slot, timed);
                tc_fence_after();
                ++use;
                return slot;
            };
            for (int it = 0; it < n_items; ++it) {
                mbar_wait_cluster_t(bar(B_A1_FULL), it & 1, w_a1, timed);
                tc_fence_after();
                stamp(it, 0);
                // GEMM1 of the chunk pair (2sc, 2sc+1): N = 256 MMAs write both D1 buffers (columns [256,384) = chunk 2sc from
                // rank 0's half of B, [384,512) = chunk 2sc+1 from rank 1's half)
                auto g1 = [&](int sc) {
                    stamp(it, 1 + 2 * sc);
                    const uint32_t d = tmem + D1_COL;
                    if constexpr (F8) {
                        constexpr uint32_t I8_256 = idesc8(256, 1, 0), I8_128 = idesc8(128, 1, 0);
                        const bool on = !(a.dbg_flags & 8);
                        for (int kb = 0; kb < NKB1 - 1; ++kb) {
                            const uint64_t ad = make_desc(sbase + SM_A1 + kb * TILE_BYTES);
                            const long long w0 = w_slot;
                            const uint32_t slot = wait_slot();
                            w_slot_g1 += w_slot - w0;
                            if (kb == 0) w_slot_first += w_slot - w0;
                            const uint64_t bh = make_desc(sbase + RING + slot * TILE_BYTES);
                            if (on) {
#pragma unroll
                                for (int ks = 0; ks < 4; ++ks) tc2_mma(d, ad + 2u * ks, bh + 2u * ks, IDESC_256x256, (kb | ks) != 0);
                            }
                            tc2_commit(bar(B_EMPTY0 + slot));
                            if ((kb & 1) && (kb >> 1) < NKB8 - 1) {
                                const uint64_t a8 = make_desc(sbase + SM_A8 + (kb >> 1) * TILE_BYTES);
                                const long long w1 = w_slot;
                                const uint32_t slot8 = wait_slot();
                                w_slot_g1 += w_slot - w1;
                                const uint64_t b8 = make_desc(sbase + RING + slot8 * TILE_BYTES);
                                if (on) {
#pragma unroll
                                    for (int ks = 0; ks < 4; ++ks) tc2_mma8(d, a8 + 2u * ks, b8 + 2u * ks, I8_256, 1u);
                                }
                                tc2_commit(bar(B_EMPTY0 + slot8));
                            }
                        }
                        {   // last hi k-block + last one-byte k-block, chunk 2sc first (rows 0..63 of both slots), then chunk 2sc+1
                            const int kb = NKB1 - 1;
                            const uint64_t ad = make_desc(sbase + SM_A1 + kb * TILE_BYTES);
                            const uint64_t a8 = make_desc(sbase + SM_A8 + (NKB8 - 1) * TILE_BYTES);
                            const long long w0 = w_slot;
                            const uint32_t slot_h = wait_slot();
                            const uint32_t slot_l = wait_slot();
                            w_slot_g1 += w_slot - w0;
                            if (kb == 0) w_slot_first += w_slot - w0;
                            const uint64_t bh = make_desc(sbase + RING + slot_h * TILE_BYTES);
                            const uint64_t bl = make_desc(sbase + RING + slot_l * TILE_BYTES);
                            const uint64_t half = (uint64_t)((64 * 128) >> 4);
                            if (on) {
#pragma unroll
                                for (int ks = 0; ks < 4; ++ks) tc2_mma(d, ad + 2u * ks, bh + 2u * ks, IDESC_256x128, (kb | ks) != 0);
#pragma unroll
                                for (int ks = 0; ks < 4; ++ks) tc2_mma8(d, a8 + 2u * ks, bl + 2u * ks, I8_128, 1u);
                            }
                            tc2_commit(bar(B_D1_FULL0));
                            if (on) {
#pragma unroll
                                for (int ks = 0; ks < 4; ++ks) tc2_mma(d + 128u, ad + 2u * ks, bh + half + 2u * ks, IDESC_256x128, (kb | ks) != 0);
#pragma unroll
                                for (int ks = 0; ks < 4; ++ks) tc2_mma8(d + 128u, a8 + 2u * ks, bl + half + 2u * ks, I8_128, 1u);
                            }
                            tc2_commit(bar(B_EMPTY0 + slot_h));
                            tc2_commit(bar(B_EMPTY0 + slot_l));
                            tc2_commit(bar(B_D1_FULL1));
                        }
                        if (sc == NC / 2 - 1) tc2_commit(bar(B_A1_EMPTY));
                        d1use += 2;
                        return;
                    }
                    for (int kb = 0; kb < NKB1 - 1; ++kb) {
                        const uint64_t ad = make_desc(sbase + SM_A1 + kb * TILE_BYTES);
                        const long long w0 = w_slot;
                        const uint32_t slot_h = wait_slot();
                        const uint32_t slot_l = g1_lo ? wait_slot() : slot_h;
                        w_slot_g1 += w_slot - w0;
                        if (kb == 0) w_slot_first += w_slot - w0;
                        const uint64_t bh = make_desc(sbase + RING + slot_h * TILE_BYTES);
                        const uint64_t bl = make_desc(sbase + RING + slot_l * TILE_BYTES);
                        if (!(a.dbg_flags & 8)) {
                            // per k-step: table_hi then table_lo against the SAME one-hot A tile -- back-to-back MMAs that share
                            // their shared-memory A operand issue faster than the (all hi, then all lo) order: +4 % on the whole
                            // collect; explicit collector::a::fill / lastuse hints on the pair add nothing on top
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks) {
                                tc2_mma(d, ad + 2u * ks, bh + 2u * ks, IDESC_256x256, (kb | ks) != 0);
                                if (g1_lo) tc2_mma(d, ad + 2u * ks, bl + 2u * ks, IDESC_256x256, 1u);
                            }
                        }
                        tc2_commit(bar(B_EMPTY0 + slot_h));
                        if (g1_lo) tc2_commit(bar(B_EMPTY0 + slot_l));
                    }
                    // last k-block: chunk 2sc is completed first (N = 128 MMAs on rows 0..63 of the hi and the lo slot) and
                    // published, so that its epilogue-1 runs while chunk 2sc+1 (rows 64..127 of the same two slots) finishes --
                    // otherwise GEMM2 would wait a whole epilogue-1 after the pair
                    {
                        const int kb = NKB1 - 1;
                        const uint64_t ad = make_desc(sbase + SM_A1 + kb * TILE_BYTES);
                        const long long w0 = w_slot;
                        const uint32_t slot_h = wait_slot();
                        const uint32_t slot_l = g1_lo ? wait_slot() : slot_h;
                        w_slot_g1 += w_slot - w0;
                        const uint64_t bh = make_desc(sbase + RING + slot_h * TILE_BYTES);
                        const uint64_t bl = make_desc(sbase + RING + slot_l * TILE_BYTES);
                        const uint64_t half = (uint64_t)((64 * 128) >> 4);          // 64 rows further into the slot (descriptor address units of 16 B)
                        if (!(a.dbg_flags & 8)) {
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks) {
                                tc2_mma(d, ad + 2u * ks, bh + 2u * ks, IDESC_256x128, (kb | ks) != 0);
                                if (g1_lo) tc2_mma(d, ad + 2u * ks, bl + 2u * ks, IDESC_256x128, 1u);
                            }
                        }
                        tc2_commit(bar(B_D1_FULL0));
                        if (!(a.dbg_flags & 8)) {
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks) {
                                tc2_mma(d + 128u, ad + 2u * ks, bh + half + 2u * ks, IDESC_256x128, (kb | ks) != 0);
                                if (g1_lo) tc2_mma(d + 128u, ad + 2u * ks, bl + half + 2u * ks, IDESC_256x128, 1u);
                            }
                        }
                        tc2_commit(bar(B_EMPTY0 + slot_h));
                        if (g1_lo) tc2_commit(bar(B_EMPTY0 + slot_l));
                        tc2_commit(bar(B_D1_FULL1));
                    }
                    if (sc == NC / 2 - 1) tc2_commit(bar(B_A1_EMPTY));
                    d1use += 2;
                };
                auto g2 = [&](int j) {
                    const uint32_t buf = a2use & 1u;
                    mbar_wait_cluster_t(bar(B_A2_FULL0 + buf), (a2use >> 1) & 1u, w_a2, timed);
                    tc_fence_after();
                    if (j == 0) { mbar_wait_cluster_t(bar(B_D2_EMPTY), (it & 1) ^ 1, w_d2, timed); tc_fence_after(); }
                    stamp(it, 5 + j);
                    const uint32_t a_base = tmem + D1_COL + buf * 128u;
                    const uint32_t d = tmem + D2_COL;
                    if constexpr (F8) {
                        // hi slots (H = 256: k-blocks 0, 1; H = 128: one slot with both), then the one-byte slot: the chunk's
                        // 128 features as 4 MMAs of K = 32, A = the e5m2 residues at columns +16..+23 of every 32-feature group
                        constexpr uint32_t I8 = idesc8((uint32_t)H, 1, 1);
                        const bool on = !(a.dbg_flags & 4);
#pragma unroll
                        for (int u = 0; u < (H == 256 ? 2 : 1); ++u) {
                            const uint32_t slot = wait_slot();
                            const uint64_t bd = make_desc(sbase + RING + slot * TILE_BYTES);
                            constexpr int nks = H == 256 ? 4 : 8;
                            if (on) {
#pragma unroll
                                for (int ks = 0; ks < nks; ++ks) {
                                    const uint32_t sidx = H == 256 ? (uint32_t)(u * 4 + ks) : (uint32_t)ks;
                                    const uint32_t ah = a_base + 32u * (sidx >> 1) + 8u * (sidx & 1u);
                                    const uint64_t bk = H == 256 ? bd + 2u * ks : bd + (uint64_t)((ks >> 2) * (8192 >> 4)) + 2u * (ks & 3);
                                    tc2_mma_ts(d, ah, bk, idesc2, !(j == 0 && u == 0 && ks == 0));
                                }
                            }
                            tc2_commit(bar(B_EMPTY0 + slot));
                        }
                        {
                            const uint32_t slot = wait_slot();
                            const uint64_t bd = make_desc(sbase + RING + slot * TILE_BYTES);
                            if (on) {
#pragma unroll
                                for (int ks = 0; ks < 4; ++ks) tc2_mma8_ts(d, a_base + 32u * ks + 16u, bd + 2u * ks, I8, 1u);
                            }
                            tc2_commit(bar(B_EMPTY0 + slot));
                        }
                        ++a2use;
                        if (j == NC - 1) tc2_commit(bar(B_D2_FULL));
                        return;
                    }
                    // unit u = one ring slot: H = 256 -> (kb, part) = (u >> 1, u & 1), 4 k-steps of 16 features;
                    // H = 128 -> part = u, both k-blocks (two 64-row sub-tiles), 8 k-steps
#pragma unroll
                    for (int u = 0; u < g2_units; ++u) {
                        const int part = u & 1;
                        if (part && !g2_wlo) continue;
                        const uint32_t slot = wait_slot();
                        const uint64_t bd = make_desc(sbase + RING + slot * TILE_BYTES);
                        const bool first = (j == 0 && u == 0);
                        if (!(a.dbg_flags & 4)) {
                            constexpr int nks = H == 256 ? 4 : 8;
#pragma unroll
                            for (int ks = 0; ks < nks; ++ks) {
                                const uint32_t sidx = H == 256 ? (uint32_t)((u >> 1) * 4 + ks) : (uint32_t)ks;
                                const uint32_t ah = a_base + 32u * (sidx >> 1) + 8u * (sidx & 1u);
                                const uint64_t bk = H == 256 ? bd + 2u * ks : bd + (uint64_t)((ks >> 2) * (8192 >> 4)) + 2u * (ks & 3);
                                tc2_mma_ts(d, ah, bk, idesc2, !(first && ks == 0));
                                if (part == 0 && g2_alo) tc2_mma_ts(d, ah + 16u, bk, idesc2, 1u);
                            }
                        }
                        tc2_commit(bar(B_EMPTY0 + slot));
                    }
                    ++a2use;
                    if (j == NC - 1) tc2_commit(bar(B_D2_FULL));
                };
                for (int sc = 0; sc < NC / 2; ++sc) { g1(sc); g2(2 * sc); g2(2 * sc + 1); }
                stamp(it, 9);
            }
            if (a.dbg) {
                long long* d = a.dbg + blockIdx.x * 16;
                d[0] = clock64() - t_begin; d[1] = w_slot; d[2] = w_a1; d[3] = w_a2; d[4] = w_d2; d[5] = my_tiles;
                d[6] = w_slot_g1; d[7] = w_slot_first;
            }
        }
        __syncwarp();
    } else {
        // =============================== epilogue warps (both CTAs) =================
        // Two warps per TMEM lane quarter: `chalf` picks which half of the columns a thread handles.
        const int quarter = warp & 3;
        const int chalf = (warp - 2) >> 2;
        const int row = quarter * 32 + lane;
        const uint32_t lane_addr = ((uint32_t)(quarter * 32)) << 16;
        const int n_obs = p.n_obs;
        uint32_t d1use = 0;
        int perm_cur = -1, perm_next = -1;
        long long w_d1 = 0, w_d2f = 0, w_a1e = 0, c_epi1 = 0, c_build = 0, c_epi2 = 0;
        const long long t_begin = clock64();
        const uint32_t l_a1_full = lbar(B_A1_FULL), l_d2_empty = lbar(B_D2_EMPTY);
        const uint32_t l_a2_full0 = lbar(B_A2_FULL0), l_a2_full1 = lbar(B_A2_FULL1);
        float ba_r[4];                         // head biases: read once, not once per item
#pragma unroll
        for (int o = 0; o < 4; ++o) ba_r[o] = o < p.A ? p.ba[o] : 0.0f;
        const float bv_r = p.bv[0];

        // Global loads of the env state for item `it`, issued early (at the start of the previous item) so
        // their latency is off the critical path of the one-hot build.
        struct Pre { int64_t pos; int64_t e; uint4 c; int step; };
        // (group, step, extra) of items it-1, it, it+1: sched_item divides by run-time values, so every item is resolved ONCE
        // per thread (at the end of the iteration two before it) instead of once per use
        struct Ent { int group, step, extra; };
        Ent e_prev{0, 0, 0}, e_cur{0, 0, 0}, e_next{0, 0, 0};
        sched_item(sch, pair_id, 0, e_cur.group, e_cur.step, e_cur.extra);
        if (n_items > 1) sched_item(sch, pair_id, 1, e_next.group, e_next.step, e_next.extra);
        auto prefetch = [&](const Ent& en) -> Pre {
            const int group = en.group, step = en.step, extra = en.extra;
            // first step of a piece whose earlier steps ran on another pair: wait until both of its CTAs published them
            if (extra == 1 && step == sch.sA0 && sch.sA0 > 0) wait_handoff(a.bal_flags + sch.gA, 2 * sch.sA0);
            Pre q; q.pos = ((int64_t)group * 2 + crank) * TM + row; q.e = 0; q.c = make_uint4(0, 0, 0, 0); q.step = step;
            if (q.pos < n) {
                q.e = a.live ? a.live[q.pos] : q.pos;
                if (!a.obs_rows) q.c = __ldcg(a.cells + q.e);   // written by the partner thread's fused step >= 1 item earlier
            }
            return q;
        };
        auto build_a1 = [&](int it, const Pre& q) -> int {
            const int64_t pos = q.pos;
            const int t_cur = a.t + q.step;
            int perm = -1;
            EnvState s; s.blank = 0; s.depth = 0;
            s.lo = (uint64_t)q.c.x | ((uint64_t)q.c.y << 32);
            s.hi = (uint64_t)q.c.z | ((uint64_t)q.c.w << 32);
            if (pos < n) {
                if (a.perm_idx) {
                    perm = a.perm_idx[pos];
                } else if (p.n_perms > 0 && a.t >= 0) {
                    uint32_t w[4];
                    philox4x32_10(a.ids.gid((uint32_t)q.e), (uint32_t)t_cur, TWR_RNG_PERM, a.cid, (uint32_t)a.seed,
                                  (uint32_t)(a.seed >> 32), w);
                    perm = (int)mulhi_u32(w[0], (uint32_t)p.n_perms);
                }
            }
            // One-hot row of this env: zero the whole row (NKB1 x 128 B, eight 16-byte stores per k-block, no
            // bookkeeping of the previous tile's ones), then set one fp16 1.0 per observation index.
            const uint32_t rx = (uint32_t)row & 7u;
            const uint32_t row_base = ((uint32_t)row >> 3) * 1024u + rx * 128u;
            // Puzzle from the env state, at most 16 cells; a twist is one more byte lookup when its table sits in shared memory
            const bool fast = a.env.kind == 0 && !a.obs_rows && (perm < 0 || operm_smem) && n_obs <= 16 && t.cN == 0;
            const uint8_t* otab = perm >= 0 ? operm_s + perm * p.obs_size : nullptr;
            if (threadIdx.x == 192) stamp(it, 20);
            mbar_wait_t(bar(B_A1_EMPTY), (it & 1) ^ 1, w_a1e, timed);      // GEMM1 of the previous item is done with A1
            if (threadIdx.x == 192) stamp(it, 21);
            // the 32 rows of this warp are 4 KB contiguous per k-block: lanes write consecutive 16-byte chunks
            // (conflict-free), then the warp syncs before anyone sets a one in a row another lane zeroed
            for (int kb = 0; kb < NKB1; ++kb) {
                uint4* dst = reinterpret_cast<uint4*>(smem + SM_A1 + kb * TILE_BYTES + quarter * 4096) + lane;
#pragma unroll
                for (int j = 0; j < 8; ++j) dst[j * 32] = make_uint4(0, 0, 0, 0);
            }
            if constexpr (F8) {
                for (int kb = 0; kb < NKB8; ++kb) {
                    uint4* dst = reinterpret_cast<uint4*>(smem + SM_A8 + kb * TILE_BYTES + quarter * 4096) + lane;
#pragma unroll
                    for (int j = 0; j < 8; ++j) dst[j * 32] = make_uint4(0, 0, 0, 0);
                }
            }
            __syncwarp();
            // the same index in the one-byte copy of the operand (k-blocks of 128)
            auto set8 = [&](uint32_t r) {
                if constexpr (F8) {
                    const uint32_t k8 = r & 127u;
                    smem[SM_A8 + (r >> 7) * TILE_BYTES + row_base + ((((k8 >> 4) ^ rx) & 7u) << 4) + (k8 & 15u)] = ONE8;
                }
            };
            if (fast) {
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    if (i < n_obs) {
                        const uint32_t v = (uint32_t)(((i < 8) ? s.lo : s.hi) >> (8 * (i & 7))) & 0xFFu;
                        uint32_t r = pos < n ? (uint32_t)(i * a.env.N) + v : 0u;
                        if (otab && pos < n) r = otab[r];                                          // twist-in, policy.rs:81-83
                        const uint32_t k = r & 63u;
                        *reinterpret_cast<__half*>(smem + SM_A1 + (r >> 6) * TILE_BYTES + row_base + ((((k >> 3) ^ rx) & 7u) << 4) + (k & 7u) * 2u) =
                            __ushort_as_half(0x3C00);
                        set8(r);
                    }
                }
            } else {
                for (int i = 0; i < n_obs; ++i) {
                    uint32_t r = 0;
                    if (pos < n) {
                        r = a.obs_rows ? (uint32_t)a.obs_rows[pos * n_obs + i] : (uint32_t)(i * a.env.N) + env_board(a.env, s, i);
                        if (perm >= 0)                                                         // twist-in, policy.rs:81-83
                            r = operm_smem ? (uint32_t)operm_s[perm * p.obs_size + (int)r] : (uint32_t)p.obs_perms[(size_t)perm * p.obs_size + r];
                        if (t.cN > 0) r = (r / (uint32_t)t.cN) * 4u + (r % (uint32_t)t.cN);   // compact GridWorld table (values 0..3)
                    }
                    const uint32_t k = r & 63u;
                    *reinterpret_cast<__half*>(smem + SM_A1 + (r >> 6) * TILE_BYTES + row_base + ((((k >> 3) ^ rx) & 7u) << 4) + (k & 7u) * 2u) =
                        __ushort_as_half(0x3C00);
                    set8(r);
                }
            }
            perm_s[(it & 3) * TM + row] = (int8_t)perm;
            fence_async_smem();
            mbar_arrive_cluster(l_a1_full);
            if (threadIdx.x == 192) stamp(it, 22);
            return perm;
        };
        // relu(x + bias) -> packed fp16 hi pair / lo pair (x = hi + lo to ~22 bits)
        // ReLU rides on the two conversions (see split4 below): hi = fp16(relu(x)) rounded toward zero, so the residue is
        // >= 0 wherever x is, and the relu of the residue's conversion zeroes exactly the lanes with x < 0
        // (only when the residue is used: a rung of the precision ladder without the h1_lo term rounds hi to nearest)
        auto split2 = [g2_alo](float x0, float x1, uint32_t& hi, uint32_t& lo) {
            if (g2_alo) {
                asm("cvt.rz.relu.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(x1), "f"(x0));   // first source -> upper half
                const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi));
                asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(x1 - hf.y), "f"(x0 - hf.x));
            } else {
                asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(x1), "f"(x0));
                lo = 0u;
            }
        };

        // fp8 variant: four features -> two fp16 pairs and ONE word of four e5m2 residues (feature k at byte k, the K order
        // of an 8-bit A operand in tensor memory).  ReLU costs nothing here: hi = fp16(relu(x)) rounded TOWARD ZERO
        // (cvt.rz.relu), so the residue x - hi is >= 0 wherever x >= 0, and the relu of the residue's own conversion
        // (cvt.rn.satfinite.relu.e5m2x2) zeroes exactly the lanes with x < 0 (hi = 0, residue = x < 0).
        auto split4 = [](float x0, float x1, float x2, float x3, uint32_t& hi01, uint32_t& hi23, uint32_t& lo) {
            asm("cvt.rz.relu.f16x2.f32 %0, %1, %2;" : "=r"(hi01) : "f"(x1), "f"(x0));     // first source -> upper half
            asm("cvt.rz.relu.f16x2.f32 %0, %1, %2;" : "=r"(hi23) : "f"(x3), "f"(x2));
            const float2 f01 = __half22float2(*reinterpret_cast<const __half2*>(&hi01)), f23 = __half22float2(*reinterpret_cast<const __half2*>(&hi23));
            const float2 r01 = __fadd2_rn(make_float2(x0, x1), make_float2(-f01.x, -f01.y));     // packed fp32: two residues per instruction
            const float2 r23 = __fadd2_rn(make_float2(x2, x3), make_float2(-f23.x, -f23.y));
            uint16_t l01, l23;
            asm("cvt.rn.satfinite.relu.e5m2x2.f32 %0, %1, %2;" : "=h"(l01) : "f"(r01.y), "f"(r01.x));
            asm("cvt.rn.satfinite.relu.e5m2x2.f32 %0, %1, %2;" : "=h"(l23) : "f"(r23.y), "f"(r23.x));
            lo = (uint32_t)l01 | ((uint32_t)l23 << 16);
        };

        // the next item's one-hot operand is normally built BEFORE this item's heads (so its GEMM1 overlaps
        // them); with a single tile per pair the next item is the same envs one step later, whose state
        // only exists after this item's fused env step
        const bool build_early = my_tiles > 1 || t_count == 1;
        // ---- epilogue 1 of chunk c: this thread's 64 columns of the D1 chunk, rewritten in place as the fp16 A operand
        auto epi1 = [&](int it, int c) {
            const uint32_t buf = d1use & 1u;
            mbar_wait_t(bar(B_D1_FULL0 + buf), (d1use >> 1) & 1u, w_d1, timed);
            tc_fence_after();
            if (threadIdx.x == 64) stamp(it, 10 + c);
            const long long t_e1 = timed ? clock64() : 0;
            if (!(a.dbg_flags & 1)) {
                uint32_t v0[32], v1[32];
                const uint32_t taddr = tmem + lane_addr + D1_COL + buf * 128u + (uint32_t)chalf * 64u;
                tc_ld32(taddr, v0);
                tc_ld32(taddr + 32u, v1);
                tc_wait_ld();
                const float* bias = embb + c * 128 + chalf * 64;
                uint32_t w[32];
                if constexpr (F8) {
                    // accumulator + embedding bias; with the bias folded into the operand image the accumulator is the sum
                    // (x + 0.0f would not do: the compiler must keep an add that turns -0.0 into +0.0)
                    auto addb = [&](uint32_t v, const float& b) -> float {
                        if constexpr (FOLD) return __uint_as_float(v); else return __uint_as_float(v) + b;
                    };
#pragma unroll
                    for (int e4 = 0; e4 < 8; ++e4)
                        split4(addb(v0[4 * e4], bias[4 * e4]), addb(v0[4 * e4 + 1], bias[4 * e4 + 1]),
                               addb(v0[4 * e4 + 2], bias[4 * e4 + 2]), addb(v0[4 * e4 + 3], bias[4 * e4 + 3]),
                               w[2 * e4], w[2 * e4 + 1], w[16 + e4]);
#pragma unroll
                    for (int e4 = 24; e4 < 32; ++e4) w[e4] = 0u;
                    tc_st32(taddr, w);
#pragma unroll
                    for (int e4 = 0; e4 < 8; ++e4)
                        split4(addb(v1[4 * e4], bias[32 + 4 * e4]), addb(v1[4 * e4 + 1], bias[32 + 4 * e4 + 1]),
                               addb(v1[4 * e4 + 2], bias[32 + 4 * e4 + 2]), addb(v1[4 * e4 + 3], bias[32 + 4 * e4 + 3]),
                               w[2 * e4], w[2 * e4 + 1], w[16 + e4]);
                    tc_st32(taddr + 32u, w);
                } else {
#pragma unroll
                    for (int e2 = 0; e2 < 16; ++e2)
                        split2(__uint_as_float(v0[2 * e2]) + bias[2 * e2], __uint_as_float(v0[2 * e2 + 1]) + bias[2 * e2 + 1], w[e2], w[16 + e2]);
                    tc_st32(taddr, w);
#pragma unroll
                    for (int e2 = 0; e2 < 16; ++e2)
                        split2(__uint_as_float(v1[2 * e2]) + bias[32 + 2 * e2], __uint_as_float(v1[2 * e2 + 1]) + bias[32 + 2 * e2 + 1], w[e2], w[16 + e2]);
                    tc_st32(taddr + 32u, w);
                }
                tc_wait_st();
            }
            tc_fence_before();
            mbar_arrive_cluster(buf ? l_a2_full1 : l_a2_full0);
            if (timed) c_epi1 += clock64() - t_e1;
            if (threadIdx.x == 64) stamp(it, 14 + c);
            ++d1use;
        };
        // ---- the collect step of one item (lower-half threads): record, sample, env step, hand-off signal
        struct Saved { float out[4]; float value; int perm; int64_t pos; int step, group, extra; bool valid; };
        auto run_step = [&](const Saved& v) {
            const bool active = v.pos < n;
            if (a.fused) {
                const int e = active ? (a.live ? a.live[v.pos] : (int)v.pos) : 0;
                StepArgs sa = a.step;
                sa.t = a.t + v.step;
                // inside a multi-step chunk an env that already recorded its terminal state idles
                const bool alive = active && (t_count == 1 || a.cb.ep_len[e] == 0);
                collect_step_body(sa, a.cb, alive, e, make_float4(v.out[0], v.out[1], v.out[2], v.out[3]), v.value, v.perm,
                                  a.live_next);
            } else if (active) {
                a.logits[v.pos] = make_float4(v.out[0], v.out[1], v.out[2], v.out[3]);
                a.values[v.pos] = v.value;
            }
            if (v.extra) {
                // a time-split group: publish this CTA's finished step to the pair that runs the next piece
                asm volatile("bar.sync 4, %0;" ::"n"(NEPI / 2) : "memory");
                if (threadIdx.x == 64) { __threadfence(); atomicAdd(a.bal_flags + (v.group - sch.lanes * sch.P), 1); }
            }
        };
        // Deferred step: the fused collect step of item `it` (global loads, Philox, record stores: ~5k cycles) would sit
        // between this item's heads and the next item's first epilogue-1, right where GEMM2 of the next item waits for its
        // A operand; it runs instead after epilogue-1 of the next item's first chunk pair, hidden behind that GEMM2.
        const bool defer = build_early && a.fused && t_count > 1;
        Saved sv;
        sv.valid = false; sv.pos = 0; sv.step = 0; sv.group = 0; sv.extra = 0; sv.perm = -1; sv.value = 0.f;
        sv.out[0] = sv.out[1] = sv.out[2] = sv.out[3] = 0.f;

        if (chalf == 1) perm_next = build_a1(0, prefetch(e_cur));      // the upper-half warps own the one-hot operand
        for (int it = 0; it < n_items; ++it) {
            Pre pre_next; pre_next.pos = 0; pre_next.e = 0; pre_next.c = make_uint4(0, 0, 0, 0); pre_next.step = 0;
            int c_done = 0;
            if (defer) {
                // Item it+1's env state was last written by the step of an earlier item of the same group (same-group
                // items are >= 2 apart).  Steps of items <= it-2 finished before the previous iteration's bar.sync 1; only
                // when item it-1 IS that earlier item do the upper-half threads have to wait (barrier 3) for the step the
                // lower half runs right now -- otherwise their loads go out at once and the one-hot build of item it+1 does
                // not queue behind a 5k-cycle step it does not depend on.
                const bool dep = it >= 1 && it + 1 < n_items && e_prev.group == e_next.group;
                for (; c_done < 2 && c_done < NC; ++c_done) epi1(it, c_done);
                if (chalf == 1 && it + 1 < n_items && !dep) pre_next = prefetch(e_next);
                if (chalf == 0 && sv.valid) {                          // step of item it-1
                    if (threadIdx.x == 64) stamp(it, 23);
                    run_step(sv);
                    if (threadIdx.x == 64) stamp(it, 24);
                    sv.valid = false;
                    if (dep) asm volatile("bar.arrive 3, %0;" ::"n"(NEPI) : "memory");
                }
                if (chalf == 1 && dep) {
                    asm volatile("bar.sync 3, %0;" ::"n"(NEPI) : "memory");
                    pre_next = prefetch(e_next);
                }
            } else if (build_early && chalf == 1 && it + 1 < n_items) {
                // with >= 2 tiles per pair, item it+1's env state was last written by the fused step of item
                // it+1-my_tiles <= it-1 (lower-half threads); barrier 3 orders that step before these loads
                if (t_count > 1 && it >= 1) asm volatile("bar.sync 3, %0;" ::"n"(NEPI) : "memory");
                pre_next = prefetch(e_next);
            }
            for (; c_done < NC; ++c_done) epi1(it, c_done);
            // ---- next tile's one-hot operand, so its GEMM1 overlaps this tile's heads
            {
                const long long t_b = timed ? clock64() : 0;
                if (build_early && chalf == 1 && it + 1 < n_items) perm_next = build_a1(it + 1, pre_next);
                if (timed) c_build += clock64() - t_b;
            }

            // ---- epilogue 2: heads on CUDA cores; each thread reduces its 128 columns of the accumulator row
            mbar_wait_t(bar(B_D2_FULL), it & 1, w_d2f, timed);
            tc_fence_after();
            if (threadIdx.x == 64) stamp(it, 18);
            const long long t_e2 = timed ? clock64() : 0;
            // packed fp32 (fma.rn.f32x2 / add.f32x2, sm_100): even and odd columns accumulate in the two halves of a register
            // pair -- the activations of two adjacent accumulator columns and the two weights of an output's row are
            // adjacent already -- and are added at the end: 10 FFMA2 + 2 FADD2 instead of 20 FFMA + 4 FADD per four columns
            float2 acc2[5];
#pragma unroll
            for (int o = 0; o < 5; ++o) acc2[o] = make_float2(0.f, 0.f);
#pragma unroll 1
            for (int q = 0; q < H / 128; ++q) {
                uint32_t v0[32], v1[32];
                const uint32_t col0 = (uint32_t)(chalf * (H / 2)) + (uint32_t)q * 64u;
                tc_ld32(tmem + lane_addr + D2_COL + col0, v0);
                tc_ld32(tmem + lane_addr + D2_COL + col0 + 32u, v1);
                tc_wait_ld();
#pragma unroll
                for (int j4 = 0; j4 < 16; ++j4) {
                    const int col = (int)col0 + 4 * j4;
                    const float4 bb = *reinterpret_cast<const float4*>(b1s + col);
                    float hv[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int j = 4 * j4 + k;
                        hv[k] = __uint_as_float(j < 32 ? v0[j & 31] : v1[j & 31]);
                    }
                    float2 h01 = __fadd2_rn(make_float2(hv[0], hv[1]), make_float2(bb.x, bb.y));
                    float2 h23 = __fadd2_rn(make_float2(hv[2], hv[3]), make_float2(bb.z, bb.w));
                    h01.x = fmaxf(h01.x, 0.f); h01.y = fmaxf(h01.y, 0.f); h23.x = fmaxf(h23.x, 0.f); h23.y = fmaxf(h23.y, 0.f);
#pragma unroll
                    for (int o = 0; o < 5; ++o) {
                        const float4 w = *reinterpret_cast<const float4*>(headw + o * H + col);
                        acc2[o] = __ffma2_rn(h01, make_float2(w.x, w.y), acc2[o]);
                        acc2[o] = __ffma2_rn(h23, make_float2(w.z, w.w), acc2[o]);
                    }
                }
            }
            float acc[5];
#pragma unroll
            for (int o = 0; o < 5; ++o) acc[o] = acc2[o].x + acc2[o].y;
            tc_fence_before();
            mbar_arrive_cluster(l_d2_empty);
            float* ps = part_s + ((it & 1) * TM + row) * 8;
            if (chalf == 1) {
                *reinterpret_cast<float4*>(ps) = make_float4(acc[0], acc[1], acc[2], acc[3]);
                ps[4] = acc[4];
            }
            if (threadIdx.x == 64) stamp(it, 25);
            asm volatile("bar.sync 1, %0;" ::"n"(NEPI) : "memory");     // the 8 epilogue warps only
            if (threadIdx.x == 64) stamp(it, 26);
            if (chalf == 0) {                                          // warp-uniform: whole warps take this branch
                Saved cur;
                cur.group = e_cur.group; cur.step = e_cur.step; cur.extra = e_cur.extra;
                cur.pos = ((int64_t)cur.group * 2 + crank) * TM + row;
                cur.valid = true;
                cur.out[0] = cur.out[1] = cur.out[2] = cur.out[3] = 0.f;
                cur.value = 0.f;
                perm_cur = perm_s[(it & 3) * TM + row];             // written by the partner thread when it built this tile
                cur.perm = perm_cur;
                if (cur.pos < n) {
                    const float4 o4 = *reinterpret_cast<const float4*>(ps);
                    acc[0] += o4.x; acc[1] += o4.y; acc[2] += o4.z; acc[3] += o4.w; acc[4] += ps[4];
                    float l[4];
#pragma unroll
                    for (int o = 0; o < 4; ++o) l[o] = o < p.A ? acc[o] + ba_r[o] : 0.0f;
#pragma unroll
                    for (int o = 0; o < 4; ++o) cur.out[o] = l[o];
                    if (perm_cur >= 0) {                               // twist-out, nn/policy.rs:95-97
#pragma unroll
                        for (int o = 0; o < 4; ++o) {
                            if (o < p.A) {
                                const int src = aperm_smem ? (int)aperm_s[perm_cur * p.A + o] : p.act_perms[perm_cur * p.A + o];
                                cur.out[o] = src == 0 ? l[0] : src == 1 ? l[1] : src == 2 ? l[2] : l[3];
                            }
                        }
                    }
                    cur.value = acc[4] + bv_r;
                }
                if (defer && it + 1 < n_items) {
                    sv = cur;                                          // runs inside the next iteration
                } else {
                    run_step(cur);
                    // publish "step of item `it` done" to the upper-half threads (matched by their bar.sync 3 at item it+1)
                    if (!defer && build_early && t_count > 1 && it + 2 < n_items) asm volatile("bar.arrive 3, %0;" ::"n"(NEPI) : "memory");
                }
            }
            if (!build_early && it + 1 < n_items) {                    // single tile per pair: the next item is these envs one step later
                asm volatile("bar.sync 2, %0;" ::"n"(NEPI) : "memory");  // their fused env step (lower-half threads) is done
                if (chalf == 1) perm_next = build_a1(it + 1, prefetch(e_next));
            }
            e_prev = e_cur; e_cur = e_next;
            if (it + 2 < n_items) sched_item(sch, pair_id, it + 2, e_next.group, e_next.step, e_next.extra);
            if (timed) c_epi2 += clock64() - t_e2;
            if (threadIdx.x == 64) stamp(it, 19);
        }
        if (a.dbg && threadIdx.x == 64) {
            long long* d = a.dbg + blockIdx.x * 16;
            d[9] = clock64() - t_begin; d[10] = w_d1; d[11] = w_d2f; d[12] = w_a1e; d[13] = c_epi1; d[14] = c_build; d[15] = c_epi2;
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u));
    }
}

Tc2Params make_params2(const PolicyDev& p, bool f8 = false) {
    Tc2Params t;
    t.E = p.E; t.H = p.H; t.NC = 2 * ((p.E + 255) / 256); t.cN = p.tc_compact_n;   // E % 256 == 128: zero-padded to a chunk pair
    t.NKB1 = ((p.tc_compact_n > 0 ? 4 * p.tc_compact_n : p.obs_size) + 63) / 64;
    t.NKB8 = (t.NKB1 + 1) / 2;
    t.f8 = 0; t.row0 = 0; t.fold = 0;
    if (f8) {                                   // the fp8-correction image follows the standard one; it carries the folded bias
        t.row0 = (int)(2 * slots_per_rank(t) * (TILE_BYTES / 128));
        t.f8 = 1;
        t.fold = p.tc_fold;
    }
    return t;
}

// Per-device launch state (one engine per device, several devices per process): SM count, whether every cluster of a
// full grid is resident at once (the balanced schedule needs it), the shared-memory attribute, and the tensor maps of
// the operand images that live on that device.
struct DevState {
    int sms = 0;
    int max_clusters = -1;
    bool attr_set = false;
    std::map<std::pair<const void*, size_t>, CUtensorMap> tmaps;   // keyed by (image address, bytes): a freed image's address can be reused by a larger one
};
constexpr int MAX_DEVICES = 64;
std::mutex g_dev_mu;
DevState g_dev[MAX_DEVICES];

DevState* dev_state() {                      // call with g_dev_mu held
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEVICES) return nullptr;
    DevState& d = g_dev[dev];
    if (d.sms == 0) cudaDeviceGetAttribute(&d.sms, cudaDevAttrMultiProcessorCount, dev);
    return &d;
}

// Tensor map over the packed operand image viewed as [rows][128 bytes]; one 128 x 128 box = one ring slot.
bool get_tmap(DevState& d, const void* pack, size_t bytes, CUtensorMap* out) {
    const std::pair<const void*, size_t> key(pack, bytes);
    auto it = d.tmaps.find(key);
    if (it != d.tmaps.end()) { *out = it->second; return true; }
    typedef CUresult (*encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn) return false;
    const cuuint64_t gdim[2] = {128, (cuuint64_t)(bytes / 128)};
    const cuuint64_t gstride[1] = {128};
    const cuuint32_t box[2] = {128, 128};
    const cuuint32_t estr[2] = {1, 1};
    CUtensorMap m;
    const CUresult r = reinterpret_cast<encode_fn>(fn)(&m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(pack), gdim, gstride, box,
                                                       estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                                       CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return false;
    d.tmaps[key] = m;
    *out = m;
    return true;
}

}  // namespace

// E in 128-feature chunks (an odd count is padded to a pair), the one-hot operand holds <= 256 (compact) rows, GEMM2 is
// N = H in {128, 256}
int forward_tc2_supported(const PolicyDev& p) {
    const int k1 = p.tc_compact_n > 0 ? 4 * p.tc_compact_n : p.obs_size;
    return (p.H == 256 || p.H == 128) && p.E % 128 == 0 && p.E <= 1024 && k1 <= 64 * MAX_KB1;
}

size_t forward_tc2_pack_bytes(const PolicyDev& p) {
    if (!forward_tc2_supported(p)) return 0;
    return 2 * (slots_per_rank(make_params2(p)) + slots_per_rank(make_params2(p, true))) * TILE_BYTES;
}

void launch_forward_tc2_pack(cudaStream_t st, const PolicyDev& p, void* pack) {
    k_tc2_pack<<<1024, 256, 0, st>>>(p, make_params2(p), reinterpret_cast<__half*>(pack));
    const Tc2Params t8 = make_params2(p, true);
    k_tc2_pack8<<<1024, 256, 0, st>>>(p, t8, reinterpret_cast<unsigned char*>(pack) + (size_t)t8.row0 * 128);
    g_twr_launches.fetch_add(2, std::memory_order_relaxed);
}

// Everything a launch needs besides the arguments, resolved once (at policy creation) so that a launch cannot fail for
// a reason known earlier: the tensor map of `pack`, the kernel's shared-memory attribute, cluster residency.
bool forward_tc2_prepare(const PolicyDev& p, const void* pack) {
    std::lock_guard<std::mutex> lk(g_dev_mu);
    DevState* d = dev_state();
    if (!d) return false;
    CUtensorMap tmap;
    if (!get_tmap(*d, pack, forward_tc2_pack_bytes(p), &tmap)) return false;
    if (!d->attr_set) {
        for (auto k : {k_forward_tc2<256, 7>, k_forward_tc2<256, 3>, k_forward_tc2<256, -1>, k_forward_tc2<128, 7>, k_forward_tc2<128, 3>,
                       k_forward_tc2<128, -1>, k_forward_tc2<256, 19>, k_forward_tc2<128, 19>, k_forward_tc2<256, 19, true>,
                       k_forward_tc2<128, 19, true>})
            if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL) != cudaSuccess) return false;
        d->attr_set = true;
    }
    if (d->max_clusters < 0) {
        // The balanced schedule lets a pair wait for another pair's progress, which needs every cluster of the grid to
        // be resident at once: query it once per device and keep the plain schedule when the device cannot hold them all.
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)((d->sms / 2) * 2)); cfg.blockDim = dim3(NTHREADS); cfg.dynamicSmemBytes = SM_TOTAL;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        int nc = 0;
        d->max_clusters = cudaOccupancyMaxActiveClusters(&nc, k_forward_tc2<256, 7>, &cfg) == cudaSuccess ? nc : 0;
        cudaGetLastError();
    }
    return true;
}

void forward_tc2_forget(const void* pack) {   // the operand image is being freed: drop its tensor map
    std::lock_guard<std::mutex> lk(g_dev_mu);
    DevState* d = dev_state();
    if (!d) return;
    for (auto it = d->tmaps.begin(); it != d->tmaps.end();)
        it = it->first.first == pack ? d->tmaps.erase(it) : std::next(it);
}

bool launch_forward_tc2(cudaStream_t st, const PolicyDev& p, const ForwardArgs& a, const void* pack) {
    if (a.n <= 0) return true;
    CUtensorMap tmap;
    int sms, max_clusters;
    {
        std::lock_guard<std::mutex> lk(g_dev_mu);
        DevState* d = dev_state();
        if (!d || !d->attr_set || !get_tmap(*d, pack, forward_tc2_pack_bytes(p), &tmap)) return false;   // forward_tc2_prepare did not run / failed
        sms = d->sms; max_clusters = d->max_clusters;
    }
    const int n_tiles = (int)((a.n + TM - 1) / TM);
    const int n_groups = (n_tiles + 1) / 2, max_pairs = sms / 2;
    const int grid = (n_groups < max_pairs ? n_groups : max_pairs) * 2;
    ForwardArgs args = a;
    if (a.bal_flags && max_clusters < grid / 2) { args.bal_flags = nullptr; args.bal_delta = 0; }
    const int terms = a.tc_terms ? (a.tc_terms & 7) : 7;
    // fp8 corrections: only defined for the f16x2w16 terms.  A policy whose fp8 image carries the folded embedding bias
    // (tc_fold) serves observations with one index per block -- every env-driven launch, and explicit rows the host has
    // checked; anything else takes the same terms with fp16 corrections on the standard image.
    const bool blocks = a.obs_rows ? a.obs_blocks != 0 : p.n_obs == p.tc_fold;
    const bool f8 = (a.tc_terms & 16) != 0 && terms == 3 && (p.tc_fold == 0 || blocks);
    const bool fold = f8 && p.tc_fold > 0;
    const Tc2Params t = make_params2(p, f8);
    auto go = [&](auto kern) { kern<<<grid, NTHREADS, SM_TOTAL, st>>>(p, args, t, tmap); };
    if (fold) { if (p.H == 256) go(k_forward_tc2<256, 19, true>); else go(k_forward_tc2<128, 19, true>); }
    else if (p.H == 256) { if (f8) go(k_forward_tc2<256, 19>); else if (terms == 7) go(k_forward_tc2<256, 7>); else if (terms == 3) go(k_forward_tc2<256, 3>); else go(k_forward_tc2<256, -1>); }
    else            { if (f8) go(k_forward_tc2<128, 19>); else if (terms == 7) go(k_forward_tc2<128, 7>); else if (terms == 3) go(k_forward_tc2<128, 3>); else go(k_forward_tc2<128, -1>); }
    g_twr_launches.fetch_add(1, std::memory_order_relaxed);
    return true;
}
